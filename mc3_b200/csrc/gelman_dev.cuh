// mc3_b200 -- the Gelman-Rubin arithmetic (gelman.py:75-92) shared by the one-population
// kernels (k_gr_stats, k_gr_psrf in sampler.cu) and the batched one (k_batch_gr in
// batch.cu): the same operations in the same order, so the two give the same bits.
#pragma once
#include <stdint.h>

// v + d*d in one rounding: the DFMA nvcc contracts `v += d * d` to (--fmad=true), written
// out so that the contraction does not depend on the surrounding code.
__device__ __forceinline__ double gr_sq_add(double v, double d) { return fma(d, d, v); }

// Sum of the 256 slots of a CTA of 256 threads (slot i = thread i's v), fixed tree order.
__device__ __forceinline__ double gr_block_sum(double* sh, double v) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    const double r = sh[0];
    __syncthreads();
    return r;
}

// PSRF of free parameter p from the per-chain means mu[c * nfree + p] and population
// variances var[c * nfree + p] of niter samples each (global or shared memory), by a CTA of
// 256 threads: W, B, V, sqrt(V/W) with sums over chains in the tree of gr_block_sum, chain c
// in slot c mod 256.  Every thread takes part; the result is thread 0's.
__device__ __forceinline__ double gr_psrf(const double* mu, const double* var, int64_t nfree, int64_t nchains,
                                          int64_t niter, int64_t p, double* sh) {
    double a = 0.0, b = 0.0;
    for (int64_t c = threadIdx.x; c < nchains; c += 256) { a += var[c * nfree + p]; b += mu[c * nfree + p]; }
    const double W = gr_block_sum(sh, a) / (double)nchains;
    const double mm = gr_block_sum(sh, b) / (double)nchains;
    double d2 = 0.0;
    for (int64_t c = threadIdx.x; c < nchains; c += 256) d2 = gr_sq_add(d2, mu[c * nfree + p] - mm);
    const double B = (double)niter / ((double)nchains - 1.0) * gr_block_sum(sh, d2);
    // V = W (n-1)/n + B (m+1)/(n m), the first product fused into the sum (as nvcc contracts it)
    const double V = fma(W, ((double)niter - 1.0) / (double)niter,
                         B * (((double)nchains + 1.0) / ((double)niter * (double)nchains)));
    return sqrt(V / W);
}
