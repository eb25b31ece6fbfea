// mc3_b200 -- the generation loop of the persistent small-population kernel, as device
// functions of one CTA: k_run_small (small.cu) runs it over one problem, k_run_batch and
// k_init_batch (batch.cu) over one problem per CTA.
#pragma once
#include "models.cuh"
#include "sampler_dev.cuh"

namespace {

constexpr int SW = 8;       // warps

// Shared-memory image of the per-chain state: every array a generation touches
// except the history (Z, log_post, zchain) lives on chip for the whole launch.
struct SmallLayout {
    int oX, oNext, oBestX, oCur, oMr, oU, oBestC, oNew, oVec, oBestG, oInb, oAcc, oOob, oIfree, bytes;
};
__host__ __device__ inline SmallLayout small_layout(int nch, int npars, int nfree) {
    SmallLayout L;
    int o = 0;                                   // in doubles
    L.oX = o; o += nch * nfree;
    L.oNext = o; o += nch * npars;
    L.oBestX = o; o += nch * nfree;
    L.oCur = o; o += nch;
    L.oMr = o; o += nch;
    L.oU = o; o += nch;
    L.oBestC = o; o += nch;
    L.oNew = o; o += nch;
    L.oVec = o; o += 7 * npars;                  // pstep pmin pmax params0 prior priorlow priorup
    L.oBestG = o; o += nch;                      // int64
    L.oInb = o; o += (nch + 1) / 2;              // int32 pairs
    L.oAcc = o; o += (nch + 1) / 2;
    L.oOob = o; o += (nfree + 1) / 2;
    L.oIfree = o; o += (nfree + 1) / 2;
    L.bytes = o * 8;
    return L;
}

// Data chi-squared of the model m over n points, by one warp: lanes stride the points
// with two accumulators, then a fixed-order lane tree (every lane returns the sum).
template <class M>
__device__ __forceinline__ double warp_chisq(const M& m, const double* __restrict__ x, const double* __restrict__ d,
                                             const double* __restrict__ w, int64_t n, int lane) {
    double a0 = 0.0, a1 = 0.0;
    int64_t i = lane;
    for (; i + 32 < n; i += 64) {
        const double r0 = (m.eval_safe(x[i]) - d[i]) * w[i];
        const double r1 = (m.eval_safe(x[i + 32]) - d[i + 32]) * w[i + 32];
        a0 = fma(r0, r0, a0);
        a1 = fma(r1, r1, a1);
    }
    if (i < n) { const double r0 = (m.eval_safe(x[i]) - d[i]) * w[i]; a0 = fma(r0, r0, a0); }
    double a = a0 + a1;
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    return a;
}

// Generations gen0 .. gen0+ngen-1 of the population G inside the calling CTA (SW * 32
// threads; sm: small_layout(...).bytes of dynamic shared memory):
//
//     threads 0..nchains-1   propose_chain()            (sampler_dev.cuh)
//     __syncthreads
//     one warp per chain     model + chi-squared over the data (warp_chisq)
//     __syncthreads
//     threads 0..nchains-1   metropolis_chain()         (priors, accept, write)
//     __syncthreads
//
// The per-chain state is copied to shared memory once and written back at the end;
// only the history rows go to global memory.
template <class M>
__device__ __forceinline__ void small_generations(const mc3b_sampler_t& G, const double* __restrict__ x,
                                                  const double* __restrict__ d, const double* __restrict__ w,
                                                  int64_t n, int64_t gen0, int64_t ngen, double* sm) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    const int nch = (int)G.nchains, npars = G.npars, nfree = G.nfree;
    const SmallLayout L = small_layout(nch, npars, nfree);
    // S = G with the hot arrays redirected to shared memory
    mc3b_sampler_t S = G;
    S.X = sm + L.oX; S.nextp = sm + L.oNext; S.best_x = sm + L.oBestX; S.chisq_cur = sm + L.oCur;
    S.mrfactor = sm + L.oMr; S.u = sm + L.oU; S.best_chisq = sm + L.oBestC;
    double* chisq_new = sm + L.oNew;
    double* vec = sm + L.oVec;
    S.pstep = vec; S.pmin = vec + npars; S.pmax = vec + 2 * npars; S.params0 = vec + 3 * npars;
    if (G.prior) { S.prior = vec + 4 * npars; S.priorlow = vec + 5 * npars; S.priorup = vec + 6 * npars; }
    S.best_gen = reinterpret_cast<int64_t*>(sm + L.oBestG);
    S.inb = reinterpret_cast<int32_t*>(sm + L.oInb);
    S.naccept = reinterpret_cast<int32_t*>(sm + L.oAcc);
    S.outbounds = reinterpret_cast<int32_t*>(sm + L.oOob);
    int32_t* ifree_s = reinterpret_cast<int32_t*>(sm + L.oIfree);
    S.ifree = ifree_s;
    for (int i = tid; i < nch * nfree; i += SW * 32) { S.X[i] = G.X[i]; S.best_x[i] = G.best_x[i]; }
    for (int i = tid; i < nch; i += SW * 32) {
        S.chisq_cur[i] = G.chisq_cur[i]; S.best_chisq[i] = G.best_chisq[i]; S.best_gen[i] = G.best_gen[i];
        S.naccept[i] = G.naccept[i];
    }
    for (int i = tid; i < npars; i += SW * 32) {
        vec[i] = G.pstep[i]; vec[npars + i] = G.pmin[i]; vec[2 * npars + i] = G.pmax[i];
        vec[3 * npars + i] = G.params0[i];
        if (G.prior) { vec[4 * npars + i] = G.prior[i]; vec[5 * npars + i] = G.priorlow[i]; vec[6 * npars + i] = G.priorup[i]; }
    }
    for (int i = tid; i < nfree; i += SW * 32) { ifree_s[i] = G.ifree[i]; S.outbounds[i] = G.outbounds[i]; }
    __syncthreads();

    const mc3b_draws_t none = {};
    for (int64_t g = gen0; g < gen0 + ngen; g++) {
        const int64_t zsize = S.M0 + (g / S.thinning) * S.nchains;
        const int64_t zrow0 = ((g + 1) % S.thinning == 0) ? S.M0 + ((g + 1) / S.thinning - 1) * S.nchains : -1;
        if (tid < nch) propose_chain<false>(S, none, g, zsize, tid);
        __syncthreads();
        for (int c = warp; c < nch; c += SW) {
            if (S.inb[c]) {                              // chain.py:241: no evaluation out of bounds
                M m;
                m.load(S.nextp + (int64_t)c * npars);
                const double a = warp_chisq(m, x, d, w, n, lane);
                if (lane == 0) chisq_new[c] = a;
            }
        }
        __syncthreads();
        if (tid < nch) metropolis_chain(S, chisq_new[tid], g, zrow0, tid);
        __syncthreads();
    }
    // state back to global memory
    for (int i = tid; i < nch * nfree; i += SW * 32) { G.X[i] = S.X[i]; G.best_x[i] = S.best_x[i]; }
    for (int i = tid; i < nch * npars; i += SW * 32) G.nextp[i] = S.nextp[i];
    for (int i = tid; i < nch; i += SW * 32) {
        G.chisq_cur[i] = S.chisq_cur[i]; G.best_chisq[i] = S.best_chisq[i]; G.best_gen[i] = S.best_gen[i];
        G.naccept[i] = S.naccept[i]; G.inb[i] = S.inb[i]; G.mrfactor[i] = S.mrfactor[i]; G.u[i] = S.u[i];
    }
    for (int i = tid; i < nfree; i += SW * 32) G.outbounds[i] = S.outbounds[i];
    if (tid == 0 && G.gen_dev) *G.gen_dev = gen0 + ngen;
}

}  // namespace
