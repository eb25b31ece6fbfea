// mc3_b200 -- the kernels of many independent small problems at once, one persistent CTA
// per problem.  Device code only: batch.cu instantiates them for the built-in models and
// launches them, jit.cu has NVRTC instantiate them for a user model (the header travels
// inside the library as a string, csrc/jit_headers.inc written by build.py).
//
// The reference's everyday fits (7-21 chains on 1e2-1e4 points) keep one CTA of
// k_run_small busy and leave the rest of the GPU idle.  A catalogue of such fits (one
// per star, transit or band) is a set of independent problems: grid = B CTAs, CTA b
// runs problem b from its own row of a device table of mc3b_sampler_t.
//
//   k_init_batch   the initial population of problem b inside its CTA: trial points of
//                  init_trial (k_init_trials' draws), bounds test, a warp per in-bounds
//                  trial for chi-squared + priors, selection in draw order
//   k_run_batch    small_generations (the loop of k_run_small) over problem b
//   k_batch_eval   the model values of every problem's parameter row over its own points
//                  (a user model's best_model; the built-ins use k_model_eval)
//
// A user model of NX > 1 inputs reads inputs 2..NX of problem b at xe[j] + offsets[b], and
// a model of constants its row consts + b * nk (BatchExtra; the built-ins read neither).
//
// Bound: latency per CTA, as k_run_small; problems run side by side up to the
// resident-CTA count.
#pragma once
#ifndef __CUDACC_RTC__          // NVRTC has no math.h (isfinite and fmin are built in)
#include <math.h>
#endif
#include "small_dev.cuh"

// NVRTC: a named namespace, so that the instantiations have names the loader can
// look up (jit.cu); the library keeps them local to batch.cu.
#ifdef __CUDACC_RTC__
namespace mc3b_jit {
#else
namespace {
#endif

constexpr int IB = 64;              // trials per chunk of k_init_batch

// (SW * 32, 3): 80 registers, the budget of k_run_small, whose state comes from the parameter bank;
// unbounded, the problem's row of the table held in registers takes 127 and two CTAs per SM.
// A user model keeps its [parameters | constants | work] slots in registers (up to 32
// doubles per lane), and NVRTC's k_run_batch of the README's transit models takes 216-218
// registers unbounded.  Under (SW * 32, 2), 128 registers, all three spill (56-72 bytes
// of stack); under (SW * 32, 1) none does: one CTA per SM, a problem per SM at a time.
#ifdef __CUDACC_RTC__
constexpr int BATCH_BLOCKS = 1;
#else
constexpr int BATCH_BLOCKS = 3;
#endif

// The per-point inputs 2..NX and the constants of every problem, as mc3b_batch_t holds x:
// input j + 1 of problem b is xe[j] + offsets[b], its constants consts[b * nk .. b * nk + nk).
struct BatchExtra {
    const double* xe[MC3B_MAX_INPUTS - 1];
    const double* consts;
    int64_t nk;
};

// (left empty for a model that reads neither: the built-ins' code stays as it was)
template <class M>
__device__ __forceinline__ ModelExtra problem_extra(const BatchExtra& X, int64_t b, int64_t o) {
    ModelExtra e = {};
    if constexpr (ninputs_of<M>::value > 1 || takes_consts<M>::value) {
#pragma unroll
        for (int j = 0; j < MC3B_MAX_INPUTS - 1; j++) e.xe[j] = X.xe[j] + o;
        e.k = X.consts + b * X.nk;
    }
    return e;
}

__device__ __forceinline__ bool same_shape(const mc3b_sampler_t& G, int nch, int npars, int nfree, int64_t n) {
    return G.nchains == nch && G.npars == npars && G.nfree == nfree && n > 0;
}

template <class M>
__global__ void __launch_bounds__(SW * 32, BATCH_BLOCKS) k_run_batch(mc3b_batch_t B, int nch, int npars, int nfree,
                                                                     int64_t gen0, int64_t ngen, BatchExtra X) {
    extern __shared__ __align__(16) double sm[];
    const int64_t b = blockIdx.x;
    if (B.status[b] != 0) return;                   // never initialised
    mc3b_sampler_t G = B.problems[b];
    G.gen_dev = nullptr;
    const int64_t o = B.offsets[b], n = B.offsets[b + 1] - o;
    if (!same_shape(G, nch, npars, nfree, n)) return;
    small_generations<M>(G, B.x + o, problem_extra<M>(X, b, o), B.data + o, B.invsig + o, n, gen0, ngen, sm);
}

// Population.init_population (engine.py) for problem b, in rounds of nt trials taken in
// chunks of IB: thread i < IB draws trial t0 + i into shared memory; thread 0 marks, in draw
// order, the in-bounds trials up to the round's cap; a warp per marked trial adds its data
// chi-squared (warp_chisq) and prior terms (as metropolis_apply); thread 0 assigns the finite
// ones, in draw order, the next history rows; the CTA copies them.
template <class M>
__global__ void __launch_bounds__(SW * 32) k_init_batch(mc3b_batch_t B, int kickoff, int nch, int npars, int nfree,
                                                        BatchExtra X) {
    __shared__ double cand[IB * MC3B_MAX_PARS];
    __shared__ double lpv[IB];
    __shared__ int mark[IB];
    __shared__ int64_t dst[IB];
    __shared__ int64_t s_ninb, s_last, s_got;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t b = blockIdx.x;
    const mc3b_sampler_t G = B.problems[b];
    const int64_t o = B.offsets[b], n = B.offsets[b + 1] - o;
    if (!same_shape(G, nch, npars, nfree, n)) {
        if (tid == 0) B.status[b] = 2;
        return;
    }
    const double *x = B.x + o, *d = B.data + o, *w = B.invsig + o;
    const ModelExtra ex = problem_extra<M>(X, b, o);
    const int64_t M0 = G.M0;
    int64_t got = 0, tried = 0, rnd = 0;
    while (got < M0 && tried < 100 * M0) {
        const double want = (double)(M0 - got > 64 ? M0 - got : 64) * 1.25 + 64.0;
        const int64_t nt = (int64_t)fmin(want, (double)(100 * M0 - tried));
        const int64_t need = M0 - got;
        const int64_t cap = need + (need / 100 > 8 ? need / 100 : 8);
        int64_t ninb = 0, last = -1;
        for (int64_t t0 = 0; t0 < nt && ninb < cap && got < M0; t0 += IB) {
            if (tid < IB) {
                const int64_t t = t0 + tid;
                mark[tid] = t < nt ? init_trial(G, kickoff, t, rnd, cand + tid * npars) : 0;
            }
            __syncthreads();
            if (tid == 0) {
                for (int i = 0; i < IB; i++) {
                    if (mark[i] && ninb < cap) { ninb++; last = t0 + i; }
                    else mark[i] = 0;
                }
                s_ninb = ninb; s_last = last;
            }
            __syncthreads();
            ninb = s_ninb; last = s_last;
            for (int i = warp; i < IB; i += SW) {
                if (!mark[i]) continue;
                const double* p = cand + i * npars;
                M m;
                load_model(m, p, ex);
                double chi = warp_chisq(m, x, ex, d, w, n, lane);
                if (lane == 0) {
                    if (G.prior != nullptr) {                // stats.py:208-216
                        double pr = 0.0;
                        for (int k = 0; k < npars; k++) {
                            const double lo = G.priorlow[k], up = G.priorup[k];
                            if (lo > 0.0 && up > 0.0) {
                                const double off = p[k] - G.prior[k];
                                const double t = off / (off > 0.0 ? up : lo);
                                pr += t * t;
                            }
                        }
                        chi += pr;
                    }
                    lpv[i] = -0.5 * chi;
                }
            }
            __syncthreads();
            if (tid == 0) {
                for (int i = 0; i < IB; i++) {
                    dst[i] = -1;
                    if (mark[i] && got < M0 && isfinite(lpv[i])) dst[i] = got++;
                }
                s_got = got;
            }
            __syncthreads();
            got = s_got;
            for (int e = tid; e < IB * nfree; e += SW * 32) {
                const int i = e / nfree, j = e - i * nfree;
                if (dst[i] >= 0) G.Z[dst[i] * nfree + j] = cand[i * npars + G.ifree[j]];
            }
            for (int i = tid; i < IB; i += SW * 32)
                if (dst[i] >= 0) G.log_post[dst[i]] = lpv[i];
            __syncthreads();                                 // cand, mark and dst are reused
        }
        tried += ninb ? last + 1 : nt;
        rnd++;
    }
    if (got < M0) {
        if (tid == 0) B.status[b] = 1;
        return;
    }
    // chain.py:163-170: chain c starts at Z[c], chi-squared -2 log_post[c]
    for (int i = tid; i < nch * nfree; i += SW * 32) G.X[i] = G.Z[i];
    for (int c = tid; c < nch; c += SW * 32) G.chisq_cur[c] = -2.0 * G.log_post[c];
    if (tid == 0) B.status[b] = 0;
}

// out[i] = model(params + b * ldp) at point i of problem b, for the points [offsets[b],
// offsets[b+1]) of every problem: grid (point blocks, problem strides), 256 threads.
template <class M>
__global__ void k_batch_eval(const double* params, int64_t ldp, mc3b_batch_t B, BatchExtra X, double* out) {
    for (int64_t b = blockIdx.y; b < B.nproblems; b += gridDim.y) {
        const int64_t o = B.offsets[b], n = B.offsets[b + 1] - o;
        const ModelExtra ex = problem_extra<M>(X, b, o);
        M m;
        load_model(m, params + b * ldp, ex);
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
            out[o + i] = model_at(m, B.x + o, ex, i);
    }
}

}  // namespace

#ifndef __CUDACC_RTC__
// The checks of a batch's problem 0, read back into s (batch.cu; jit.cu's entry points too).
int mc3b_batch_shape(const mc3b_batch_t* b, mc3b_sampler_t* s, cudaStream_t st);
#endif
