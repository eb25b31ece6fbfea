// mc3_b200 -- many independent small problems at once, one persistent CTA per problem.
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
//
// Bound: latency per CTA, as k_run_small; problems run side by side up to the
// resident-CTA count.
#include <math.h>
#include "small_dev.cuh"

namespace {

constexpr int IB = 64;              // trials per chunk of k_init_batch

__device__ __forceinline__ bool same_shape(const mc3b_sampler_t& G, int nch, int npars, int nfree, int64_t n) {
    return G.nchains == nch && G.npars == npars && G.nfree == nfree && n > 0;
}

// (SW * 32, 3): 80 registers, the budget of k_run_small, whose state comes from the parameter bank;
// unbounded, the problem's row of the table held in registers takes 127 and two CTAs per SM.
template <class M>
__global__ void __launch_bounds__(SW * 32, 3) k_run_batch(mc3b_batch_t B, int nch, int npars, int nfree, int64_t gen0,
                                                          int64_t ngen) {
    extern __shared__ __align__(16) double sm[];
    const int64_t b = blockIdx.x;
    if (B.status[b] != 0) return;                   // never initialised
    mc3b_sampler_t G = B.problems[b];
    G.gen_dev = nullptr;
    const int64_t o = B.offsets[b], n = B.offsets[b + 1] - o;
    if (!same_shape(G, nch, npars, nfree, n)) return;
    small_generations<M>(G, B.x + o, B.data + o, B.invsig + o, n, gen0, ngen, sm);
}

// Population.init_population (engine.py) for problem b, in rounds of nt trials taken in
// chunks of IB: thread i < IB draws trial t0 + i into shared memory; thread 0 marks, in draw
// order, the in-bounds trials up to the round's cap; a warp per marked trial adds its data
// chi-squared (warp_chisq) and prior terms (as metropolis_apply); thread 0 assigns the finite
// ones, in draw order, the next history rows; the CTA copies them.
template <class M>
__global__ void __launch_bounds__(SW * 32) k_init_batch(mc3b_batch_t B, int kickoff, int nch, int npars, int nfree) {
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
                m.load(p);
                double chi = warp_chisq(m, x, d, w, n, lane);
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

// Problem 0's description, read back to the host for the argument checks and the launch shape.
int batch_shape(const mc3b_batch_t* b, int model_id, int nmodel, mc3b_sampler_t* s, cudaStream_t st) {
    MC3B_CHECK_ARG(b && b->nproblems > 0 && b->nproblems <= 0x7fffffff && b->problems && b->offsets && b->x &&
                   b->data && b->invsig && b->status, "bad arguments");
    MC3B_CUDA(cudaMemcpyAsync(s, b->problems, sizeof(*s), cudaMemcpyDeviceToHost, st));
    MC3B_CUDA(cudaStreamSynchronize(st));
    MC3B_CHECK_ARG(s->nchains <= SW * 32 && s->chain0 == 0 && s->nlocal == s->nchains,
                   "a batch problem has at most %d chains on one device", SW * 32);
    MC3B_CHECK_ARG(s->nfree > 0 && s->nfree <= MC3B_MAX_PARS && s->npars <= MC3B_MAX_PARS && s->thinning > 0,
                   "nfree/npars/thinning out of range");
    MC3B_CHECK_ARG(s->sampler == MC3B_MRW || s->sampler == MC3B_DEMC || s->sampler == MC3B_SNOOKER,
                   "unknown sampler %d", s->sampler);
    MC3B_CHECK_ARG(s->sampler != MC3B_DEMC || s->nchains >= 3, "demc needs at least 3 chains");
    MC3B_CHECK_ARG(s->sampler != MC3B_SNOOKER || s->M0 >= 2, "snooker needs at least 2 history rows");
    MC3B_CHECK_ARG(s->M0 >= s->nchains && s->zlen >= s->M0, "M0/zlen out of range");
    MC3B_CHECK_ARG(mc3b_model_nparams(model_id, nmodel) == nmodel, "model %d does not take %d parameters", model_id,
                   nmodel);
    return MC3B_OK;
}

template <class M>
int launch_init(const mc3b_batch_t* b, const mc3b_sampler_t& s, int kickoff, cudaStream_t st) {
    k_init_batch<M><<<(unsigned)b->nproblems, SW * 32, 0, st>>>(*b, kickoff, (int)s.nchains, s.npars, s.nfree);
    MC3B_CHECK_LAUNCH("k_init_batch");
    return MC3B_OK;
}

template <class M>
int launch_run(const mc3b_batch_t* b, const mc3b_sampler_t& s, int64_t gen0, int64_t ngen, int bytes,
               cudaStream_t st) {
    MC3B_CUDA(cudaFuncSetAttribute(k_run_batch<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    for (int64_t done = 0; done < ngen;) {           // as Population.run splits mc3b_run_small
        const int64_t step = ngen - done < 200000 ? ngen - done : 200000;
        k_run_batch<M><<<(unsigned)b->nproblems, SW * 32, bytes, st>>>(*b, (int)s.nchains, s.npars, s.nfree,
                                                                        gen0 + done, step);
        MC3B_CHECK_LAUNCH("k_run_batch");
        done += step;
    }
    return MC3B_OK;
}

}  // namespace

extern "C" int mc3b_batch_init(const mc3b_batch_t* b, int model_id, int nmodel, int kickoff, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (model_id == MC3B_MODEL_SINUSOID_GRID) model_id = MC3B_MODEL_SINUSOID;
    mc3b_sampler_t s;
    if (int rc = batch_shape(b, model_id, nmodel, &s, st)) return rc;
    MC3B_CHECK_ARG(kickoff == 0 || kickoff == 1, "kickoff must be 0 (normal) or 1 (uniform)");
    MC3B_DISPATCH_MODEL(double, model_id, nmodel, return (launch_init<M>(b, s, kickoff, st)));
    return MC3B_OK;
}

extern "C" int mc3b_batch_run(const mc3b_batch_t* b, int model_id, int nmodel, int64_t gen0, int64_t ngen,
                              void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (model_id == MC3B_MODEL_SINUSOID_GRID) model_id = MC3B_MODEL_SINUSOID;
    MC3B_CHECK_ARG(gen0 >= 0 && ngen > 0, "bad arguments");
    mc3b_sampler_t s;
    if (int rc = batch_shape(b, model_id, nmodel, &s, st)) return rc;
    const SmallLayout L = small_layout((int)s.nchains, s.npars, s.nfree);
    MC3B_CHECK_ARG(L.bytes <= 200 * 1024, "population too large for the persistent kernel");
    MC3B_DISPATCH_MODEL(double, model_id, nmodel, return (launch_run<M>(b, s, gen0, ngen, L.bytes, st)));
    return MC3B_OK;
}
