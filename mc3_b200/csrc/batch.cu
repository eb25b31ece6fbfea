// mc3_b200 -- many independent small problems at once, one persistent CTA per problem:
// the launchers and C entry points of the built-in models.  The kernels are in
// batch_dev.cuh; jit.cu launches them for a user model.  k_batch_gr, the Gelman-Rubin
// test of every problem, reads only the history and serves both.
#include "batch_dev.cuh"
#include "gelman_dev.cuh"

// Problem 0's description, read back to the host for the argument checks and the launch
// shape (the user-model entry points of jit.cu check their model themselves).
int mc3b_batch_shape(const mc3b_batch_t* b, mc3b_sampler_t* s, cudaStream_t st) {
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
    return MC3B_OK;
}

namespace {

int batch_shape(const mc3b_batch_t* b, int model_id, int nmodel, mc3b_sampler_t* s, cudaStream_t st) {
    if (int rc = mc3b_batch_shape(b, s, st)) return rc;
    MC3B_CHECK_ARG(mc3b_model_nparams(model_id, nmodel) == nmodel, "model %d does not take %d parameters", model_id,
                   nmodel);
    return MC3B_OK;
}

template <class M>
int launch_init(const mc3b_batch_t* b, const mc3b_sampler_t& s, int kickoff, cudaStream_t st) {
    k_init_batch<M><<<(unsigned)b->nproblems, SW * 32, 0, st>>>(*b, kickoff, (int)s.nchains, s.npars, s.nfree,
                                                                 BatchExtra{});
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
                                                                        gen0 + done, step, BatchExtra{});
        MC3B_CHECK_LAUNCH("k_run_batch");
        done += step;
    }
    return MC3B_OK;
}


// ---- Gelman-Rubin test of every problem (mcmc_driver.py:325-346) ------------------------
constexpr int GR_THREADS = 256;                               // chain c in slot c of gr_psrf's tree
constexpr int GR_SLOTS = (MC3B_MAX_PARS * SW * 32) / GR_THREADS;  // (chain, parameter) pairs per thread
constexpr int64_t GR_CHUNK = 4096;                            // doubles per staging buffer, unless a step needs more

__device__ __forceinline__ void cp_async8(double* dst, const double* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)),
                 "l"(src)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One pass over the thinned steps [0, niter) of the problem's block src (step s holds the
// nn = nchains * nfree doubles of its rows, element e = chain e / nfree, parameter e % nfree):
// acc[j] of element t + 256 j takes, in step order, x (PASS 0) or (x - mu[e])^2 (PASS 1), as
// k_gr_stats' serial loops do.  The CTA stages chunks of `steps` steps through two shared
// buffers with 8-byte cp.async (coalesced: consecutive threads, consecutive doubles), the
// next chunk in flight while the current one is summed.
template <int PASS>
__device__ __forceinline__ void gr_pass(const double* src, int64_t niter, int nn, int64_t steps, double* buf,
                                        const double* mu, double (&acc)[GR_SLOTS]) {
    const int t = threadIdx.x;
#pragma unroll
    for (int j = 0; j < GR_SLOTS; j++) acc[j] = 0.0;
    const int64_t nchunk = (niter + steps - 1) / steps;
    auto issue = [&](int64_t ci) {
        const int64_t s0 = ci * steps, cnt = (niter - s0 < steps ? niter - s0 : steps) * nn;
        double* dst = buf + (ci & 1) * steps * nn;
        for (int64_t i = t; i < cnt; i += GR_THREADS) cp_async8(dst + i, src + s0 * nn + i);
        cp_async_commit();
    };
    issue(0);
    for (int64_t ci = 0; ci < nchunk; ci++) {
        if (ci + 1 < nchunk) {
            issue(ci + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const double* cur = buf + (ci & 1) * steps * nn;
        const int64_t ns = niter - ci * steps < steps ? niter - ci * steps : steps;
#pragma unroll
        for (int j = 0; j < GR_SLOTS; j++) {
            const int e = t + GR_THREADS * j;
            if (e < nn) {
                double a = acc[j];
                if (PASS == 0) {
                    for (int64_t r = 0; r < ns; r++) a += cur[r * nn + e];
                } else {
                    const double m = mu[e];
                    for (int64_t r = 0; r < ns; r++) a = gr_sq_add(a, cur[r * nn + e] - m);
                }
                acc[j] = a;
            }
        }
        __syncthreads();                              // the buffer is refilled two chunks on
    }
}

// PSRF at report point k of every problem whose status is 0, one CTA per problem: the
// moments of k_gr_stats (two passes over the thinned steps [zburn, k), rows
// M0 + k' nchains + c, contiguous for the problem) and the PSRF of k_gr_psrf (gr_psrf), with
// the same arithmetic in the same order.  Shared memory: two staging buffers of `steps`
// steps, the means [nn] and gr_psrf's 256 slots; the variances reuse the first buffer.
__global__ void __launch_bounds__(GR_THREADS) k_batch_gr(mc3b_batch_t B, int64_t k, int64_t zburn, double grbreak,
                                                         int64_t grnmin, int64_t steps, double* psrf, int64_t ldpsrf,
                                                         int64_t* kstop) {
    extern __shared__ __align__(16) double sm[];
    const int64_t b = blockIdx.x;
    if (B.status[b] != 0) return;                     // never initialised, or stopped
    const mc3b_sampler_t& G = B.problems[b];
    const int64_t nch = G.nchains, nf = G.nfree, M0 = G.M0;
    const int nn = (int)(nch * nf);
    const int64_t niter = k - zburn;
    const double* src = G.Z + (M0 + zburn * nch) * nf;
    double* buf = sm;
    double* mu = sm + 2 * steps * nn;
    double* sh = mu + nn;
    double acc[GR_SLOTS];
    gr_pass<0>(src, niter, nn, steps, buf, mu, acc);
#pragma unroll
    for (int j = 0; j < GR_SLOTS; j++) {
        const int e = threadIdx.x + GR_THREADS * j;
        if (e < nn) mu[e] = acc[j] / (double)niter;
    }
    gr_pass<1>(src, niter, nn, steps, buf, mu, acc);
    double* var = buf;                                // free after the last chunk's barrier
#pragma unroll
    for (int j = 0; j < GR_SLOTS; j++) {
        const int e = threadIdx.x + GR_THREADS * j;
        if (e < nn) var[e] = acc[j] / (double)niter;
    }
    __syncthreads();
    bool pass = true;                                 // NaN never passes
    for (int64_t p = 0; p < nf; p++) {
        const double r = gr_psrf(mu, var, nf, nch, niter, p, sh);
        if (threadIdx.x == 0) {
            psrf[b * ldpsrf + p] = r;
            pass = pass && r < grbreak;
        }
    }
    if (threadIdx.x == 0 && grbreak > 0.0 && pass && M0 + k * nch > grnmin) {
        B.status[b] = 3;
        kstop[b] = k;
    }
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

extern "C" int mc3b_batch_gelman_rubin(const mc3b_batch_t* b, int64_t k, int64_t zburn, double grbreak,
                                       int64_t grnmin, double* psrf, int64_t ldpsrf, int64_t* kstop, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    mc3b_sampler_t s;
    if (int rc = mc3b_batch_shape(b, &s, st)) return rc;
    MC3B_CHECK_ARG(s.nchains >= 2, "the Gelman-Rubin test needs at least 2 chains");
    MC3B_CHECK_ARG(zburn >= 0 && k > zburn && s.M0 + k * s.nchains <= s.zlen,
                   "report point out of range (need 0 <= zburn < k and M0 + k nchains <= zlen)");
    MC3B_CHECK_ARG(psrf && ldpsrf >= s.nfree && (kstop || !(grbreak > 0.0)), "bad arguments");
    const int64_t nn = s.nchains * s.nfree;
    int64_t steps = GR_CHUNK / nn > 1 ? GR_CHUNK / nn : 1;
    if (steps > k - zburn) steps = k - zburn;
    const int bytes = (int)((2 * steps * nn + nn + GR_THREADS) * sizeof(double));
    MC3B_CUDA(cudaFuncSetAttribute(k_batch_gr, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    k_batch_gr<<<(unsigned)b->nproblems, GR_THREADS, bytes, st>>>(*b, k, zburn, grbreak, grnmin, steps, psrf, ldpsrf,
                                                                   kstop);
    MC3B_CHECK_LAUNCH("k_batch_gr");
    return MC3B_OK;
}
