// mc3_b200 -- persistent kernel for small populations.
//
// The reference's everyday use (7-21 chains, 1e2-1e4 data points, ~1e5
// samples) is launch-latency bound when every generation is three kernel
// launches: the arithmetic of a generation takes well under a microsecond.
// k_run_small keeps one CTA resident and runs `ngen` generations inside it:
//
// The per-chain state (X, chi-squared, proposals, counters, bounds, priors) is
// copied to shared memory once and written back at the end; only the history
// rows go to global memory.  Measured: 5.9 us per generation for 7 chains x 100
// points (the proposal arithmetic of one thread per chain dominates), against
// 21 us with one CUDA-graph node per kernel.
//
//     threads 0..nchains-1   propose_chain()            (sampler_dev.cuh)
//     __syncthreads
//     one warp per chain     model + chi-squared over the data (lanes stride the
//                            points, fixed-order lane tree)
//     __syncthreads
//     threads 0..nchains-1   metropolis_chain()         (priors, accept, write)
//     __syncthreads
//
// (small_generations in small_dev.cuh, which the batched kernels of batch.cu share).
// Same Philox streams, same proposal and acceptance code as the per-generation
// kernels; only the order in which a chain's chi-squared terms are added
// differs (rounding-level).  Bound: latency (one CTA by construction).
#include "small_dev.cuh"

namespace {

template <class M>
__global__ void __launch_bounds__(SW * 32) k_run_small(mc3b_sampler_t G, const double* __restrict__ x,
                                                       const double* __restrict__ d,
                                                       const double* __restrict__ w, int64_t n, int64_t gen0,
                                                       int64_t ngen) {
    extern __shared__ __align__(16) double sm[];
    small_generations<M>(G, x, d, w, n, gen0, ngen, sm);
}

template <class M>
int launch_small(const mc3b_sampler_t* s, const double* x, const double* data, const double* invsig, int64_t n,
                 int64_t gen0, int64_t ngen, int bytes, cudaStream_t st) {
    MC3B_CUDA(cudaFuncSetAttribute(k_run_small<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    k_run_small<M><<<1, SW * 32, bytes, st>>>(*s, x, data, invsig, n, gen0, ngen);
    MC3B_CHECK_LAUNCH("k_run_small");
    return MC3B_OK;
}

}  // namespace

extern "C" int mc3b_run_small(const mc3b_sampler_t* s, int model_id, int nmodel, const double* x, const double* data,
                              const double* invsig, int64_t n, int64_t gen0, int64_t ngen, void* stream) {
    MC3B_CHECK_ARG(s && x && data && invsig && n > 0 && gen0 >= 0 && ngen > 0, "bad arguments");
    MC3B_CHECK_ARG(s->nchains <= SW * 32 && s->chain0 == 0 && s->nlocal == s->nchains,
                   "run_small handles one device and at most %d chains", SW * 32);
    MC3B_CHECK_ARG(s->nfree > 0 && s->nfree <= MC3B_MAX_PARS && s->npars <= MC3B_MAX_PARS && s->thinning > 0,
                   "nfree/npars/thinning out of range");
    MC3B_CHECK_ARG(s->sampler != MC3B_DEMC || s->nchains >= 3, "demc needs at least 3 chains");
    MC3B_CHECK_ARG(s->sampler != MC3B_SNOOKER || s->M0 >= 2, "snooker needs at least 2 history rows");
    if (model_id == MC3B_MODEL_SINUSOID_GRID) model_id = MC3B_MODEL_SINUSOID;
    MC3B_CHECK_ARG(mc3b_model_nparams(model_id, nmodel) == nmodel, "model %d does not take %d parameters", model_id,
                   nmodel);
    cudaStream_t st = (cudaStream_t)stream;
    const SmallLayout L = small_layout((int)s->nchains, s->npars, s->nfree);
    MC3B_CHECK_ARG(L.bytes <= 200 * 1024, "population too large for the persistent kernel");
    MC3B_DISPATCH_MODEL(double, model_id, nmodel,
                        return (launch_small<M>(s, x, data, invsig, n, gen0, ngen, L.bytes, st)));
    return MC3B_OK;
}
