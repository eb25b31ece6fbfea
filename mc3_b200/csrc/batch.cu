// mc3_b200 -- many independent small problems at once, one persistent CTA per problem:
// the launchers and C entry points of the built-in models.  The kernels are in
// batch_dev.cuh; jit.cu launches them for a user model.
#include "batch_dev.cuh"

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
