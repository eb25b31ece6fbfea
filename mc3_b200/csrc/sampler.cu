// mc3_b200 -- the per-generation sampler kernels (replace the body of
// Chain.run(), mc3/chain.py:183-299, for the whole population at once).
//
//   k_propose      one thread per chain: draws, jump, bounds, shared fill
//   k_metropolis   one thread per chain: partial sums + priors, accept/reject,
//                  counters, per-chain best, thinned history write
//   k_init_trials  initial-population trial points (mcmc_driver.py:229-262)
//   k_gr_*         Gelman-Rubin on device (gelman.py:36-92)
//
// Jump arithmetic uses explicit round-to-nearest mul/add/sub intrinsics (no FMA
// contraction) so that, fed the reference's recorded draws (replay mode), the
// proposed points equal numpy's elementwise results.
#include <stdlib.h>
#include "sampler_dev.cuh"

namespace {

// PDL: launched as a programmatic dependent of the previous kernel of the stream (the
// model kernel that ends the previous generation, which releases its dependents as soon
// as it starts): the draws of this generation -- Philox, Box-Muller, partner indices --
// are taken while that kernel still runs, and only the state-dependent half waits for
// it (griddepcontrol.wait returns when the previous grid has completed and its writes
// are visible).  In device-driven mode the generation counter is written at the very end
// of that kernel, so the draws are taken for counter + 1 and taken again in the rare case
// that the counter had already advanced.
template <bool REPLAY>
__global__ void __launch_bounds__(128) k_propose(mc3b_sampler_t S, mc3b_draws_t D, int64_t gen, int64_t zsize,
                                                 int64_t c_begin, int64_t c_end, int pdl) {
    const int64_t c = c_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = c < c_end;
    const bool devgen = gen < 0;                     // device-driven generation (graph mode)
    // the counter is requested with the staging loads, not one round trip after them
    const int64_t g0 = devgen ? *reinterpret_cast<volatile int64_t*>(S.gen_dev) : gen;
    // Without PDL or peers the population is final at entry: the chain's own row is requested now,
    // and every thread sends one 128-byte line of the population to L2 (all of it at config 2's
    // 4096 chains), where the partner rows, known only once the draws are taken, then hit.  (Not in
    // replay mode, a check against the reference's draws: there it would spill.)
    const bool early = !REPLAY && !pdl && S.X_peers == nullptr;
    double xv0[PCHUNK];
    if (early) {
        const int64_t at = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 128;
        if (at < S.nchains * S.nfree * 8)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(S.X) + at));
#pragma unroll
        for (int q = 0; q < PCHUNK; q++) xv0[q] = live && q < S.nfree ? S.X[c * S.nfree + q] : 0.0;
    }
    __shared__ double vbuf[STAGE_DOUBLES];
    stage_vectors<128>(S, vbuf);                     // constant during a run: safe before the wait
    Draws dr;
    double nrm[PCHUNK];                              // support draws of the first chunk of free parameters
    int64_t gspec = gen;
    if (!REPLAY) {
        if (devgen) {
            gspec = g0 + (pdl ? 1 : 0);
            zsize = S.M0 + (gspec / S.thinning) * S.nchains;
        }
        if (live) { chain_draws<false>(S, D, gspec, zsize, c, dr); chain_normals<false>(S, D, gspec, c, 0, nrm); }
    }
    if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
    if (devgen) {
        gen = pdl ? *reinterpret_cast<volatile int64_t*>(S.gen_dev) : g0;
        zsize = S.M0 + (gen / S.thinning) * S.nchains;
    }
    if (REPLAY) {
        if (live) { chain_draws<true>(S, D, gen, zsize, c, dr); chain_normals<true>(S, D, gen, c, 0, nrm); }
    } else if (gen != gspec && live) {
        chain_draws<false>(S, D, gen, zsize, c, dr);
        chain_normals<false>(S, D, gen, c, 0, nrm);
    }
    if (!REPLAY && S.F_peers) flags_wait(S, gen);    // every device has finished generation gen-1
    if (!live) return;
    propose_apply<REPLAY>(S, D, dr, nrm, gen, c, early, xv0);
}

__global__ void __launch_bounds__(128) k_metropolis(mc3b_sampler_t S, const double* partial, int64_t ldpartial, int nsplit,
                                                    int64_t c_off, int64_t gen, int64_t zrow0, int64_t c_begin,
                                                    int64_t c_end) {
    const int64_t c = c_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ double vbuf[STAGE_DOUBLES];
    stage_vectors<128>(S, vbuf);
    if (c >= c_end) return;
    if (gen < 0) {                                   // device-driven generation (graph mode)
        gen = *S.gen_dev;
        zrow0 = ((gen + 1) % S.thinning == 0) ? S.M0 + ((gen + 1) / S.thinning - 1) * S.nchains : -1;
    }
    const double nxt = S.inb[c] ? sum_partials<false>(partial, ldpartial, nsplit, c - c_off) : 0.0;
    metropolis_chain(S, nxt, gen, zrow0, c);
    if (S.X_peers) __threadfence_system();           // peer stores performed before the kernel ends (k_advance publishes)
}

__global__ void __launch_bounds__(128) k_init_trials(mc3b_sampler_t S, int kickoff, int64_t ntrials, int64_t round,
                                                     double* trial, int32_t* ok) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntrials) return;
    ok[t] = init_trial(S, kickoff, t, round, trial + t * S.npars);
}

__global__ void k_advance(mc3b_sampler_t S) {
    const int64_t g = *S.gen_dev + 1;
    *S.gen_dev = g;
    if (S.F_peers) flags_publish(S, g);              // k_metropolis (previous launch) has stored everywhere
}

// Report-point counters of this device's chains in ONE small buffer (one D2H per
// report instead of five): out = [sum naccept, best chisq, its generation, its
// chain, best x (nfree), outbounds (nfree)].  Best = lowest chi-squared, ties to
// the earlier (generation, chain) -- the order chain.py:268-274 would have met them.
__global__ void __launch_bounds__(256) k_pack_counters(mc3b_sampler_t S, double* out) {
    __shared__ double s_acc[256], s_chi[256];
    __shared__ long long s_gen[256], s_ch[256];
    const int t = threadIdx.x;
    double acc = 0.0, chi = INFINITY;
    long long gen = 0x7fffffffffffffffLL, ch = 0x7fffffffffffffffLL;
    auto better = [](double c1, long long g1, long long h1, double c2, long long g2, long long h2) {
        return c1 < c2 || (c1 == c2 && (g1 < g2 || (g1 == g2 && h1 < h2)));
    };
    for (int64_t c = S.chain0 + t; c < S.chain0 + S.nlocal; c += 256) {
        acc += (double)S.naccept[c];
        const double bc = S.best_chisq[c];
        if (better(bc, S.best_gen[c], c, chi, gen, ch)) { chi = bc; gen = S.best_gen[c]; ch = c; }
    }
    s_acc[t] = acc; s_chi[t] = chi; s_gen[t] = gen; s_ch[t] = ch;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (t < o) {
            s_acc[t] += s_acc[t + o];
            if (better(s_chi[t + o], s_gen[t + o], s_ch[t + o], s_chi[t], s_gen[t], s_ch[t])) {
                s_chi[t] = s_chi[t + o]; s_gen[t] = s_gen[t + o]; s_ch[t] = s_ch[t + o];
            }
        }
        __syncthreads();
    }
    const bool any = s_chi[0] < INFINITY;
    if (t == 0) {
        out[0] = s_acc[0];
        out[1] = s_chi[0];
        out[2] = any ? (double)s_gen[0] : -1.0;
        out[3] = any ? (double)s_ch[0] : -1.0;
    }
    if (t < S.nfree) {
        out[4 + t] = any ? S.best_x[s_ch[0] * S.nfree + t] : 0.0;
        out[4 + S.nfree + t] = (double)S.outbounds[t];
    }
}

// log_prior of history rows (mc3/stats/stats.py:367-392) and the data chi-squared
// it implies: lpr = -0.5 sum_j t_j^2 with t_j = (z-prior)/low|up for Gaussian
// priors (low, up > 0), t_j = 2 log z where priorlow < 0; chisq = -2 (log_post - lpr).
__global__ void __launch_bounds__(128) k_log_prior(const double* Z, int64_t nrows, int nfree, const int32_t* ifree,
                                                   const double* prior, const double* plo, const double* pup,
                                                   const double* log_post, double* lpr, double* chisq) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    double acc = 0.0;
    for (int j = 0; j < nfree; j++) {
        const int k = ifree[j];
        const double z = Z[r * nfree + j], lo = plo[k], up = pup[k];
        double t = 0.0;
        if (lo > 0.0 && up > 0.0) {
            const double d = z - prior[k];
            t = d < 0.0 ? d / lo : (d > 0.0 ? d / up : d);
        } else if (lo < 0.0) {
            t = 2.0 * log(z);
        }
        acc += t * t;
    }
    const double v = -0.5 * acc;
    if (lpr) lpr[r] = v;
    if (chisq) chisq[r] = -2.0 * (log_post[r] - v);
}

// ---- Gelman-Rubin ----------------------------------------------------------
// Stage 1: one thread per (chain, parameter): mean and population variance of
// its niter samples (two passes, as numpy's var).  Stage 2: one CTA, fixed-order
// sums over chains -> W, B, V, sqrt(V/W)   (gelman.py:75-92).
__global__ void __launch_bounds__(128) k_gr_stats(const double* Z, int64_t nfree, int64_t nchains, int64_t M0,
                                                  const int64_t* rows, int64_t ldr, int64_t burnin, int64_t niter,
                                                  int64_t c_begin, int64_t c_end, double* work) {
    const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t0 >= (c_end - c_begin) * nfree) return;
    const int64_t t = c_begin * nfree + t0;
    const int64_t c = t / nfree, p = t % nfree;
    auto at = [&](int64_t k) -> double {
        const int64_t row = rows ? rows[c * ldr + k] : M0 + k * nchains + c;
        return Z[row * nfree + p];
    };
    double s = 0.0;
    for (int64_t k = burnin; k < burnin + niter; k++) s += at(k);
    const double mu = s / (double)niter;
    double v = 0.0;
    for (int64_t k = burnin; k < burnin + niter; k++) { const double d = at(k) - mu; v += d * d; }
    work[t] = mu;
    work[nchains * nfree + t] = v / (double)niter;
}

__global__ void __launch_bounds__(256) k_gr_psrf(const double* work, int64_t nfree, int64_t nchains, int64_t niter,
                                                 double* psrf) {
    __shared__ double sh[256];
    const int p = blockIdx.x;
    const double* mu = work;
    const double* var = work + nchains * nfree;
    auto block_sum = [&](double v) -> double {
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
            __syncthreads();
        }
        const double r = sh[0];
        __syncthreads();
        return r;
    };
    double a = 0.0, b = 0.0;
    for (int64_t c = threadIdx.x; c < nchains; c += 256) { a += var[c * nfree + p]; b += mu[c * nfree + p]; }
    const double W = block_sum(a) / (double)nchains;
    const double mm = block_sum(b) / (double)nchains;
    double d2 = 0.0;
    for (int64_t c = threadIdx.x; c < nchains; c += 256) { const double d = mu[c * nfree + p] - mm; d2 += d * d; }
    const double B = (double)niter / ((double)nchains - 1.0) * block_sum(d2);
    if (threadIdx.x == 0) {
        const double V = W * (((double)niter - 1.0) / (double)niter) +
                         B * (((double)nchains + 1.0) / ((double)niter * (double)nchains));
        psrf[p] = sqrt(V / W);
    }
}

int check_sampler(const mc3b_sampler_t* s, int64_t c_begin, int64_t c_end) {
    MC3B_CHECK_ARG(s != nullptr, "null sampler");
    MC3B_CHECK_ARG(s->nfree > 0 && s->nfree <= MAXP && s->npars >= s->nfree && s->npars <= MAXP,
                   "nfree/npars out of range (max %d)", MAXP);
    MC3B_CHECK_ARG(c_begin >= s->chain0 && c_end <= s->chain0 + s->nlocal && c_begin <= c_end,
                   "chain range outside this device's slice");
    MC3B_CHECK_ARG(s->sampler == MC3B_MRW || s->sampler == MC3B_DEMC || s->sampler == MC3B_SNOOKER,
                   "unknown sampler %d", s->sampler);
    return MC3B_OK;
}

}  // namespace

extern "C" int mc3b_propose(const mc3b_sampler_t* s, int64_t gen, int64_t zsize, int64_t c_begin, int64_t c_end,
                            void* stream) {
    if (int rc = check_sampler(s, c_begin, c_end)) return rc;
    MC3B_CHECK_ARG(s->sampler != MC3B_DEMC || s->nchains >= 3, "demc needs at least 3 chains");
    MC3B_CHECK_ARG(gen >= 0 || (s->gen_dev && s->thinning > 0), "graph mode needs gen_dev and thinning");
    MC3B_CHECK_ARG(s->sampler != MC3B_SNOOKER || gen < 0 || zsize >= 2, "snooker needs at least 2 history rows");
    if (c_end == c_begin) return MC3B_OK;
    mc3b_draws_t none = {};
    // opt-in (MC3B_PDL=1): back-to-back proposal launches drop from 8.2 to 5.9 us, but inside
    // the captured generation graph the replay time did not change (192.9 vs 191.8 us at
    // config 2, profiles/r2_generation_breakdown.md), so the plain launch stays the default
    static const bool pdl = getenv("MC3B_PDL") && atoi(getenv("MC3B_PDL")) == 1;
    if (pdl) {                                       // programmatic dependent of the previous kernel
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)ceil_div64(c_end - c_begin, 128));
        cfg.blockDim = dim3(128);
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        MC3B_CUDA(cudaLaunchKernelEx(&cfg, k_propose<false>, *s, none, gen, zsize, c_begin, c_end, 1));
        return MC3B_OK;
    }
    k_propose<false><<<(unsigned)ceil_div64(c_end - c_begin, 128), 128, 0, (cudaStream_t)stream>>>(
        *s, none, gen, zsize, c_begin, c_end, 0);
    MC3B_CHECK_LAUNCH("k_propose");
    return MC3B_OK;
}

extern "C" int mc3b_propose_replay(const mc3b_sampler_t* s, const mc3b_draws_t* d, int64_t c_begin, int64_t c_end,
                                   void* stream) {
    if (int rc = check_sampler(s, c_begin, c_end)) return rc;
    MC3B_CHECK_ARG(d && d->normal && d->u, "replay draws missing");
    MC3B_CHECK_ARG(s->sampler == MC3B_MRW || (d->a && d->b), "replay partner indices missing");
    MC3B_CHECK_ARG(s->sampler != MC3B_SNOOKER || (d->iz && d->usj && d->gs), "replay snooker draws missing");
    if (c_end == c_begin) return MC3B_OK;
    k_propose<true><<<(unsigned)ceil_div64(c_end - c_begin, 128), 128, 0, (cudaStream_t)stream>>>(
        *s, *d, 0, 0, c_begin, c_end, 0);
    MC3B_CHECK_LAUNCH("k_propose<replay>");
    return MC3B_OK;
}

extern "C" int mc3b_metropolis(const mc3b_sampler_t* s, const double* partial, int64_t ldpartial, int nsplit,
                               int64_t c_off, int64_t gen, int64_t zrow0, int64_t c_begin, int64_t c_end,
                               void* stream) {
    if (int rc = check_sampler(s, c_begin, c_end)) return rc;
    MC3B_CHECK_ARG(partial && nsplit > 0 && c_off <= c_begin && ldpartial >= c_end - c_off, "bad partial workspace");
    MC3B_CHECK_ARG(gen >= 0 || (s->gen_dev && s->thinning > 0), "graph mode needs gen_dev and thinning");
    if (c_end == c_begin) return MC3B_OK;
    k_metropolis<<<(unsigned)ceil_div64(c_end - c_begin, 128), 128, 0, (cudaStream_t)stream>>>(
        *s, partial, ldpartial, nsplit, c_off, gen, zrow0, c_begin, c_end);
    MC3B_CHECK_LAUNCH("k_metropolis");
    return MC3B_OK;
}

extern "C" int mc3b_advance(const mc3b_sampler_t* s, void* stream) {
    MC3B_CHECK_ARG(s && s->gen_dev, "no device generation counter");
    k_advance<<<1, 1, 0, (cudaStream_t)stream>>>(*s);
    MC3B_CHECK_LAUNCH("k_advance");
    return MC3B_OK;
}

extern "C" int mc3b_pack_counters(const mc3b_sampler_t* s, double* out, void* stream) {
    MC3B_CHECK_ARG(s && out, "bad arguments");
    MC3B_CHECK_ARG(s->nfree > 0 && s->nfree <= MAXP, "nfree out of range");
    k_pack_counters<<<1, 256, 0, (cudaStream_t)stream>>>(*s, out);
    MC3B_CHECK_LAUNCH("k_pack_counters");
    return MC3B_OK;
}

extern "C" int mc3b_log_prior(const double* Z, int64_t nrows, int nfree, const int32_t* ifree, const double* prior,
                              const double* priorlow, const double* priorup, const double* log_post, double* lpr,
                              double* chisq, void* stream) {
    MC3B_CHECK_ARG(Z && ifree && prior && priorlow && priorup && nrows > 0 && nfree > 0, "bad arguments");
    MC3B_CHECK_ARG((lpr || chisq) && (!chisq || log_post), "need an output (chisq needs log_post)");
    k_log_prior<<<(unsigned)ceil_div64(nrows, 128), 128, 0, (cudaStream_t)stream>>>(Z, nrows, nfree, ifree, prior,
                                                                                     priorlow, priorup, log_post,
                                                                                     lpr, chisq);
    MC3B_CHECK_LAUNCH("k_log_prior");
    return MC3B_OK;
}

extern "C" int mc3b_init_trials(const mc3b_sampler_t* s, int kickoff, int64_t ntrials, int64_t round,
                                double* trial, int32_t* ok, void* stream) {
    MC3B_CHECK_ARG(s && trial && ok && ntrials > 0, "bad arguments");
    MC3B_CHECK_ARG(s->nfree > 0 && s->nfree <= MAXP && s->npars <= MAXP, "nfree/npars out of range");
    MC3B_CHECK_ARG(kickoff == 0 || kickoff == 1, "kickoff must be 0 (normal) or 1 (uniform)");
    k_init_trials<<<(unsigned)ceil_div64(ntrials, 128), 128, 0, (cudaStream_t)stream>>>(*s, kickoff, ntrials, round,
                                                                                        trial, ok);
    MC3B_CHECK_LAUNCH("k_init_trials");
    return MC3B_OK;
}

extern "C" int mc3b_gelman_rubin_moments(const double* Z, int64_t nfree, int64_t nchains, int64_t M0,
                                         const int64_t* rows, int64_t ldr, int64_t burnin, int64_t niter,
                                         int64_t c_begin, int64_t c_end, double* work, void* stream) {
    MC3B_CHECK_ARG(Z && work && nfree > 0 && nchains > 1 && niter > 0 && burnin >= 0, "bad arguments");
    MC3B_CHECK_ARG(c_begin >= 0 && c_begin <= c_end && c_end <= nchains, "bad chain range");
    if (c_end == c_begin) return MC3B_OK;
    k_gr_stats<<<(unsigned)ceil_div64((c_end - c_begin) * nfree, 128), 128, 0, (cudaStream_t)stream>>>(
        Z, nfree, nchains, M0, rows, ldr, burnin, niter, c_begin, c_end, work);
    MC3B_CHECK_LAUNCH("k_gr_stats");
    return MC3B_OK;
}

extern "C" int mc3b_gelman_rubin_psrf(const double* work, int64_t nfree, int64_t nchains, int64_t niter,
                                      double* psrf, void* stream) {
    MC3B_CHECK_ARG(work && psrf && nfree > 0 && nchains > 1 && niter > 0, "bad arguments");
    k_gr_psrf<<<(unsigned)nfree, 256, 0, (cudaStream_t)stream>>>(work, nfree, nchains, niter, psrf);
    MC3B_CHECK_LAUNCH("k_gr_psrf");
    return MC3B_OK;
}

extern "C" int mc3b_gelman_rubin(const double* Z, int64_t nfree, int64_t nchains, int64_t M0, const int64_t* rows,
                                 int64_t ldr, int64_t burnin, int64_t niter, double* work, double* psrf,
                                 void* stream) {
    if (int rc = mc3b_gelman_rubin_moments(Z, nfree, nchains, M0, rows, ldr, burnin, niter, 0, nchains, work, stream))
        return rc;
    return mc3b_gelman_rubin_psrf(work, nfree, nchains, niter, psrf, stream);
}
