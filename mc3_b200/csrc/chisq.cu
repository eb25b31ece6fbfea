// mc3_b200 -- chi-squared family (replaces src_c/_chisq.c and the model +
// chi-squared half of Chain.eval_model, mc3/chain.py:302-340).
//
// The model + chi-squared kernel k_model_chisq and the model-value kernel live in
// chisq_kernel.cuh, which user models compiled at run time share (jit.cu); this file
// instantiates them for the built-in models, plans their launch shape and checks
// their arguments (mc3b_chisq_setup, used by both paths).
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <type_traits>
#include "chisq_kernel.cuh"

namespace {

// Shape policy: a pure function of (plan_chains, n, dtype, SM count).  plan_chains
// is the chain count the shape is planned FOR -- by default the chains of the
// launch; a caller that wants identical chi-squared bits however the chains are
// spread over launches or devices plans for the whole population and launches any
// subset of it with that plan (the split boundaries, hence the order in which a
// chain's terms are added, then do not depend on the subset).
// kind: MC3B_PLAN_GENERAL, or MC3B_PLAN_MOMENT for the sufficient-statistics kernel: it runs 4
// CTAs per SM and its CTAs are short, so its waves are planned for 4 and its splits shrink
// more slowly and stop at 8 tiles (measured at config 2: 0.0954 against 0.0985 ms; the same plan
// costs the other kernels 3-16 %, profiles/r2_plan_ab.txt).
// MC3B_PLAN_SPECTRAL: one thread per chain and no data stream, so one split.
Shape plan_shape(int64_t nchains, int64_t n, int dtype, int sms, int kind = MC3B_PLAN_GENERAL) {
    Shape s;
    if (kind == MC3B_PLAN_SPECTRAL) {
        s.lc = 32; s.nsplit = 1; s.nsched = 0;
        return s;
    }
    int RESIDENT = kind == MC3B_PLAN_MOMENT ? 4 : mc3b_chisq::RESIDENT;    // MC3B_PLAN_RESIDENT: experiments
    if (const char* e = getenv("MC3B_PLAN_RESIDENT")) RESIDENT = atoi(e) > 0 ? atoi(e) : RESIDENT;
    s.lc = nchains >= 96 ? 32 : (nchains >= 12 ? 8 : 1);
    const int tile = dtype == MC3B_F32 ? tilecfg<float>::TILE : tilecfg<double>::TILE;
    const int64_t groups = ceil_div64(nchains, (int64_t)WARPS * s.lc);
    const int64_t nfull = n / tile;
    int waves = 2;
    if (const char* e = getenv("MC3B_WAVES")) waves = atoi(e) > 0 ? atoi(e) : 1;
    // whole waves of RESIDENT CTAs per SM (round to nearest: a few CTAs over one
    // wave cost a whole extra wave, so round down unless clearly closer to the next)
    int64_t want = ((int64_t)sms * RESIDENT * waves) / groups;
    int64_t ns = want < 1 ? 1 : want;
    if (ns > nfull) ns = nfull;
    if (ns > MC3B_MAX_SPLIT) ns = MC3B_MAX_SPLIT;
    if (ns < 1) ns = 1;
    s.nsplit = (int)ns;
    s.nsched = 0;
    // Decreasing split sizes ("factoring"): CTAs are dispatched in split order, so the
    // last ones to start are short and the SMs run dry together.  Each batch of
    // ~one wave of splits takes 1/f of the tiles that remain.
    // f = 2, at least 4 tiles per split measured best at config 2 (0.203 -> 0.186 ms;
    // profiles/r1_split_schedule.md); MC3B_SCHED="f,min" overrides, "0" gives equal splits.
    double f = kind == MC3B_PLAN_MOMENT ? 1.5 : 2.0; int mn = kind == MC3B_PLAN_MOMENT ? 8 : 4;
    if (const char* e = getenv("MC3B_SCHED")) { f = 0.0; sscanf(e, "%lf,%d", &f, &mn); }
    if (mn < 1) mn = 1;
    if (f >= 1.0 && s.lc == 32 && nfull < (1 << 30) && ns >= 8) {
        const double rows = (double)sms * RESIDENT / (double)groups;
        const int per = (int)(rows + 0.999);
        int64_t R = nfull; int k = 0; bool fits = true;
        s.tstart[0] = 0;
        while (R > 0 && fits) {
            int64_t sz = (int64_t)((double)R / (f * rows) + 0.5);
            if (sz < mn) sz = mn;
            for (int j = 0; j < per && R > 0; j++) {
                const int64_t t = sz < R ? sz : R;
                if (k >= SCHED_MAX) { fits = false; break; }
                s.tstart[k + 1] = (int32_t)(s.tstart[k] + t);
                k++; R -= t;
            }
        }
        if (fits && k >= 1) { s.nsched = k; s.nsplit = k; }
    }
    return s;
}

template <class M, typename T, bool USIG>
int launch_model_chisq(const Shape& sh, const ChisqArgs<T>& a, dim3 grid, cudaStream_t st) {
    dim3 block(WARPS * 32);
    if (sh.lc == 32) k_model_chisq<M, T, 32, 1, USIG><<<grid, block, 0, st>>>(a);
    else if (sh.lc == 8) k_model_chisq<M, T, 8, 1, USIG><<<grid, block, 0, st>>>(a);
    else k_model_chisq<M, T, 1, 1, USIG><<<grid, block, 0, st>>>(a);
    MC3B_CHECK_LAUNCH("k_model_chisq");
    return MC3B_OK;
}

template <typename T>
int model_chisq_t(int model_id, const double* params, int64_t ldp, int64_t nchains, int nmodel,
                  const void* x, const void* d, const void* w, int64_t n, double* partial, int64_t ldpartial,
                  int nsplit, int dtype, const mc3b_chisq_opts_t& o, cudaStream_t st) {
    ChisqArgs<T> A;
    Shape sh;
    dim3 grid;
    const int rc = mc3b_chisq_setup<T>(params, ldp, nchains, x, d, w, n, partial, ldpartial, nsplit, dtype, o, A, sh,
                                       grid);
    if (rc != MC3B_OK) return rc;
    const bool usig = o.uniform_sigma != 0;
    const unsigned groups = grid.x;
    dim3 block(WARPS * 32);
    if (model_id == MC3B_MODEL_SINUSOID_GRID) {
        if constexpr (std::is_same<T, double>::value) {
            if (sh.lc == 32 && A.use_tma && n >= 2) {
                if (o.tile_x != nullptr) {
                    MC3B_CHECK_ARG(o.dx != 0.0 && o.ntiles >= 0 && o.ntiles * 128 <= n, "tile_x needs dx and ntiles <= n/128");
                    A.xt = o.tile_x; A.dxg = o.dx; A.ntiles = o.ntiles;
                }
                MC3B_CHECK_ARG(o.moment == nullptr || !o.moment->record || o.moment->guard_hits,
                               "a guard record ring needs guard_hits");
                if (usig && o.moment != nullptr && o.moment->spectral != nullptr) {
                    const mc3b_spectral_t& s = *o.moment->spectral;
                    MC3B_CHECK_ARG(s.table && (((uintptr_t)s.table) & 15) == 0 && s.n1 > 0 && s.n2 > 0 &&
                                   (s.order == 9 || s.order == 15) && s.delta > 0.0 && o.moment->amp_max > 0.0,
                                   "bad spectral table");
                    A.m.c0ref = o.moment->c0ref; A.m.slref = o.moment->slref; A.m.d2tot = o.moment->d2tot;
                    A.m.amp_max = o.moment->amp_max; A.m.guard_hits = o.moment->guard_hits;
                    A.m.xlo = o.moment->xlo; A.m.xhi = o.moment->xhi; A.m.record = o.moment->record;
                    A.m.spec = s.table; A.m.sw1 = s.w1; A.m.sw2 = s.w2; A.m.sdelta = s.delta; A.m.sxc = s.xc;
                    A.m.sn1 = s.n1; A.m.sn2 = s.n2; A.m.sorder = s.order;
                    return mc3b_launch_spectral_chisq(A, (unsigned)groups, st);
                }
                if (usig && o.moment != nullptr) {
                    MC3B_CHECK_ARG(o.work, "the moment form needs the constants workspace (work)");
                    MC3B_CHECK_ARG(o.moment->folded && o.moment->tiles && o.moment->amp_max > 0.0 &&
                                   (((uintptr_t)o.moment->folded | (uintptr_t)o.moment->tiles) & 31) == 0,
                                   "bad moment data");
                    A.m.folded = o.moment->folded; A.m.tiles = o.moment->tiles;
                    A.m.c0ref = o.moment->c0ref; A.m.slref = o.moment->slref; A.m.d2tot = o.moment->d2tot;
                    A.m.amp_max = o.moment->amp_max; A.m.guard_hits = o.moment->guard_hits;
                    A.m.xlo = o.moment->xlo; A.m.xhi = o.moment->xhi; A.m.layout = o.moment->layout;
                    A.m.record = o.moment->record;
                    MC3B_CHECK_ARG(A.m.layout == 0 || A.m.layout == 1, "bad moment layout %d", A.m.layout);
                    return mc3b_launch_sinefold(A, (double*)o.work, (unsigned)groups, (unsigned)nsplit, st);
                }
                if (usig && A.fold != nullptr && ((uintptr_t)A.fold & 15) == 0)
                    return mc3b_launch_sinefold(A, (double*)o.work, (unsigned)groups, (unsigned)nsplit, st);
                if (!getenv("MC3B_OLD_GRID"))
                    return mc3b_launch_sinegrid(A, usig, (unsigned)groups, (unsigned)nsplit, st);
                if (!usig) {                        // round-1 kernel, kept for A/B measurements
                    k_model_chisq<SineGridModel, double, 32, 1, false><<<grid, block, 0, st>>>(A);
                    MC3B_CHECK_LAUNCH("k_model_chisq<grid>");
                    return MC3B_OK;
                }
            }
        }
        model_id = MC3B_MODEL_SINUSOID;             // small populations, fp32, unaligned: plain model
    }
    if (usig) { MC3B_DISPATCH_MODEL(T, model_id, nmodel, return (launch_model_chisq<M, T, true>(sh, A, grid, st))); }
    else { MC3B_DISPATCH_MODEL(T, model_id, nmodel, return (launch_model_chisq<M, T, false>(sh, A, grid, st))); }
    return MC3B_OK;
}

// ---- sum of partials + priors ----------------------------------------------
__global__ void k_chisq_finish(const double* partial, int64_t ldpartial, int nsplit, int64_t nchains, const double* params,
                               int64_t ldp, int npars, const double* prior, const double* plo,
                               const double* pup, double* chisq) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    double acc = 0.0;
    for (int s = 0; s < nsplit; s++) acc += partial[(int64_t)s * ldpartial + c];
    if (prior != nullptr) {
        double pr = 0.0;
        for (int j = 0; j < npars; j++) {
            const double lo = plo[j], up = pup[j];
            if (lo > 0.0 && up > 0.0) {
                const double off = params[c * ldp + j] - prior[j];
                const double t = off / (off > 0.0 ? up : lo);
                pr += t * t;
            }
        }
        acc += pr;
    }
    chisq[c] = acc;
}

// ---- chi-squared of given models (user callables): HBM-bound ---------------
// One CTA per chain row; 256 threads stride the row (coalesced 8-byte loads),
// fixed-order reduction (lane tree, then warps in order).
__global__ void __launch_bounds__(256) k_chisq_rows(const double* model, int64_t ldm, const double* data,
                                                    const double* uncert, int64_t n, double* chisq) {
    const double* m = model + (int64_t)blockIdx.x * ldm;
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 256) {
        const double r = (m[i] - data[i]) / uncert[i];
        acc = fma(r, r, acc);
    }
    __shared__ double ws[8];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < 8; k++) t += ws[k];
        chisq[blockIdx.x] = t;
    }
}

__global__ void k_residuals(const double* model, const double* data, const double* uncert, int64_t n,
                            const double* off, const double* low, const double* up, int64_t np, double* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (model[i] - data[i]) / uncert[i];
    else if (i < n + np) {
        const int64_t k = i - n;
        out[i] = off[k] / (off[k] > 0.0 ? up[k] : low[k]);
    }
}

}  // namespace

// Argument block, launch shape and argument checks of one model + chi-squared launch:
// the part shared by the built-in models (above) and user models (jit.cu).
template <typename T>
int mc3b_chisq_setup(const double* params, int64_t ldp, int64_t nchains, const void* x, const void* d, const void* w,
                     int64_t n, double* partial, int64_t ldpartial, int nsplit, int dtype, const mc3b_chisq_opts_t& o,
                     ChisqArgs<T>& A, Shape& sh, dim3& grid) {
    A.params = params; A.ldp = ldp; A.nchains = nchains;
    A.x = (const T*)x; A.d = (const T*)d; A.w = (const T*)w; A.fold = (const T*)o.folded; A.consts = nullptr; A.ldc = 0; A.consts_wait = 0; A.m = MomentArgs{}; A.n = n;
    A.xt = nullptr; A.dxg = 0.0; A.ntiles = 0; A.partial = partial; A.ldpartial = ldpartial;
    A.xs[0] = (const T*)x;
    for (int j = 1; j < MC3B_MAX_INPUTS; j++) A.xs[j] = nullptr;
    A.uconst = nullptr; A.uconst_pad = nullptr;
    const bool usig = o.uniform_sigma != 0;
    A.use_tma = ((((uintptr_t)x | (uintptr_t)d | (usig ? 0 : (uintptr_t)w)) & 15) == 0) ? 1 : 0;
    const int64_t plan_chains = o.plan_chains > 0 ? o.plan_chains : nchains;
    MC3B_CHECK_ARG(plan_chains >= nchains, "plan_chains (%lld) is smaller than the launch (%lld chains)",
                   (long long)plan_chains, (long long)nchains);
    sh = plan_shape(plan_chains, n, dtype, mc3b_sm_count(),
                    o.moment != nullptr && usig ? (o.moment->spectral ? MC3B_PLAN_SPECTRAL : MC3B_PLAN_MOMENT)
                                                : MC3B_PLAN_GENERAL);
    A.nsched = sh.nsched;
    if (sh.nsched > 0) memcpy(A.tstart, sh.tstart, sizeof(int32_t) * (sh.nsched + 1));
    MC3B_CHECK_ARG(nsplit == sh.nsplit, "nsplit %d does not match the plan (%d)", nsplit, sh.nsplit);
    const int64_t groups = ceil_div64(nchains, (int64_t)WARPS * sh.lc);
    MC3B_CHECK_ARG(groups <= 0x7fffffff, "too many chains for one launch");
    A.f.on = 0;
    if (o.fuse != nullptr) {
        MC3B_CHECK_ARG(o.fuse_done != nullptr && ((uintptr_t)o.fuse_done & 7) == 0,
                       "the fused Metropolis epilogue needs its counters (fuse_done, 8-byte aligned)");
        MC3B_CHECK_ARG(o.gen >= 0 || (o.fuse->gen_dev && o.fuse->thinning > 0),
                       "device-driven generations need gen_dev and thinning");
        MC3B_CHECK_ARG(!o.advance || o.fuse->gen_dev, "advance needs gen_dev");
        MC3B_CHECK_ARG(o.c_off >= o.fuse->chain0 && o.c_off + nchains <= o.fuse->chain0 + o.fuse->nlocal,
                       "chain range outside this device's slice");
        A.f.on = 1; A.f.advance = o.advance; A.f.done = o.fuse_done; A.f.c_off = o.c_off;
        A.f.gen = o.gen; A.f.zrow0 = o.zrow0; A.f.S = *o.fuse;
    }
    grid = dim3((unsigned)groups, (unsigned)nsplit);
    return MC3B_OK;
}
template int mc3b_chisq_setup<double>(const double*, int64_t, int64_t, const void*, const void*, const void*, int64_t,
                                      double*, int64_t, int, int, const mc3b_chisq_opts_t&, ChisqArgs<double>&, Shape&,
                                      dim3&);
template int mc3b_chisq_setup<float>(const double*, int64_t, int64_t, const void*, const void*, const void*, int64_t,
                                     double*, int64_t, int, int, const mc3b_chisq_opts_t&, ChisqArgs<float>&, Shape&,
                                     dim3&);

extern "C" int mc3b_model_chisq_plan_kind(int kind, int64_t nchains, int64_t n, int dtype, int* nsplit) {
    MC3B_CHECK_ARG(nchains > 0 && n > 0 && nsplit != nullptr, "bad plan arguments");
    MC3B_CHECK_ARG(dtype == MC3B_F64 || dtype == MC3B_F32, "bad dtype %d", dtype);
    MC3B_CHECK_ARG(kind == MC3B_PLAN_GENERAL || kind == MC3B_PLAN_MOMENT || kind == MC3B_PLAN_SPECTRAL,
                   "bad plan kind %d", kind);
    int sms = mc3b_sm_count();
    if (sms <= 0) sms = 148;        // planning without a device (CPU-side sizing)
    *nsplit = plan_shape(nchains, n, dtype, sms, kind).nsplit;
    return MC3B_OK;
}

extern "C" int mc3b_model_chisq_plan(int64_t nchains, int64_t n, int dtype, int* nsplit) {
    return mc3b_model_chisq_plan_kind(MC3B_PLAN_GENERAL, nchains, n, dtype, nsplit);
}

extern "C" int mc3b_model_chisq_splits(int64_t nchains, int64_t n, int dtype, int64_t* point_start, int cap,
                                       int* nsplit) {
    MC3B_CHECK_ARG(nchains > 0 && n > 0 && nsplit != nullptr && point_start != nullptr, "bad plan arguments");
    MC3B_CHECK_ARG(dtype == MC3B_F64 || dtype == MC3B_F32, "bad dtype %d", dtype);
    int sms = mc3b_sm_count();
    if (sms <= 0) sms = 148;
    const Shape sh = plan_shape(nchains, n, dtype, sms);
    MC3B_CHECK_ARG(cap >= sh.nsplit + 1, "point_start holds %d entries, the plan needs %d", cap, sh.nsplit + 1);
    const int64_t tile = dtype == MC3B_F32 ? tilecfg<float>::TILE : tilecfg<double>::TILE;
    const int64_t nfull = n / tile;
    for (int y = 0; y <= sh.nsplit; y++)
        point_start[y] = tile * (sh.nsched > 0 ? (int64_t)sh.tstart[y] : nfull * y / sh.nsplit);
    point_start[sh.nsplit] = n;                       // the ragged tail belongs to the last split
    *nsplit = sh.nsplit;
    return MC3B_OK;
}

extern "C" int mc3b_model_chisq_ex(int model_id, int dtype, const double* params, int64_t ldp, int64_t nchains,
                                   int nmodel, const void* x, const void* data, const void* invsig, int64_t n,
                                   double* partial, int64_t ldpartial, int nsplit, const mc3b_chisq_opts_t* opts,
                                   void* stream) {
    MC3B_CHECK_ARG(params && x && data && invsig && partial, "null pointer");
    MC3B_CHECK_ARG(ldpartial >= nchains, "ldpartial < nchains");
    MC3B_CHECK_ARG(nchains > 0 && n > 0 && nmodel > 0 && nmodel <= ldp, "bad sizes");
    MC3B_CHECK_ARG(mc3b_model_nparams(model_id, nmodel) == nmodel, "model %d does not take %d parameters",
                   model_id, nmodel);
    mc3b_chisq_opts_t o = {};
    if (opts) o = *opts;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MC3B_F64)
        return model_chisq_t<double>(model_id, params, ldp, nchains, nmodel, x, data, invsig, n, partial, ldpartial,
                                     nsplit, dtype, o, st);
    if (dtype == MC3B_F32)
        return model_chisq_t<float>(model_id, params, ldp, nchains, nmodel, x, data, invsig, n, partial, ldpartial,
                                    nsplit, dtype, o, st);
    mc3b_set_error("bad dtype %d", dtype);
    return MC3B_ERR_ARG;
}

extern "C" int mc3b_fold_data(const double* data, int64_t n, double* out, void* stream) {
    MC3B_CHECK_ARG(data && out && n > 0, "bad fold arguments");
    return mc3b_launch_fold(data, n, out, (cudaStream_t)stream);
}

extern "C" int mc3b_moment_finish(const mc3b_moment_t* m, const double* partial, int64_t ldpartial, int nsplit,
                                  int64_t nchains, const double* params, int64_t ldp, int npars, const double* x,
                                  const double* data, const double* invsig, int64_t n, const double* prior,
                                  const double* priorlow, const double* priorup, double* chisq, void* stream) {
    MC3B_CHECK_ARG(m && partial && params && x && data && invsig && chisq, "null pointer");
    MC3B_CHECK_ARG(nchains > 0 && nsplit > 0 && n > 0 && ldpartial >= nchains && ldp >= 5 && m->amp_max > 0.0,
                   "bad moment_finish arguments");
    MC3B_CHECK_ARG(prior == nullptr || (priorlow && priorup && npars > 0 && npars <= ldp), "bad prior arguments");
    ChisqArgs<double> A = {};
    A.params = params; A.ldp = ldp; A.nchains = nchains; A.x = x; A.d = data; A.w = invsig; A.n = n;
    A.partial = const_cast<double*>(partial); A.ldpartial = ldpartial;
    A.m.folded = m->folded; A.m.tiles = m->tiles; A.m.c0ref = m->c0ref; A.m.slref = m->slref;
    A.m.d2tot = m->d2tot; A.m.amp_max = m->amp_max; A.m.xlo = m->xlo; A.m.xhi = m->xhi; A.m.guard_hits = m->guard_hits;
    return mc3b_launch_moment_finish(A, nsplit, npars, prior, priorlow, priorup, chisq, (cudaStream_t)stream);
}

extern "C" int mc3b_moment_prepare(const double* data, int64_t ntiles, double x0, double dx, const double* tile_x,
                                   double c0ref, double slref, int layout, double* folded, double* tiles, void* stream) {
    MC3B_CHECK_ARG(data && folded && tiles && ntiles >= 0, "bad moment_prepare arguments");
    MC3B_CHECK_ARG(layout == 0 || layout == 1, "bad moment layout %d", layout);
    MC3B_CHECK_ARG((((uintptr_t)tiles) & 31) == 0, "tiles must be 32-byte aligned");
    return mc3b_launch_moment_prepare(data, ntiles, x0, dx, tile_x, c0ref, slref, folded, tiles, layout, (cudaStream_t)stream);
}

extern "C" int mc3b_spectral_size(int n1, int n2, int order, int64_t* ndoubles) {
    MC3B_CHECK_ARG(n1 > 0 && n2 > 0 && (order == 9 || order == 15) && ndoubles, "bad spectral_size arguments");
    *ndoubles = MC3B_SPECTRAL_HEAD + 2 * ((int64_t)n1 * (2 * order + 3) + (int64_t)n2 * (order + 1));
    return MC3B_OK;
}

extern "C" int mc3b_spectral_prepare(const double* x, const double* data, int64_t n, double c0ref, double slref,
                                     const mc3b_spectral_t* s, void* stream) {
    MC3B_CHECK_ARG(x && data && s && s->table && n > 0, "bad spectral_prepare arguments");
    MC3B_CHECK_ARG(s->n1 > 0 && s->n2 > 0 && (int64_t)s->n1 + s->n2 < 0x7fffffff && (s->order == 9 || s->order == 15) &&
                   s->delta > 0.0, "bad spectral table description");
    return mc3b_launch_spectral_prepare(x, data, n, c0ref, slref, *s, (cudaStream_t)stream);
}

extern "C" int mc3b_model_chisq(int model_id, int dtype, const double* params, int64_t ldp, int64_t nchains,
                                int nmodel, const void* x, const void* data, const void* invsig, int64_t n,
                                double* partial, int64_t ldpartial, int nsplit, void* stream) {
    return mc3b_model_chisq_ex(model_id, dtype, params, ldp, nchains, nmodel, x, data, invsig, n, partial,
                               ldpartial, nsplit, nullptr, stream);
}

extern "C" int mc3b_model_eval(int model_id, const double* params, int64_t ldp, int64_t nchains, int nmodel,
                               const double* x, int64_t n, double* out, void* stream) {
    if (model_id == MC3B_MODEL_SINUSOID_GRID) model_id = MC3B_MODEL_SINUSOID;
    MC3B_CHECK_ARG(params && x && out && nchains > 0 && n > 0, "bad arguments");
    MC3B_CHECK_ARG(mc3b_model_nparams(model_id, nmodel) == nmodel, "model %d does not take %d parameters",
                   model_id, nmodel);
    MC3B_CHECK_ARG(nchains <= 65535, "model_eval is for small batches (<= 65535 rows)");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t bx = ceil_div64(n, 256);
    if (bx > 1184) bx = 1184;
    dim3 grid((unsigned)bx, (unsigned)nchains);
    MC3B_DISPATCH_MODEL(double, model_id, nmodel, (k_model_eval<M><<<grid, 256, 0, st>>>(params, ldp, x, n, out)));
    MC3B_CHECK_LAUNCH("k_model_eval");
    return MC3B_OK;
}

extern "C" int mc3b_chisq_finish(const double* partial, int64_t ldpartial, int nsplit, int64_t nchains, const double* params,
                                 int64_t ldp, int npars, const double* prior, const double* priorlow,
                                 const double* priorup, double* chisq, void* stream) {
    MC3B_CHECK_ARG(partial && chisq && nsplit > 0 && nchains > 0, "bad arguments");
    MC3B_CHECK_ARG(prior == nullptr || (params && priorlow && priorup), "priors need params, priorlow, priorup");
    k_chisq_finish<<<(unsigned)ceil_div64(nchains, 128), 128, 0, (cudaStream_t)stream>>>(
        partial, ldpartial, nsplit, nchains, params, ldp, npars, prior, priorlow, priorup, chisq);
    MC3B_CHECK_LAUNCH("k_chisq_finish");
    return MC3B_OK;
}

extern "C" int mc3b_chisq_batch(const double* model, int64_t ldm, int64_t nchains, const double* data,
                                const double* uncert, int64_t n, double* chisq, void* stream) {
    MC3B_CHECK_ARG(model && data && uncert && chisq && nchains > 0 && n > 0 && ldm >= n, "bad arguments");
    k_chisq_rows<<<(unsigned)nchains, 256, 0, (cudaStream_t)stream>>>(model, ldm, data, uncert, n, chisq);
    MC3B_CHECK_LAUNCH("k_chisq_rows");
    return MC3B_OK;
}

extern "C" int mc3b_residuals(const double* model, const double* data, const double* uncert, int64_t n,
                              const double* off, const double* low, const double* up, int64_t np, double* out,
                              void* stream) {
    MC3B_CHECK_ARG(model && data && uncert && out && n > 0, "bad arguments");
    if (off == nullptr) np = 0;
    k_residuals<<<(unsigned)ceil_div64(n + np, 256), 256, 0, (cudaStream_t)stream>>>(model, data, uncert, n, off,
                                                                                      low, up, np, out);
    MC3B_CHECK_LAUNCH("k_residuals");
    return MC3B_OK;
}
