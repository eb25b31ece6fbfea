// mc3_b200 -- the fused model + chi-squared kernel and the model-value kernel.
// Device code only: chisq.cu instantiates them for the built-in models, jit.cu has
// NVRTC instantiate them for a user model (the header travels inside the library as
// a string, csrc/jit_headers.inc written by build.py).  One kernel for both.
//
// k_model_chisq is the hot kernel of the sampler: one launch evaluates the
// model and the data chi-squared of EVERY chain of the population.
//
//   grid  = (chain groups, data splits); block = 4 warps.
//   warp  = LC chains x LP = 32/LC point lanes.  LC = 32: one chain per lane,
//           every lane walks all points of a tile (shared-memory broadcast);
//           LC = 8 / 1: fewer chains, lanes share the points of the tile.
//   data  = x, data, 1/sigma tiles of TILE points (and the tiles of inputs 2..NX
//           of a user model of several inputs), staged into shared memory
//           by 1-D TMA bulk copies (cp.async.bulk + mbarrier, 3 stages), so a
//           tile is fetched once per CTA and serves all its chains; the
//           per-chain constants live in registers for the whole launch.
//   sum   = per lane in registers, then a fixed-order xor-shuffle over the
//           point lanes, one partial per (split, chain): deterministic.
//
// Bound: FP64 (or FP32) pipe -- nchains*F flops per 24 bytes of data.
#pragma once
#include "models.cuh"
#include "sampler_dev.cuh"

#include "chisq_args.cuh"

// NVRTC: a named namespace, so that the instantiations have names the loader can
// look up (jit.cu); the library keeps them local to chisq.cu.
#ifdef __CUDACC_RTC__
namespace mc3b_jit {
#else
namespace {
#endif

// USIG: one uncertainty for all points (w[0]): residuals are plain differences
// (a two-register DADD instead of a multiply or a three-register FMA) and the sum
// is scaled by w[0]^2 once per partial.
template <class M, typename T, int LC, int CPT, bool USIG>
__global__ void __launch_bounds__(WARPS * 32, (CPT == 2 ? MC3B_RESIDENT2 : RESIDENT)) k_model_chisq(ChisqArgs<T> a) {
    constexpr int TILE = tilecfg<T>::TILE;
    constexpr int LP = 32 / LC;
    constexpr int NX = ninputs_of<M>::value;
    static_assert(NX >= 1 && NX <= MC3B_MAX_INPUTS && (NX == 1 || (!M::GUARD && !M::TILE_STATE)),
                  "models of several inputs have neither guard nor tile state");
    asm volatile("griddepcontrol.launch_dependents;");   // the next proposal kernel may start its draws
    __shared__ __align__(128) T sx[STAGES][TILE];
    __shared__ __align__(128) T sd[STAGES][TILE];
    __shared__ __align__(128) T sw[STAGES][TILE];
    __shared__ __align__(8) uint64_t bar[STAGES];
    // inputs 2..NX: declared only for a model of several inputs (as sdw for PM below)
    __shared__ __align__(128) T sxe[NX > 1 ? STAGES : 1][NX > 1 ? NX - 1 : 1][NX > 1 ? TILE : 2];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lc = lane % LC, lp = lane / LC;
    const int64_t cbase = ((int64_t)blockIdx.x * WARPS + warp) * (LC * CPT) + lc;

    M mdl[CPT];
#pragma unroll
    for (int k = 0; k < CPT; k++) {
        int64_t c = cbase + (int64_t)k * LC;
        if (c >= a.nchains) c = a.nchains - 1;      // idle lanes shadow the last chain
        if constexpr (M::TILE_STATE) {
            const double dx = ((double)a.x[a.n - 1] - (double)a.x[0]) / (double)(a.n - 1);
            mdl[k].load(a.params + c * a.ldp, dx, TILE);
        } else if constexpr (takes_consts<M>::value) {
            mdl[k].load(a.params + c * a.ldp, a.uconst);
        } else {
            mdl[k].load(a.params + c * a.ldp);
        }
    }
    double acc[CPT];
#pragma unroll
    for (int k = 0; k < CPT; k++) acc[k] = 0.0;

    // Tiles of this split: balanced contiguous ranges of FULL tiles; the
    // ragged tail (n % TILE points) belongs to the last split.
    const int64_t nfull = a.n / TILE;
    int64_t tb, te;
    if (a.nsched > 0) { tb = a.tstart[blockIdx.y]; te = a.tstart[blockIdx.y + 1]; }
    else { tb = nfull * blockIdx.y / gridDim.y; te = nfull * (blockIdx.y + 1) / gridDim.y; }
    const int64_t nt = te - tb;

    if (a.use_tma) {
        if (threadIdx.x == 0) {
            for (int s = 0; s < STAGES; s++) mbar_init(&bar[s], 1);
            mbar_fence_init();
        }
        __syncthreads();
        auto issue = [&](int64_t t, int s) {
            const int64_t off = t * TILE;
            mbar_expect_tx(&bar[s], ((USIG ? 2u : 3u) + (unsigned)(NX - 1)) * TILE * sizeof(T));
            bulk_g2s(sx[s], a.x + off, TILE * sizeof(T), &bar[s]);
            bulk_g2s(sd[s], a.d + off, TILE * sizeof(T), &bar[s]);
            if constexpr (!USIG) bulk_g2s(sw[s], a.w + off, TILE * sizeof(T), &bar[s]);
            if constexpr (NX > 1) {
#pragma unroll
                for (int j = 0; j < NX - 1; j++) bulk_g2s(sxe[s][j], a.xs[j + 1] + off, TILE * sizeof(T), &bar[s]);
            }
        };
        if (threadIdx.x == 0)
            for (int s = 0; s < STAGES && s < nt; s++) issue(tb + s, s);
        constexpr bool PM = premul_of<M>::value && !USIG;
        // PM keeps d/sigma in a buffer of its own: TMA never writes it, so no generic-proxy
        // store ever meets an async-proxy refill of the same bytes (no proxy fence needed)
        __shared__ __align__(128) T sdw[PM ? STAGES : 1][PM ? TILE : 2];
        // PM: data tile <- data / sigma, once for all chains of the CTA.  Tile it+1 is
        // scaled at the end of tile it, so that the stage-release barrier publishes it.
        auto premul = [&](int64_t t) {
            const int s1 = (int)(t % STAGES);
            mbar_wait(&bar[s1], (uint32_t)((t / STAGES) & 1));
            for (int i = threadIdx.x; i < TILE; i += WARPS * 32) sdw[PM ? s1 : 0][PM ? i : 0] = sd[s1][i] * sw[s1][i];
        };
        if constexpr (PM) {
            if (nt > 0) premul(0);
            __syncthreads();
        }
        for (int64_t it = 0; it < nt; it++) {
            const int s = (int)(it % STAGES);
            if constexpr (!PM) mbar_wait(&bar[s], (uint32_t)((it / STAGES) & 1));
            constexpr int U = 4;                // points in flight per lane
            static_assert(TILE % (U * LP) == 0, "tile must hold whole groups");
            if constexpr (M::TILE_STATE) {
                static_assert(LP == 1, "stateful models walk a tile in order: one chain per lane");
#pragma unroll
                for (int k = 0; k < CPT; k++) mdl[k].begin_tile((double)sx[s][0], TILE);
            }
            T tacc[CPT], uacc[CPT][U];          // one accumulator per point slot: no serial tail
#pragma unroll
            for (int k = 0; k < CPT; k++) {
#pragma unroll
                for (int u = 0; u < U; u++) uacc[k][u] = (T)0;
            }
#pragma unroll(LOOP_UNROLL)
            for (int i = lp; i < TILE; i += U * LP) {
                T x[U], y[U];
#pragma unroll
                for (int u = 0; u < U; u++) x[u] = sx[s][i + u * LP];
                T xv[NX][U];                    // NX > 1: every input of the U points
                if constexpr (NX > 1) {
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        xv[0][u] = x[u];
#pragma unroll
                        for (int j = 1; j < NX; j++) xv[j][u] = sxe[s][j - 1][i + u * LP];
                    }
                }
#pragma unroll
                for (int k = 0; k < CPT; k++) {
                    if constexpr (NX == 1) eval_points<M, T, U>(mdl[k], x, y, 0);
                    else eval_points<M, T, NX, U>(mdl[k], xv, y);
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const T r = USIG ? y[u] - sd[s][i + u * LP]
                                    : PM ? fma(y[u], sw[s][i + u * LP], -sdw[PM ? s : 0][PM ? i + u * LP : 0])
                                         : (y[u] - sd[s][i + u * LP]) * sw[s][i + u * LP];
                        uacc[k][u] = fma(r, r, uacc[k][u]);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < CPT; k++) tacc[k] = (uacc[k][0] + uacc[k][1]) + (uacc[k][2] + uacc[k][3]);
            if constexpr (M::GUARD) {           // extreme model arguments: redo the tile safely
#pragma unroll
                for (int k = 0; k < CPT; k++) {
                    if (mdl[k].flagged()) {
                        mdl[k].clear();
                        tacc[k] = (T)0;
                        for (int i = lp; i < TILE; i += LP) {
                            const T r = USIG ? mdl[k].eval_safe(sx[s][i]) - sd[s][i]
                                        : PM ? fma(mdl[k].eval_safe(sx[s][i]), sw[s][i], -sdw[PM ? s : 0][PM ? i : 0])
                                             : (mdl[k].eval_safe(sx[s][i]) - sd[s][i]) * sw[s][i];
                            tacc[k] = fma(r, r, tacc[k]);
                        }
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < CPT; k++) acc[k] += (double)tacc[k];
            if constexpr (PM) {
                if (it + 1 < nt) premul(it + 1);
            }
            __syncthreads();                    // everyone is done reading stage s
            if (threadIdx.x == 0 && it + STAGES < nt) issue(tb + it + STAGES, s);
        }
    } else {
        for (int64_t it = 0; it < nt; it++) {   // unaligned inputs: plain staged loads
            const int64_t off = (tb + it) * TILE;
            __syncthreads();
            for (int i = threadIdx.x; i < TILE; i += WARPS * 32) {
                sx[0][i] = a.x[off + i]; sd[0][i] = a.d[off + i]; sw[0][i] = USIG ? (T)1 : a.w[off + i];
                if constexpr (NX > 1) {
#pragma unroll
                    for (int j = 0; j < NX - 1; j++) sxe[0][j][i] = a.xs[j + 1][off + i];
                }
            }
            __syncthreads();
            T tacc[CPT];
#pragma unroll
            for (int k = 0; k < CPT; k++) tacc[k] = (T)0;
            for (int i = lp; i < TILE; i += LP) {
                const T x = sx[0][i], d = sd[0][i], w = sw[0][i];
                T v[NX];
                v[0] = x;
#pragma unroll
                for (int j = 1; j < NX; j++) v[j] = sxe[0][j - 1][i];
#pragma unroll
                for (int k = 0; k < CPT; k++) {
                    const T r = (eval_safe_at(mdl[k], v) - d) * w;
                    tacc[k] = fma(r, r, tacc[k]);
                }
            }
#pragma unroll
            for (int k = 0; k < CPT; k++) acc[k] += (double)tacc[k];
        }
    }

    // Ragged tail, straight from global memory (last split only).
    if (blockIdx.y == gridDim.y - 1) {
        T tacc[CPT];
#pragma unroll
        for (int k = 0; k < CPT; k++) tacc[k] = (T)0;
        for (int64_t i = nfull * TILE + lp; i < a.n; i += LP) {
            const T x = a.x[i], d = a.d[i], w = USIG ? (T)1 : a.w[i];
            T v[NX];
            v[0] = x;
#pragma unroll
            for (int j = 1; j < NX; j++) v[j] = a.xs[j][i];
#pragma unroll
            for (int k = 0; k < CPT; k++) {
                const T r = (eval_safe_at(mdl[k], v) - d) * w;
                tacc[k] = fma(r, r, tacc[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < CPT; k++) acc[k] += (double)tacc[k];
    }

    double w2 = 1.0;
    if constexpr (USIG) { const double w0 = (double)a.w[0]; w2 = w0 * w0; }
#pragma unroll
    for (int k = 0; k < CPT; k++) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o >= LC; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        const int64_t c = cbase + (int64_t)k * LC;
        if (lp == 0 && c < a.nchains) a.partial[(int64_t)blockIdx.y * a.ldpartial + c] = USIG ? v * w2 : v;
    }
    if (a.f.on) fused_metropolis(a.f, a.partial, a.ldpartial, a.nchains, WARPS * LC * CPT);
}

// ---- model values (best_model, func(params) shape probe) -------------------
// ---- model values (best_model, func(params) shape probe) -------------------
template <class M>
__global__ void k_model_eval(const double* params, int64_t ldp, const double* x, int64_t n, double* out) {
    M m;
    m.load(params + (int64_t)blockIdx.y * ldp);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[(int64_t)blockIdx.y * n + i] = m.eval_safe(x[i]);
}

// ... of a model of NX > 1 inputs: input j of point i is xs.x[j][i]
template <class M>
__global__ void k_model_eval_x(const double* params, int64_t ldp, EvalInputs xs, int64_t n, double* out) {
    constexpr int NX = ninputs_of<M>::value;
    using T = typename M::real;
    M m;
    m.load(params + (int64_t)blockIdx.y * ldp);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        T v[NX];
#pragma unroll
        for (int j = 0; j < NX; j++) v[j] = (T)xs.x[j][i];
        out[(int64_t)blockIdx.y * n + i] = m.eval_safe(v);
    }
}

// ... of a model of run-time constants or a prepare step (takes_consts), any NX: the
// constants k are fp64 here whatever the model's type
template <class M>
__global__ void k_model_eval_k(const double* params, int64_t ldp, EvalInputs xs, const double* k, int64_t n,
                               double* out) {
    constexpr int NX = ninputs_of<M>::value;
    using T = typename M::real;
    M m;
    m.load(params + (int64_t)blockIdx.y * ldp, k);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        T v[NX];
#pragma unroll
        for (int j = 0; j < NX; j++) v[j] = (T)xs.x[j][i];
        out[(int64_t)blockIdx.y * n + i] = eval_safe_at(m, v);
    }
}

}  // namespace
