// mc3_b200 -- launch parameters and the fused Metropolis epilogue shared by the
// model + chi-squared kernels (chisq.cu, chisq_grid.cu).
#pragma once
#include "models.cuh"
#include "sampler_dev.cuh"

namespace mc3b_chisq {

#ifndef MC3B_WARPS
#define MC3B_WARPS 4
#endif
#ifndef MC3B_RESIDENT
#define MC3B_RESIDENT 6
#endif
#ifndef MC3B_RESIDENT2
#define MC3B_RESIDENT2 4
#endif
#ifndef MC3B_LOOP_UNROLL
#define MC3B_LOOP_UNROLL 2
#endif
#ifndef MC3B_TILE_F64
#define MC3B_TILE_F64 128
#endif
constexpr int WARPS = MC3B_WARPS;
constexpr int STAGES = 3;
constexpr int LOOP_UNROLL = MC3B_LOOP_UNROLL;   // point groups of the inner loop unrolled together
constexpr int RESIDENT = MC3B_RESIDENT;   // CTAs per SM the register budget is tuned for (ILP over occupancy)
template <typename T> struct tilecfg { static constexpr int TILE = MC3B_TILE_F64; };   // fp64: 128 beat 256 by 6% (finer balance)
template <> struct tilecfg<float> { static constexpr int TILE = 512; };

constexpr int SCHED_MAX = 384;      // splits a size schedule can describe (else equal splits)
// Optional epilogue of the model kernels: the LAST CTA of a chain group (the one
// whose arrival completes the group's split count) adds the group's partial rows
// in split order and takes the Metropolis step of its chains -- what k_metropolis
// does, without the extra launch and without a second pass over `partial` from a
// cold kernel; the last group to finish bumps the device generation counter
// (replaces k_advance).  Same arithmetic, same order: identical bits.
struct FuseArgs {
    int on;
    int advance;                    // bump *S.gen_dev when every group is done
    int32_t* done;                  // arrival counters (fused_metropolis_end); zero before the first launch, self-resetting
    int64_t c_off;                  // global id of the chain in row 0 of params
    int64_t gen, zrow0;             // as mc3b_metropolis (gen < 0: device-driven)
    mc3b_sampler_t S;
};

// k_sinefold<MOM>: data centred on a reference line, folded and scaled (mc3b_moment_prepare),
// the per-tile moments, and the guard of the expansion (include/mc3b200.h, mc3b_moment_t)
struct MomentArgs {
    const double* folded;           // nullptr: not the moment form
    const double* tiles;
    double c0ref, slref, d2tot, amp_max;
    double xlo, xhi;                // range of the abscissa (bound of the line term of the guard)
    int32_t* guard_hits;
    // spectral form (k_spectral_chisq, include/mc3b200.h mc3b_spectral_t): nullptr = the tile kernels
    const double* spec;             // sums, then the Taylor tables of both bands (mc3b_spectral_prepare)
    double sw1, sw2, sdelta, sxc;   // first node of the band and of the doubled band, node spacing, centre of x
    int sn1, sn2, sorder;           // nodes per band, Taylor order K
    int layout;                     // of `folded`: 0 pairs interleaved (k_sinefold<MOM>), 1 mma fragments (k_sinemma)
    int64_t* record;                // guard record ring (mc3b_moment_t.record) or nullptr
    // (layout packed with the ints above: the record adds no bytes, so that every field after
    // this block keeps its offset and the kernels without the moment form are unchanged)
};

template <typename T> struct ChisqArgs {
    int nsched;                     // > 0: split y covers tiles [tstart[y], tstart[y+1])
    int32_t tstart[SCHED_MAX + 1];
    const double* params;
    int64_t ldp, nchains;
    const T *x, *d, *w;
    const T* fold;                  // mirrored-pair copy of d (mc3b_fold_data) or nullptr
    // k_sinefold on a piecewise-uniform abscissa (include/mc3b200.h, tile_x): origin of every whole
    // 128-point tile, the common step, the number of whole tiles; x/d hold the tiles first, then
    // the points that fill no tile.  nullptr: one uniform grid, x_i = x[0] + i (x[n-1] - x[0])/(n-1)
    const double* xt;
    double dxg;
    int64_t ntiles;
    const double* consts;           // k_sinefold: per-chain constants [NCONST, ldc] (k_fold_consts) or nullptr
    int64_t ldc;
    int consts_wait;                // launched as a programmatic dependent of k_fold_consts
    MomentArgs m;
    int64_t n;
    double* partial;
    int64_t ldpartial;
    int use_tma;
    FuseArgs f;
    // the inputs of a user model of NX per-point inputs (xs[0] = x).  After every other
    // field, so that the built-in kernels read the same offsets; 32 bytes, so that the
    // parameters after this block keep their 16-byte alignment (wide constant loads)
    const T* xs[MC3B_MAX_INPUTS];
    // the run-time constants of a user model (mc3b_user_model_chisq_consts), nullptr when it
    // has none; padded to 16 bytes for the same reason as xs
    const T* uconst;
    const void* uconst_pad;
};

// Inputs of the model-value kernels of a user model of several inputs or of constants
// (k_model_eval_x, k_model_eval_k).
struct EvalInputs { const double* x[MC3B_MAX_INPUTS]; };

// The Metropolis step itself, compiled once per translation unit: S points to the
// CTA's shared-memory copy of the sampler description.
static __device__ __noinline__ void fused_metropolis_step(const mc3b_sampler_t* S, double nxt, int64_t c, int64_t gen,
                                                          int64_t zrow0) {
    metropolis_chain(*S, nxt, gen, zrow0, c);
}

// Hook between the sum of a chain's partial rows and its Metropolis step; called by
// every thread of the reducer CTA (it may use CTA barriers), it returns the CTA's count of
// hits (chains it sent to another evaluation), the same in every thread.  counter(): where
// the hits of every launch are added up (nullptr: not counted); recording(): the thread
// whose arrival completes the launch calls record(g, hits), g = generations completed,
// hits = the counter's new value.
struct NoFix {
    __device__ __forceinline__ int operator()(bool, int64_t, double&) const { return 0; }
    __device__ __forceinline__ int32_t* counter() const { return nullptr; }
    __device__ __forceinline__ bool recording() const { return false; }
    __device__ __forceinline__ void record(int64_t, int) const {}
};
// *fix.counter() read by thread 0 (the one that uses it), early in the launch
template <class Fix>
__device__ __forceinline__ int fix_count_base(const Fix& fix) {
    const int32_t* c = fix.counter();
    return threadIdx.x == 0 && c ? __ldcg(c) : 0;
}

// After every thread's step: thread 0 of each CTA counts the CTA's arrival and its hits in one
// 64-bit word, (arrivals << 32) | hits, at the first 8-byte-aligned slot of f.done after the
// group counters; the CTA whose arrival completes the launch stores the hit counter, the
// record, the generation counter and the word's reset.  base: *fix.counter() as thread 0 read it
// earlier in the launch; gdev: *S.gen_dev as read earlier in the launch (whenever f.advance is
// set).  Nothing else writes either while the launch runs.
// No fence on one device: the values the last CTA stores are read only by later kernels or by
// the host after the kernel ends, which the kernel boundary orders after every store of the
// launch, and the one value that crosses CTAs within the launch, the hit count, travels in the
// arrival atomic itself.  Every CTA consumed its load of *S.gen_dev before the barrier that
// precedes its arrival, so the bump cannot overtake it.  Peer mode: the generation flags tell
// the other devices that this device's peer stores are performed, so every CTA fences them at
// system scope (cumulative over the barrier) before it arrives.
// A launch without advance or record has no arrival: each CTA with hits adds them to the counter.
template <class Fix>
__device__ __forceinline__ void fused_metropolis_end(const FuseArgs& f, const mc3b_sampler_t& S, const Fix& fix,
                                                     int64_t gen, int64_t gdev, int hits, int base) {
    __syncthreads();
    const bool rec = fix.recording();              // false for NoFix
    int32_t* const count = fix.counter();          // nullptr for NoFix
    if (threadIdx.x != 0) return;
    if (!f.advance && !rec) {
        if (count && hits) atomicAdd(count, hits);
        return;
    }
    if (S.X_peers) __threadfence_system();
    unsigned long long* word = reinterpret_cast<unsigned long long*>(f.done) + (gridDim.x + 1) / 2;
    const unsigned long long own = (1ull << 32) + (uint32_t)hits;
    const unsigned long long old = atomicAdd(word, own);
    if ((uint32_t)(old >> 32) != gridDim.x - 1) return;
    *word = 0;
    const int total = base + (int)(uint32_t)(old + own);
    if (count) *count = total;
    if (rec) fix.record(gen + 1, total);
    if (f.advance) {
        const int64_t g = gdev + 1;
        *S.gen_dev = g;
        if (S.F_peers) flags_publish(S, g);          // every CTA's peer stores are performed
    }
}

// chains_per_cta: chains a CTA covers (its thread t < chains_per_cta owns chain
// blockIdx.x * chains_per_cta + t of the launch).  `f` must be the kernel
// parameter itself (read from the constant bank, never copied to the stack).
//
// The reducer of a chain group is the CTA of its LAST split: CTAs are dispatched in
// block order, so it starts after every other split of the group is running or done,
// and with the decreasing split schedule it is also the shortest.  The other CTAs
// publish their row with one fire-and-forget reduction (no round trip: an atomic
// whose result every CTA waited for cost ~10 us per launch over the six waves) and
// leave; the reducer spins until all nsplit-1 arrivals are in.  A one-split launch has no
// arrivals to wait for.
template <class Fix = NoFix>
__device__ __forceinline__ void fused_metropolis(const FuseArgs& f, const double* partial, int64_t ldpartial,
                                                 int64_t nchains, int chains_per_cta, Fix fix = Fix()) {
    __shared__ __align__(16) mc3b_sampler_t sS;
    __shared__ double vbuf[STAGE_DOUBLES];
    __syncthreads();                               // the CTA's partial row is written
    const int others = (int)gridDim.y - 1;
    if ((int)blockIdx.y != others) {
        if (threadIdx.x == 0) {
            __threadfence();                       // cumulative over the barrier: the row before the count
            atomicAdd(&f.done[blockIdx.x], 1);
        }
        return;
    }
    const int base = fix_count_base(fix);
    if (threadIdx.x == 0) {
        sS = f.S;                                  // constant bank -> shared, static offsets only
        if (others > 0) {
            int seen;
            do {
                asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(f.done + blockIdx.x) : "memory");
            } while (seen < others);
            f.done[blockIdx.x] = 0;                // every arrival is in: ready for the next launch
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {                        // one warp stages the per-parameter vectors
        mc3b_sampler_t T = sS;
        const int np = T.npars, nf = T.nfree;
        const double* src[7] = {T.pstep, T.pmin, T.pmax, T.params0, T.prior, T.priorlow, T.priorup};
        for (int i = threadIdx.x; i < 7 * np; i += 32) {
            const int v = i / np, k = i - v * np;
            if (src[v]) vbuf[v * MAXP + k] = src[v][k];
        }
        int32_t* ifr = reinterpret_cast<int32_t*>(vbuf + 7 * MAXP);
        for (int i = threadIdx.x; i < nf; i += 32) ifr[i] = T.ifree[i];
        stage_peers_load(T, vbuf, threadIdx.x, 32);
        __syncwarp();
        if (threadIdx.x == 0) {
            sS.pstep = vbuf; sS.pmin = vbuf + MAXP; sS.pmax = vbuf + 2 * MAXP; sS.params0 = vbuf + 3 * MAXP;
            if (T.prior) { sS.prior = vbuf + 4 * MAXP; sS.priorlow = vbuf + 5 * MAXP; sS.priorup = vbuf + 6 * MAXP; }
            sS.ifree = ifr;
            stage_peers_point(sS, vbuf);
        }
    }
    __syncthreads();
    const int64_t cl = (int64_t)blockIdx.x * chains_per_cta + threadIdx.x;
    const bool mine = (int)threadIdx.x < chains_per_cta && cl < nchains;
    const int64_t gdev = f.gen < 0 || f.advance ? *sS.gen_dev : 0;
    int64_t gen = f.gen, zrow0 = f.zrow0;
    if (gen < 0) {
        gen = gdev;
        zrow0 = ((gen + 1) % sS.thinning == 0) ? sS.M0 + ((gen + 1) / sS.thinning - 1) * sS.nchains : -1;
    }
    double nxt = 0.0;
    bool inb = false;
    if (mine) {
        inb = sS.inb[f.c_off + cl] != 0;
        if (inb) nxt = sum_partials<true>(partial, ldpartial, (int)gridDim.y, cl);
    }
    const int hits = fix(inb, cl, nxt);
    if (mine) fused_metropolis_step(&sS, nxt, f.c_off + cl, gen, zrow0);
    fused_metropolis_end(f, sS, fix, gen, gdev, hits, base);
}

// The one-split launch of k_spectral_chisq, whose thread t of CTA b owns chain b * WARPS * 32 + t,
// in two parts.  fused_metropolis_load runs at kernel entry: each thread reads the generation
// counter and its chain's state (metropolis_load), and the CTA stages the per-parameter vectors,
// every load issued before the first shared-memory store.  None of it depends on the chain's
// chi-squared and no other thread writes it during the launch, so these loads overlap the
// chi-squared instead of following it one round trip after another.
struct FusedEntry {
    int64_t gen;                    // generation of the step (f.gen, or *gen_dev when device-driven)
    int64_t gdev;                   // *gen_dev when the launch bumps it or is device-driven
    int base;                       // fix_count_base
    ChainState st;
};
template <class Fix>
__device__ __forceinline__ FusedEntry fused_metropolis_load(const FuseArgs& f, const Fix& fix, double* vbuf,
                                                            int64_t cl) {
    FusedEntry e;
    e.gdev = f.gen < 0 || f.advance ? *f.S.gen_dev : 0;
    e.gen = f.gen < 0 ? e.gdev : f.gen;
    e.base = fix_count_base(fix);
    e.st = metropolis_load(f.S, e.gen, f.c_off + cl);
    stage_vectors_load<WARPS * 32>(f.S, vbuf, threadIdx.x);
    stage_peers_load(f.S, vbuf, threadIdx.x, WARPS * 32);
    return e;
}
// Every thread of the CTA, after its partial row is written: guard(act, nxt) is the Fix hook
// (a CTA-wide call, returning the CTA's hits) with the chain's inputs already in registers;
// mine: the thread owns a chain, whose only row is `row`, added from the register (0.0 + row:
// the bits of the split-order sum).
template <class Fix, class Guard>
__device__ __forceinline__ void fused_metropolis_apply(const FuseArgs& f, const FusedEntry& e, double* vbuf, int64_t cl,
                                                       bool mine, double row, const Fix& fix, Guard guard) {
    __syncthreads();                               // the staged vectors are in
    mc3b_sampler_t S = f.S;
    stage_point(S, vbuf);
    const int64_t gen = e.gen;
    int64_t zrow0 = f.zrow0;
    if (f.gen < 0) zrow0 = ((gen + 1) % S.thinning == 0) ? S.M0 + ((gen + 1) / S.thinning - 1) * S.nchains : -1;
    const bool inb = mine && e.st.inb != 0;
    double nxt = inb ? 0.0 + row : 0.0;
    const int hits = guard(inb, nxt);
    if (mine) metropolis_apply(S, e.st, nxt, gen, zrow0, f.c_off + cl);
    fused_metropolis_end(f, S, fix, gen, e.gdev, hits, e.base);
}

#ifndef __CUDACC_RTC__
// Launch shape of a model + chi-squared launch (chisq.cu plan_shape): chains per warp,
// data splits and, for large populations, the split boundaries in tiles.
struct Shape {
    int lc, nsplit;
    int nsched; int32_t tstart[SCHED_MAX + 1];
};
#endif

}  // namespace mc3b_chisq
using namespace mc3b_chisq;

#ifndef __CUDACC_RTC__
// chisq.cu: argument block, launch shape and argument checks of a k_model_chisq launch
// (plan, TMA alignment, fuse, nsplit), shared by the built-in and the user-model paths.
template <typename T>
int mc3b_chisq_setup(const double* params, int64_t ldp, int64_t nchains, const void* x, const void* d, const void* w,
                     int64_t n, double* partial, int64_t ldpartial, int nsplit, int dtype, const mc3b_chisq_opts_t& o,
                     ChisqArgs<T>& A, Shape& sh, dim3& grid);

// chisq_grid.cu
int mc3b_launch_sinegrid(const ChisqArgs<double>& a, bool usig, unsigned groups, unsigned nsplit, cudaStream_t st);
int mc3b_launch_sinefold(const ChisqArgs<double>& a, double* work, unsigned groups, unsigned nsplit, cudaStream_t st);
int mc3b_launch_fold(const double* d, int64_t n, double* out, cudaStream_t st);
int mc3b_launch_moment_finish(const ChisqArgs<double>& a, int nsplit, int npars, const double* prior, const double* plo,
                              const double* pup, double* chisq, cudaStream_t st);
int mc3b_launch_moment_prepare(const double* d, int64_t ntiles, double x0, double dx, const double* tile_x,
                               double c0ref, double slref, double* folded, double* tiles, int layout, cudaStream_t st);
int mc3b_launch_spectral_chisq(const ChisqArgs<double>& a, unsigned groups, cudaStream_t st);
int mc3b_launch_spectral_prepare(const double* x, const double* d, int64_t n, double c0ref, double slref,
                                 const mc3b_spectral_t& s, cudaStream_t st);
#endif
