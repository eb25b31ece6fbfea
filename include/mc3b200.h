/* mc3b200.h -- C ABI of libmc3b200.so, the B200 (sm_100a) replacement for the
 * native layer of pcubillos/mc3 and for the per-iteration loop that sits on it.
 *
 * Every entry point returns an int status (MC3B_OK on success); the message of
 * the last failure on the calling thread is available from mc3b_last_error().
 * All pointers are DEVICE pointers unless a parameter is marked [host].  The
 * caller owns every buffer; the library allocates nothing persistent except the
 * peer buffers and user-model handles it hands out (see below).
 * `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls
 * are asynchronous with respect to the host and re-entrant per stream.
 *
 * Reference interfaces replaced (paths relative to the reference root):
 *   _chisq.chisq / _chisq.residuals         src_c/_chisq.c:37-79, 111-140
 *   stats.h priors()                        src_c/include/stats.h:90-109
 *   _dwt.chisq / _dwt.daub4                 src_c/_dwt.c:56-119, 154-186
 *   _time_averaging.binrms                  src_c/_time_averaging.c:55-143
 *   _binarray.binarray                      src_c/_binarray.c:34-81
 *   Chain.run() proposal / Metropolis loop  mc3/chain.py:183-299
 *   Chain.eval_model()                      mc3/chain.py:302-340
 *   gelman_rubin()                          mc3/stats/gelman.py:12-92
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference adds.
 */
#ifndef MC3B200_H
#define MC3B200_H

#ifdef __CUDACC_RTC__
/* NVRTC (user models compiled at run time) has no <stdint.h>: the LP64 types */
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long int64_t;
typedef unsigned long uint64_t;
typedef unsigned long uintptr_t;
#else
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MC3B_VERSION 100            /* 0.1.0 */

enum { MC3B_OK = 0, MC3B_ERR_ARG = 1, MC3B_ERR_CUDA = 2 };
enum { MC3B_F64 = 0, MC3B_F32 = 1 };
enum { MC3B_MODEL_POLYNOMIAL = 0, MC3B_MODEL_SINUSOID = 1,
       MC3B_MODEL_GAUSSIAN = 2, MC3B_MODEL_BOX = 3,
       /* sinusoid on a UNIFORM abscissa grid (caller's assertion: x[i] = x[0] + i dx to
        * a few ulp): same values to 2e-15 (8e-14 for steps of radians per sample) of the amplitude; the sine advances by a
        * three-term recurrence re-anchored per tile (models.cuh SineGridModel) */
       MC3B_MODEL_SINUSOID_GRID = 4 };
enum { MC3B_MRW = 0, MC3B_DEMC = 1, MC3B_SNOOKER = 2 };

#define MC3B_MAX_PARS 32            /* parameters per model vector          */
#define MC3B_MAX_SPLIT 4096         /* data splits of one chi-squared launch */
#define MC3B_MAX_INPUTS 4           /* per-point inputs of a user model      */

int mc3b_version(void);
const char* mc3b_last_error(void);
/* Number of SMs of the current device (sizes grids); <0 on error. */
int mc3b_device_sms(void);

/* ------------------------------------------------------------------------
 * Chi-squared family   (replaces _chisq.c and Chain.eval_model)
 * ---------------------------------------------------------------------- */

/* Choose the launch shape of mc3b_model_chisq for (nchains, n): writes the
 * number of data splits (rows of the `partial` workspace) to *nsplit.
 * Deterministic function of its arguments. */
int mc3b_model_chisq_plan(int64_t nchains, int64_t n, int dtype, int* nsplit);

/* The same for a given kernel family: launches with opts.moment (the
 * sufficient-statistics kernel) are planned with MC3B_PLAN_MOMENT (MC3B_PLAN_SPECTRAL when
 * opts.moment->spectral is set), everything else
 * with MC3B_PLAN_GENERAL (= mc3b_model_chisq_plan). */
#define MC3B_PLAN_GENERAL 0
#define MC3B_PLAN_MOMENT 1
#define MC3B_PLAN_SPECTRAL 2    /* the spectral form of mc3b_moment_t: always one split */
int mc3b_model_chisq_plan_kind(int kind, int64_t nchains, int64_t n, int dtype, int* nsplit);

/* The split boundaries behind that plan, in data points: split s sums the points
 * [point_start[s], point_start[s+1]); point_start has nsplit+1 entries (HOST
 * memory, `cap` >= nsplit+1) and ends at n.  Large populations get splits of
 * decreasing size: CTAs start in split order, so the last to start are short and
 * the SMs finish together.  (No reference counterpart: the reference sums one
 * chain at a time, _chisq.c:111-140.) */
int mc3b_model_chisq_splits(int64_t nchains, int64_t n, int dtype,
                            int64_t* point_start, int cap, int* nsplit);

/* Fused built-in model + data chi-squared, batched over chains:
 *   partial[s, c] = sum over the points i of split s of
 *                   ((model(params[c], x_i) - data_i) * invsig_i)^2
 * params   [nchains, ldp] fp64, row c = FULL parameter vector of chain c; the
 *          model sees its first `nmodel` entries (chain.py:316-319: with the
 *          wavelet likelihood the model gets params[0:-3]).
 * x, data, invsig  [n] fp64 (dtype F64) or fp32 (dtype F32); invsig = 1/uncert.
 * partial  [nsplit, ldpartial] fp64 workspace (ldpartial >= nchains), nsplit
 *          from mc3b_model_chisq_plan; entry [s, c] belongs to row c of params.
 * The sum over splits and the prior terms are added by mc3b_chisq_finish or,
 * inside the sampler, by mc3b_metropolis. */
int mc3b_model_chisq(int model_id, int dtype, const double* params, int64_t ldp,
                     int64_t nchains, int nmodel, const void* x,
                     const void* data, const void* invsig, int64_t n,
                     double* partial, int64_t ldpartial, int nsplit,
                     void* stream);

/* Options of mc3b_model_chisq_ex ([host] struct; NULL or all-zero = mc3b_model_chisq).
 *
 * plan_chains    chain count the launch shape is planned for (0 = nchains).  The bits
 *                of a chain's chi-squared depend on the order its terms are added,
 *                i.e. on the split boundaries = f(plan_chains, n, dtype, SM count), not
 *                on which or how many chains the launch holds: plan once for the whole
 *                population (mc3b_model_chisq_plan(plan_chains, ...)) and any subset of
 *                its chains, on any device of the same type, gets identical bits.
 * uniform_sigma  all uncertainties are equal: invsig points to ONE value; residuals are
 *                plain differences and the sums are scaled by invsig[0]^2 (no weight
 *                stream).  For MC3B_MODEL_SINUSOID_GRID the abscissa is not streamed
 *                either (x[0] and x[n-1] define the grid).
 * fuse           non-NULL: the last CTA to finish a group of chains adds their partial
 *                rows (split order) plus priors and takes their Metropolis step, exactly
 *                as mc3b_metropolis(fuse, partial, ldpartial, nsplit, c_off, gen, zrow0,
 *                c_off, c_off + nchains) would -- without the second launch.  fuse_done:
 *                device int32[groups + 3] (groups <= nchains/32 + 1), 8-byte aligned, zero
 *                before the first use, left zero by every launch: a counter per group, then
 *                the launch's 64-bit arrival word at the first 8-byte-aligned slot after them.
 *                advance: the last group also increments *fuse->gen_dev (replaces mc3b_advance).
 * folded         non-NULL (fp64, MC3B_MODEL_SINUSOID_GRID, uniform_sigma): the copy of
 *                `data` written by mc3b_fold_data; the kernel then works on point pairs
 *                mirrored about block centres (3.3 instead of 6 FP64 instructions per
 *                chain and point, same rounding-error class; csrc/chisq_grid.cu).
 * work           with `folded`: device workspace of MC3B_FOLD_WORK * nchains doubles; the
 *                per-chain constants of the kernel (wavenumber, the sine/cosine tables of
 *                the pair offsets, block and restart rotations) are then derived once per
 *                chain by a small kernel launched first, instead of by each of the nsplit
 *                CTAs of a chain group.  NULL: every CTA derives them (same bits).
 * moment         non-NULL (with uniform_sigma and work; fp64, MC3B_MODEL_SINUSOID_GRID):
 *                the sufficient-statistics form described at mc3b_moment_t below.  Its rows
 *                are UNGUARDED: either `fuse` is set (the Metropolis epilogue applies the
 *                guard) or the rows go through mc3b_moment_finish, never through
 *                mc3b_chisq_finish / mc3b_metropolis.
 * tile_x, dx, ntiles   (fp64, MC3B_MODEL_SINUSOID_GRID) PIECEWISE-uniform abscissa, e.g. a time series
 *                of constant cadence with gaps: the caller has reordered x and data so that
 *                (and invsig, when it is per point) so that
 *                entries [128 t, 128 t + 128) are the t-th run of 128 points spaced dx apart
 *                starting at tile_x[t] (device array, ntiles entries; the tiles need not be
 *                adjacent or ordered), followed by the n - 128 ntiles points that fill no
 *                tile, which are evaluated one by one.  tile_x = NULL: one uniform grid from
 *                x[0] to x[n-1].  mc3b_model_chisq_splits does not describe this layout. */
struct mc3b_sampler;
typedef struct mc3b_chisq_opts {
    int64_t plan_chains;
    int32_t uniform_sigma;
    int32_t advance;
    const struct mc3b_sampler* fuse;
    int32_t* fuse_done;
    int64_t c_off, gen, zrow0;
    const void* folded;
    void* work;
    const struct mc3b_moment* moment;
    const double* tile_x;
    double dx;
    int64_t ntiles;
} mc3b_chisq_opts_t;
#define MC3B_FOLD_WORK 27

/* Sufficient-statistics form of the uniform-grid sinusoid + line chi-squared (one
 * uncertainty for all points).  With the data centred on a reference line,
 * d' = d - (c0ref + slref x), the squares of the pair sums and differences expand to
 *   chisq sigma^2 = 2 sum_blocks [ Sc (Sc Kcc + 2 Lc Kc - 2 Pe) + Cc (Cc Kss + 2 g Ksd - 2 Po) ]
 *                 + 2 sum_tiles  [ 64 Lm^2 + 87376 g^2 - 2 Lm M0 - 2 g M1 + M2 ]
 * where only Pe = sum_p cos(dl_p h) e_p and Po = sum_p sin(dl_p h) o_p touch the data
 * (ONE multiply-add per point and chain) and M0, M1, M2 are three moments per
 * 128-point tile.  The result is what is left after sums of size (|s| + |L'| + |d'|)^2
 * cancel, so its relative error is eps_eff * amp with
 *   amp = (|A| sqrt(n) + |L'| + sqrt(d2tot))^2 / (sigma^2 chisq),   eps_eff < 3e-15;
 * the Metropolis epilogue evaluates every chain with amp > amp_max again, point by
 * point (library sine), and counts it in *guard_hits, so that every chi-squared used
 * for a decision is within 1e-10 of _chisq.c:111-140 on the same inputs.
 *   folded  [n]  from mc3b_moment_prepare     tiles  [4 * (n/128)]  likewise
 *   c0ref, slref   the reference line (any; a least-squares line through the data keeps amp small)
 *   d2tot   sum of d'^2 over the n points     amp_max  e.g. 4000 (error < 1.2e-11)
 *   xlo, xhi  smallest and largest abscissa (they bound |L'|)
 *   layout  of `folded`: 0 = pairs interleaved as in mc3b_fold_data (Pe, Po by FMAs),
 *           1 = the four B fragments of mma.m8n8k4 per tile (Pe, Po as FP64 tensor-core
 *           products: fewer operand reads, instructions and shared-memory loads)
 *   guard_hits  device int32 counter or NULL
 *   spectral  [host] NULL: the tile kernels above.  Otherwise the spectral form below replaces
 *           them (folded, tiles and opts.work are then not read); its launches are planned
 *           with MC3B_PLAN_SPECTRAL (one split) and its rows are unguarded in the same way.
 *   record  NULL, or (with guard_hits) the device address of MC3B_GUARD_RECORDS int64 slots of
 *           page-locked, device-mapped host memory (mc3b_host_device_pointer).  A launch with
 *           `fuse` then stores, from the thread that finishes last, after every hit of the
 *           launch is counted, one aligned 64-bit record into slot g % MC3B_GUARD_RECORDS:
 *           (g mod 2^32) << 32 | *guard_hits, g = the generations completed with this launch
 *           (opts.gen + 1, or *fuse->gen_dev + 1 before its increment when opts.gen < 0).  The
 *           host polls the slot until its high word is g mod 2^32 and reads the cumulative count
 *           of generation g with no copy on the stream.  Fill the slots with a stamp no
 *           generation of that slot has, e.g. slot s with stamp s + 1; a record stays until
 *           generation g + MC3B_GUARD_RECORDS overwrites it.  Launches without `fuse` (and
 *           mc3b_moment_finish) write none. */
#define MC3B_GUARD_RECORDS 64
struct mc3b_spectral;
typedef struct mc3b_moment {
    const double* folded;
    const double* tiles;
    double c0ref, slref, d2tot, amp_max;
    double xlo, xhi;
    int32_t* guard_hits;
    int32_t layout;     /* as given to mc3b_moment_prepare */
    const struct mc3b_spectral* spectral;
    int64_t* record;
} mc3b_moment_t;

/* Spectral form of the same chi-squared: O(1) per chain instead of O(n).  With
 * t = x - xc, d' = d - (c0ref + slref x), L' = a + b t the line relative to the reference
 * line (a = c0 - c0ref + (sl - slref) xc, b = sl - slref), w = 2 pi / P and
 * S_g(w) = sum_i g_i e^{i w x_i},
 *   sigma^2 chisq = A^2 [n/2 - Re(e^{2 i ph} S_1(2w))/2]
 *                 + 2 A Im(e^{i ph} [a S_1(w) + b S_t(w) - S_d'(w)])
 *                 + n a^2 + 2 a b St + b^2 St2 - 2 a Sd - 2 b Std + D2
 * (St = sum t, St2 = sum t^2, Sd = sum d', Std = sum t d', D2 = sum d'^2).  The data enter
 * only through S at the chain's own frequency.  Per node w_j = w1 + j delta (j < n1) of the
 * band and w2 + j delta (j < n2) of the doubled band, the table holds Taylor coefficients
 *   T_g[j][k] = sum_i g_i t_i^k e^{i w_j x_i} / k!,  S_g(w_j + dw) = e^{i dw xc} sum_k (i dw)^k T_g[j][k]
 * to order K = `order` (9 or 15); truncation error <= (|dw| R)^{K+1} / (K+1)! sum |g_i|,
 * R = max |t_i|, |dw| <= delta/2 (mc3_b200/spectral.py plans delta and K for 1e-18).
 * Like the tile form, the result is what is left after terms of size (|s| + |L'| + |d'|)^2
 * cancel: relative error eps_eff * amp, eps_eff < 3e-15 (profiles/spectral_error.py); the
 * same guard (amp_max of mc3b_moment_t) applies, and a chain whose w or 2w has no node
 * within delta/2 also takes the point-by-point evaluation and counts in guard_hits.
 *   table  device, mc3b_spectral_size() doubles, written by mc3b_spectral_prepare:
 *          MC3B_SPECTRAL_HEAD sums {n, St, St2, Sd, Std, D2, 0, 0}, then per node of the band
 *          K + 2 complex T_1 and K + 1 complex T_d' (T_t[k] = (k + 1) T_1[k + 1]), then per
 *          node of the doubled band K + 1 complex T_1 (complex = re, im). */
#define MC3B_SPECTRAL_HEAD 8
typedef struct mc3b_spectral {
    double* table;
    double w1, w2, delta, xc;   /* first node of the band and of the doubled band, spacing, centre */
    int32_t n1, n2, order;      /* nodes of the band, of the doubled band; K */
} mc3b_spectral_t;

/* Doubles of the table of mc3b_spectral_t for n1, n2 nodes and order K (9 or 15). */
int mc3b_spectral_size(int n1, int n2, int order, int64_t* ndoubles /*[host]*/);

/* Writes s->table from the n points x, data (device, fp64, any order: for a piecewise-
 * uniform abscissa the reordered arrays) about the reference line c0ref + slref x.  One
 * CTA per node, fixed-order sums: the same bits on every device.  Done once per data set. */
int mc3b_spectral_prepare(const double* x, const double* data, int64_t n, double c0ref,
                          double slref, const mc3b_spectral_t* s, void* stream);

/* mc3b_chisq_finish for rows written by the moment form WITHOUT `fuse`: adds the
 * nsplit rows of every chain in split order, applies the guard of mc3b_moment_t
 * (re-evaluating the chains that fail it point by point from x, data, invsig[0],
 * and counting them in *m->guard_hits), then adds the prior terms (prior may be NULL).
 * params/ldp/x/data/invsig/n: as passed to mc3b_model_chisq_ex for the same launch. */
int mc3b_moment_finish(const mc3b_moment_t* m, const double* partial,
                       int64_t ldpartial, int nsplit, int64_t nchains,
                       const double* params, int64_t ldp, int npars,
                       const double* x, const double* data, const double* invsig,
                       int64_t n, const double* prior, const double* priorlow,
                       const double* priorup, double* chisq, void* stream);

/* Chain-independent preparation for mc3b_moment_t over `ntiles` whole tiles of 128
 * points: x_i = x0 + i dx, or, with tile_x != NULL, tile_x[t] + j dx for point j of
 * tile t (piecewise-uniform abscissa, see mc3b_chisq_opts_t).  Per 16-point
 * block, pair p joins points 7-p and 8+p: layout 0: folded[16 b + 2 p] = -(d'_hi + d'_lo),
 * folded[16 b + 2 p + 1] = -(d'_hi - d'_lo); layout 1: within the tile, entry
 * 64 eo + 32 (p / 4) + 4 b + p % 4 (eo = 0 for the sums, 1 for the differences); per tile t,
 * tiles[4 t ..] = {-2 sum e, -2 (16 sum_b (b - 3.5) sum_p e + sum (p + 1/2) o), sum e^2 + o^2, 0}
 * with e, o the half sum and half difference of a pair. */
int mc3b_moment_prepare(const double* data, int64_t ntiles, double x0, double dx,
                        const double* tile_x, double c0ref, double slref, int layout,
                        double* folded, double* tiles, void* stream);

/* Chain-independent preparation for `folded` above: per block of 16 points, pair
 * p = 0..7 joins points 7-p and 8+p of the block;
 *   out[16 b + 2 p] = -(d_hi + d_lo)/2,   out[16 b + 2 p + 1] = -(d_hi - d_lo)/2.
 * data, out: [n] fp64 device arrays (the n % 16 trailing entries of out are left
 * untouched).  Done once per data set.  (No reference counterpart: the reference
 * evaluates one residual per point, _chisq.c:111-140.) */
int mc3b_fold_data(const double* data, int64_t n, double* out, void* stream);

int mc3b_model_chisq_ex(int model_id, int dtype, const double* params, int64_t ldp,
                        int64_t nchains, int nmodel, const void* x,
                        const void* data, const void* invsig, int64_t n,
                        double* partial, int64_t ldpartial, int nsplit,
                        const mc3b_chisq_opts_t* opts, void* stream);

/* model[c, i] = model(params[c], x_i), fp64, out is [nchains, n] row-major. */
int mc3b_model_eval(int model_id, const double* params, int64_t ldp,
                    int64_t nchains, int nmodel, const double* x, int64_t n,
                    double* out, void* stream);

/* ------------------------------------------------------------------------
 * User models compiled at run time   (the user's own `func`, chain.py:316-319)
 *
 * The source defines  __device__ real model(real x, const real* p)  (p[0..nmodel)),
 * with `real` = double (dtype F64) or float (F32); helpers above it are allowed and
 * models.cuh (fast_sin, fast_sincos_core, ...) is included.  NVRTC compiles it into
 * the kernels of the built-in models (csrc/chisq_kernel.cuh), so the model runs on the
 * same fused, TMA-staged, graph-capturable path.
 *
 * A model of several per-point inputs (ninputs = k, 1 <= k <= MC3B_MAX_INPUTS) takes k
 * reals before the parameters:  __device__ real model(real t, real xc, real yc, const
 * real* p)  for k = 3.  It is compiled with the _ex entry points and launched with the
 * _inputs ones; the plain entry points are those of k = 1.
 * ---------------------------------------------------------------------- */
typedef struct mc3b_user_model mc3b_user_model_t;          /* opaque */

/* source -> sm_100a CUBIN, with the NVRTC library at nvrtc_path (dlopen'ed; 12.8 or
 * newer).  Host only, needs no device.  *size always receives the size needed; the
 * CUBIN is written when cap >= *size.  log [host, logcap] receives the NVRTC log.
 * MC3B_ERR_ARG: the source does not compile (see the log), defines no `model`, or the
 * buffer is too small; MC3B_ERR_CUDA: NVRTC cannot be loaded or is too old. */
int mc3b_user_model_compile(const char* nvrtc_path, const char* source, int nmodel,
                            int dtype, void* cubin /*[host]*/, int64_t cap,
                            int64_t* size /*[host]*/, char* log /*[host]*/,
                            int64_t logcap);

/* Load a CUBIN of mc3b_user_model_compile (same nmodel and dtype) into every device
 * of the process and return a handle (allocates; release it with
 * mc3b_user_model_free).  A module built against other headers or another library
 * version is refused (MC3B_ERR_ARG). */
int mc3b_user_model_load(const void* cubin /*[host]*/, int64_t size, int nmodel,
                         int dtype, mc3b_user_model_t** out /*[host]*/);
int mc3b_user_model_free(mc3b_user_model_t* m);

/* mc3b_model_chisq_ex for a user model: the same partial layout, plan
 * (mc3b_model_chisq_plan) and fuse semantics; dtype and nmodel come from the
 * handle.  Of the options, plan_chains, uniform_sigma and fuse / fuse_done / c_off /
 * gen / zrow0 / advance apply; folded, work, moment and tile_x are refused. */
int mc3b_user_model_chisq_ex(const mc3b_user_model_t* m, const double* params,
                             int64_t ldp, int64_t nchains, const void* x,
                             const void* data, const void* invsig, int64_t n,
                             double* partial, int64_t ldpartial, int nsplit,
                             const mc3b_chisq_opts_t* opts, void* stream);

/* mc3b_model_eval for a user model: fp64 values, out is [nchains, n] row-major. */
int mc3b_user_model_eval(const mc3b_user_model_t* m, const double* params,
                         int64_t ldp, int64_t nchains, const double* x, int64_t n,
                         double* out, void* stream);

/* mc3b_user_model_compile / _load for a model of `ninputs` per-point inputs
 * (1..MC3B_MAX_INPUTS); ninputs = 1 is exactly the plain entry point.  A source whose
 * `model` takes another number of inputs fails to compile (MC3B_ERR_ARG, see the log). */
int mc3b_user_model_compile_ex(const char* nvrtc_path, const char* source, int nmodel,
                               int ninputs, int dtype, void* cubin /*[host]*/,
                               int64_t cap, int64_t* size /*[host]*/,
                               char* log /*[host]*/, int64_t logcap);
int mc3b_user_model_load_ex(const void* cubin /*[host]*/, int64_t size, int nmodel,
                            int ninputs, int dtype, mc3b_user_model_t** out /*[host]*/);

/* mc3b_user_model_chisq_ex and _eval with the inputs as an array xs [host] of nx
 * device pointers (nx must equal the handle's ninputs), each n values of the
 * handle's dtype (_chisq_inputs) or fp64 (_eval_inputs).  The plain entry points
 * refuse a handle of more than one input (MC3B_ERR_ARG).  A launch whose inputs
 * are not all 16-byte aligned reads them without TMA, as for an unaligned x. */
int mc3b_user_model_chisq_inputs(const mc3b_user_model_t* m, const double* params,
                                 int64_t ldp, int64_t nchains,
                                 const void* const* xs /*[host] nx device pointers*/,
                                 int nx, const void* data, const void* invsig, int64_t n,
                                 double* partial, int64_t ldpartial, int nsplit,
                                 const mc3b_chisq_opts_t* opts, void* stream);
int mc3b_user_model_eval_inputs(const mc3b_user_model_t* m, const double* params,
                                int64_t ldp, int64_t nchains,
                                const double* const* xs /*[host] nx device pointers*/,
                                int nx, int64_t n, double* out, void* stream);

/* A model of run-time constants and a per-chain prepare step.  The array p that
 * `model` sees has nmodel + nconst + nwork slots (at most MC3B_MAX_PARS):
 * [parameters | constants | work].  The constants come with each launch, so their
 * values are not compiled into the module.  The source may define
 *     __device__ void prepare(real* p)
 * which runs once per chain wherever the parameters are loaded (once per chain and
 * CTA), after the constants, and may write any slot of that private copy: the place to
 * hoist what depends on the chain alone (1/sigma, 2 pi/P) into the work slots.  It is
 * found by name lookup, so a comment that mentions it does not count; a `prepare` that
 * cannot be called with a real* fails to compile at its own line, and nwork > 0 without
 * one is refused (MC3B_ERR_ARG).  nconst = nwork = 0 with no prepare is exactly
 * mc3b_user_model_compile_ex / _load_ex. */
typedef struct {
    int nmodel, ninputs, nconst, nwork, dtype;
} mc3b_user_model_desc_t;

int mc3b_user_model_compile_desc(const char* nvrtc_path, const char* source,
                                 const mc3b_user_model_desc_t* desc /*[host]*/,
                                 void* cubin /*[host]*/, int64_t cap,
                                 int64_t* size /*[host]*/, char* log /*[host]*/,
                                 int64_t logcap);
int mc3b_user_model_load_desc(const void* cubin /*[host]*/, int64_t size,
                              const mc3b_user_model_desc_t* desc /*[host]*/,
                              mc3b_user_model_t** out /*[host]*/);

/* _chisq_inputs and _eval_inputs with the nk constants at `consts` [device], in the
 * handle's dtype (_chisq_consts) or fp64 (_eval_consts); nk must equal the handle's
 * nconst, and consts may be NULL when it is 0.  They take every handle; the entry points
 * above refuse one of nconst > 0 (MC3B_ERR_ARG). */
int mc3b_user_model_chisq_consts(const mc3b_user_model_t* m, const double* params,
                                 int64_t ldp, int64_t nchains,
                                 const void* const* xs /*[host] nx device pointers*/,
                                 int nx, const void* consts, int nk, const void* data,
                                 const void* invsig, int64_t n, double* partial,
                                 int64_t ldpartial, int nsplit,
                                 const mc3b_chisq_opts_t* opts, void* stream);
int mc3b_user_model_eval_consts(const mc3b_user_model_t* m, const double* params,
                                int64_t ldp, int64_t nchains,
                                const double* const* xs /*[host] nx device pointers*/,
                                int nx, const double* consts, int nk, int64_t n,
                                double* out, void* stream);

/* chisq[c] = sum_s partial[s*ldpartial + c] (fixed order s = 0..nsplit-1)
 *          + sum over j with priorlow_j > 0 and priorup_j > 0 of
 *            ((p_cj - prior_j) / (p_cj > prior_j ? priorup_j : priorlow_j))^2
 * (mc3/stats/stats.py:208-216 + stats.h:90-109).  prior* may be NULL. */
int mc3b_chisq_finish(const double* partial, int64_t ldpartial, int nsplit,
                      int64_t nchains,
                      const double* params, int64_t ldp, int npars,
                      const double* prior, const double* priorlow,
                      const double* priorup, double* chisq, void* stream);

/* _chisq.chisq for models evaluated elsewhere (user callables):
 *   chisq[c] = sum_i ((model[c, i] - data_i) / uncert_i)^2, model [nchains, ldm]. */
int mc3b_chisq_batch(const double* model, int64_t ldm, int64_t nchains,
                     const double* data, const double* uncert, int64_t n,
                     double* chisq, void* stream);

/* _chisq.residuals: out[i] = (model_i - data_i)/uncert_i, i < n; then the np
 * prior terms off_k / (off_k > 0 ? up_k : low_k).  off may be NULL (np = 0). */
int mc3b_residuals(const double* model, const double* data,
                   const double* uncert, int64_t n, const double* off,
                   const double* low, const double* up, int64_t np,
                   double* out, void* stream);

/* ------------------------------------------------------------------------
 * Sampler   (replaces the body of Chain.run, mc3/chain.py:183-299)
 * ---------------------------------------------------------------------- */

/* Population state.  Per-chain arrays are indexed by GLOBAL chain id and have
 * `nchains` entries on every device; a device only touches its own slice
 * [chain0, chain0 + nlocal). */
typedef struct mc3b_sampler {
    int64_t nchains, chain0, nlocal;
    int32_t npars, nfree, sampler, reflect;   /* reflect: 0 = reject out-of-bounds (reference) */
    const int32_t* ifree;        /* [nfree] indices of free parameters            */
    const double* pstep;         /* [npars] >0 free, 0 fixed, <0 shared (-(k+1))  */
    const double* pmin;          /* [npars]                                        */
    const double* pmax;          /* [npars]                                        */
    const double* params0;       /* [npars] template: values of fixed parameters   */
    const double* prior;         /* [npars] or NULL                                */
    const double* priorlow;      /* [npars] or NULL                                */
    const double* priorup;       /* [npars] or NULL                                */
    double gamma;                /* fgamma * 2.38 / sqrt(2 nfree)  chain.py:175    */
    double fepsilon;
    uint64_t seed;               /* Philox key                                     */
    double* X;                   /* [nchains, nfree] current states (freepars)     */
    double* chisq_cur;           /* [nchains] chi-squared of X                     */
    double* Z;                   /* [zlen, nfree] history (reference layout)       */
    double* log_post;            /* [zlen]                                         */
    int32_t* zchain;             /* [zlen]                                         */
    int64_t zlen, M0;
    double* nextp;               /* [nchains, npars] proposed full vectors         */
    double* mrfactor;            /* [nchains] snooker Metropolis factor            */
    double* u;                   /* [nchains] Metropolis uniform                   */
    int32_t* inb;                /* [nchains] 1 = proposal within bounds           */
    int32_t* naccept;            /* [nchains] accepted proposals                   */
    int32_t* outbounds;          /* [nfree] out-of-bound counts (chain.py:242)     */
    double* best_chisq;          /* [nchains] lowest accepted chi-squared          */
    double* best_x;              /* [nchains, nfree] its free parameters           */
    int64_t* best_gen;           /* [nchains] generation where it was reached      */
    int64_t* gen_dev;            /* device generation counter (graph mode) or NULL */
    int64_t thinning;            /* generations per history row (graph mode)       */
    /* Multi-GPU exchange fused into the Metropolis kernel (peer stores over NVLink).
     * X_peers: NULL, or [world] device pointers (in device memory) to every
     * device's [2, nchains, nfree] population buffer; generation g reads half g&1
     * and k_metropolis writes every chain's next state (moved or not) into half
     * (g+1)&1 of EVERY device, so one cross-device barrier per generation orders
     * the exchange (X is then ignored).  Z_peers: NULL, or [world] pointers to
     * every device's history Z; thinned rows are stored to all of them (snooker). */
    double* const* X_peers;
    double* const* Z_peers;
    int32_t world, rank;
    /* Generation flags of the peer-memory exchange: NULL, or [world] device pointers
     * to every device's int64[world] flag array.  flag[p] on a device = generations
     * device p has completed with all its peer stores performed.  The kernel that
     * ends a generation (mc3b_model_chisq_ex with fuse + advance, or mc3b_advance)
     * writes gen+1 into flag[rank] of EVERY device (release, system scope);
     * mc3b_propose of generation gen waits until its own device's flags all read
     * >= gen (acquire): no barrier kernel, no collective call per generation. */
    int64_t* const* F_peers;
} mc3b_sampler_t;

/* Recorded random stream of one generation (replay mode), indexed by global
 * chain id; produced by the oracle's draw recorder from the reference's numpy
 * stream.  a/b: snooker iR1,iR2 or demc r1,r2 after the reference's fix-ups. */
typedef struct mc3b_draws {
    const double* normal;        /* [nfree] shared support draw (chain.py:185) */
    const int64_t* a;
    const int64_t* b;
    const int64_t* iz;           /* snooker jump: z row, -1 = none               */
    const double* usj;           /* snooker: uniform tested against 0.1          */
    const double* gs;            /* snooker jump: U(1.2, 2.2)                    */
    const double* u;             /* Metropolis uniform                           */
} mc3b_draws_t;

/* Proposal for generation `gen`, chains [c_begin, c_end) of this device's
 * slice (global ids): draws (Philox, keyed by seed/chain/generation), jump
 * (chain.py:195-232), nextp = X + jump, bounds test with outbounds counters
 * (chain.py:235-243), shared-parameter fill (chain.py:246-247), snooker
 * Metropolis factor (chain.py:251-255) and the Metropolis uniform.  zsize is
 * the number of history rows a snooker draw may use.  [host] s. */
int mc3b_propose(const mc3b_sampler_t* s, int64_t gen, int64_t zsize,
                 int64_t c_begin, int64_t c_end, void* stream);

/* Device-driven generations (so one captured CUDA graph can be replayed):
 * pass gen < 0 to mc3b_propose / mc3b_metropolis and they read the generation
 * g from *s->gen_dev and derive, for the lock-step history layout,
 *   zsize = M0 + (g / thinning) * nchains
 *   zrow0 = M0 + ((g+1)/thinning - 1) * nchains  if (g+1) % thinning == 0, else -1.
 * mc3b_advance increments *s->gen_dev (one thread) at the end of a generation. */
int mc3b_advance(const mc3b_sampler_t* s, void* stream);

/* Same, with every random number taken from `d` instead of Philox.  [host] s, d */
int mc3b_propose_replay(const mc3b_sampler_t* s, const mc3b_draws_t* d,
                        int64_t c_begin, int64_t c_end, void* stream);

/* Metropolis step for chains [c_begin, c_end): chisq* of chain c = sum over s of
 * partial[s*ldpartial + (c - c_off)] (fixed order) + priors; accept iff exp(0.5 (chisq - chisq*)) * mrfactor > u
 * (chain.py:257-274); update X, chisq_cur, naccept, per-chain best; when
 * zrow0 >= 0 write the thinned sample of chain c to history row zrow0 + c
 * (chain.py:276-289).  [host] s. */
int mc3b_metropolis(const mc3b_sampler_t* s, const double* partial,
                    int64_t ldpartial, int nsplit, int64_t c_off, int64_t gen,
                    int64_t zrow0, int64_t c_begin, int64_t c_end, void* stream);

/* Peer memory for the exchange above, mapped with CUDA IPC (one process per GPU of
 * one box).  mc3b_peer_alloc: zero-filled device buffer on the current device +
 * its 64-byte IPC handle [host].  mc3b_peer_open: map another process's buffer
 * into this one (peer access is enabled on demand); *ptr [host] receives the local
 * address.  mc3b_peer_close / mc3b_peer_free undo them.  These four,
 * mc3b_user_model_load and mc3b_user_batch_load are the only entry points that allocate. */
int mc3b_peer_alloc(int64_t nbytes, void** ptr, unsigned char* handle64);
int mc3b_peer_open(const unsigned char* handle64, void** ptr);
int mc3b_peer_close(void* ptr);
int mc3b_peer_free(void* ptr);

/* Device address of page-locked host memory mapped into the current device's address
 * space (cudaHostGetDevicePointer), e.g. for mc3b_moment_t.record; fails when `host` is
 * not such memory.  *dev [host]. */
int mc3b_host_device_pointer(void* host, void** dev);

/* Report-point counters of this device's chains, packed for one D2H copy
 * (replaces the hub's reads of the shared numaccept / outbounds / bestp arrays,
 * mcmc_driver.py:302-320): out[0] = accepted proposals summed over the device's
 * chains, out[1] = lowest accepted chi-squared (inf if none), out[2], out[3] = the
 * generation and chain where it was reached first (-1 if none), out[4 .. 4+nfree) =
 * its free parameters, out[4+nfree .. 4+2 nfree) = the out-of-bounds counters.
 * out: 4 + 2 nfree doubles.  [host] s. */
int mc3b_pack_counters(const mc3b_sampler_t* s, double* out, void* stream);

/* Small populations (<= 256 chains, one device, built-in model, data chi-squared):
 * run generations gen0 .. gen0+ngen-1 inside ONE resident CTA -- proposal,
 * model + chi-squared (a warp per chain), Metropolis step and history write per
 * generation, same Philox streams and lock-step semantics as mc3b_propose /
 * mc3b_model_chisq / mc3b_metropolis.  For launch-latency-bound problems (the
 * reference's everyday 7-21 chains on 1e2-1e4 points).
 * Writes gen0+ngen to *s->gen_dev when it is set.  [host] s. */
int mc3b_run_small(const mc3b_sampler_t* s, int model_id, int nmodel,
                   const double* x, const double* data, const double* invsig,
                   int64_t n, int64_t gen0, int64_t ngen, void* stream);

/* Many independent small problems at once, one resident CTA each (a catalogue of
 * fits on different data).  problems[b] describes problem b exactly as
 * mc3b_run_small takes it (pointers into that problem's own slices of the state,
 * its own seed, vectors and history); every problem has the nchains, npars, nfree,
 * sampler, M0, zlen and thinning of problem 0.  Problem b owns the data points
 * [offsets[b], offsets[b+1]) of x, data and invsig. */
typedef struct mc3b_batch {
    int64_t nproblems;
    const mc3b_sampler_t* problems;   /* [nproblems], device memory: each problem's state (pointers into its slices) */
    const int64_t* offsets;           /* [nproblems + 1], device: problem b owns points [offsets[b], offsets[b+1]) */
    const double* x; const double* data; const double* invsig;
    int32_t* status;                  /* [nproblems], device: 0 ok, 1 initial population not filled,
                                         2 shape differs from problem 0's or no data points,
                                         3 stopped by the convergence test (mc3b_batch_gelman_rubin) */
} mc3b_batch_t;

/* Initial population of every problem (mcmc_driver.py:229-278), one CTA per
 * problem: the trial points of mc3b_init_trials (same Philox counters and kickoff
 * rules), in rounds sized as Population.init_population sizes them (trials
 * min(max(M0 - got, 64) 1.25 + 64, 100 M0 - tried); the first need + max(8, need/100)
 * in-bounds ones evaluated, a warp per trial, chi-squared + prior terms; the first
 * `need` with a finite log-posterior taken in draw order; at most 100 M0 trials).
 * Writes Z[0:M0], log_post[0:M0], X = Z[0:nchains], chisq_cur = -2 log_post[0:nchains]
 * and status[b].  model_id / nmodel / kickoff as mc3b_run_small / mc3b_init_trials. */
int mc3b_batch_init(const mc3b_batch_t* b, int model_id, int nmodel, int kickoff, void* stream);

/* mc3b_run_small over every problem whose status is 0, one CTA per problem
 * (Chain.run, mc3/chain.py:183-299): generations gen0 .. gen0+ngen-1, the same
 * arithmetic, bit for bit, as mc3b_run_small on that problem alone.  The per-problem
 * gen_dev is ignored.  Split into launches of at most 200 000 generations. */
int mc3b_batch_run(const mc3b_batch_t* b, int model_id, int nmodel, int64_t gen0, int64_t ngen, void* stream);

/* Gelman-Rubin at report point k (k thinned steps done) of every problem whose status is
 * 0 (mcmc_driver.py:325-346, gelman.py:36-92), one CTA per problem; model-independent, so
 * it serves mc3b_batch_run and mc3b_user_batch_run alike:
 *   psrf[b * ldpsrf + p]  PSRF of free parameter p over thinned steps [zburn, k) (lock-step
 *                         rows M0 + k' nchains + c), bit for bit mc3b_gelman_rubin on that
 *                         problem's history; left untouched for the problems it skips
 *   grbreak > 0, every psrf < grbreak (NaN never passes) and M0 + k nchains > grnmin:
 *                         status[b] = 3 and kstop[b] = k, so that later mc3b_batch_run /
 *                         mc3b_user_batch_run launches skip the problem.
 * Needs nchains >= 2, 0 <= zburn < k, M0 + k nchains <= zlen, ldpsrf >= nfree; kstop may
 * be NULL when grbreak <= 0.  Reads problem 0's description back as mc3b_batch_run does. */
int mc3b_batch_gelman_rubin(const mc3b_batch_t* b, int64_t k, int64_t zburn, double grbreak,
                            int64_t grnmin, double* psrf, int64_t ldpsrf, int64_t* kstop, void* stream);

/* The batch of a user model (mc3b_user_model_desc_t, fp64 only): k_init_batch, k_run_batch
 * and a batched model-value kernel compiled by NVRTC into a module of their own, so that
 * mc3b_user_model_compile_desc's module and compile time do not change.  A handle of one
 * kind cannot be launched as the other.  Each launch takes, besides the batch:
 *   xs [host]     nx == ninputs device pointers, input j of every problem concatenated as
 *                 mc3b_batch_t.x is (problem b owns [offsets[b], offsets[b+1])), xs[0] == b->x
 *   consts        [nproblems, nk] device, nk == nconst: problem b's constants in row b (the
 *                 values its chains see in p[nmodel .. nmodel + nk)); NULL only when nk == 0
 * and every problem has npars == nmodel.  mc3b_user_batch_compile / _load as
 * mc3b_user_model_compile_desc / _load_desc (the module carries its own ABI record: one
 * built against another sampler or batch layout is refused, MC3B_ERR_ARG). */
typedef struct mc3b_user_batch mc3b_user_batch_t;          /* opaque */

int mc3b_user_batch_compile(const char* nvrtc_path, const char* source,
                            const mc3b_user_model_desc_t* desc /*[host]*/,
                            void* cubin /*[host]*/, int64_t cap, int64_t* size /*[host]*/,
                            char* log /*[host]*/, int64_t logcap);
int mc3b_user_batch_load(const void* cubin /*[host]*/, int64_t size,
                         const mc3b_user_model_desc_t* desc /*[host]*/,
                         mc3b_user_batch_t** out /*[host]*/);
int mc3b_user_batch_free(mc3b_user_batch_t* m);

/* mc3b_batch_init for a user model (mcmc_driver.py:229-278, one CTA per problem). */
int mc3b_user_batch_init(const mc3b_user_batch_t* m, const mc3b_batch_t* b,
                         const double* const* xs /*[host] nx device pointers*/, int nx,
                         const double* consts, int nk, int kickoff, void* stream);

/* mc3b_batch_run for a user model (Chain.run, mc3/chain.py:183-299): launches of at most
 * 200 000 generations. */
int mc3b_user_batch_run(const mc3b_user_batch_t* m, const mc3b_batch_t* b,
                        const double* const* xs /*[host] nx device pointers*/, int nx,
                        const double* consts, int nk, int64_t gen0, int64_t ngen, void* stream);

/* mc3b_model_eval for a user model and every problem of a batch in one launch (the
 * best_model of each output dictionary): out[i] = model(params + b * ldp) at point i of
 * problem b, for i in [offsets[b], offsets[b+1]); out has the layout of b->x. */
int mc3b_user_batch_eval(const mc3b_user_batch_t* m, const mc3b_batch_t* b,
                         const double* const* xs /*[host] nx device pointers*/, int nx,
                         const double* consts, int nk, const double* params, int64_t ldp,
                         double* out, void* stream);

/* Trial points of the initial population (mcmc_driver.py:229-262):
 * trial[t, :] = params0 with free entries drawn N(params0, pstep) (kickoff 0)
 * or U(pmin, pmax) (kickoff 1), shared parameters filled; ok[t] = 1 when all
 * parameters are inside [pmin, pmax].  Trial t uses Philox counter
 * (t, slot, round, 0xFFFFFFFF).  [host] s. */
int mc3b_init_trials(const mc3b_sampler_t* s, int kickoff, int64_t ntrials,
                     int64_t round, double* trial, int32_t* ok, void* stream);

/* log_prior of nrows history rows Z [nrows, nfree] (mc3/stats/stats.py:367-392):
 * lpr = -0.5 sum_j t_j^2, t_j = (z_j - prior)/priorlow|priorup for Gaussian priors,
 * 2 log z_j where priorlow < 0, else 0 (prior* are [npars], ifree maps columns);
 * and/or chisq = -2 (log_post - lpr) as update_output builds it (stats.py:822).
 * lpr or chisq may be NULL. */
int mc3b_log_prior(const double* Z, int64_t nrows, int nfree,
                   const int32_t* ifree, const double* prior,
                   const double* priorlow, const double* priorup,
                   const double* log_post, double* lpr, double* chisq,
                   void* stream);

/* Gelman-Rubin PSRF per free parameter (gelman.py:36-92) over samples
 * k = burnin .. burnin+niter-1 of every chain; sample k of chain c is history
 * row  rows[c*ldr + k]  when rows != NULL, else  M0 + k*nchains + c  (the
 * lock-step layout).  work: [2, nchains, nfree] fp64.  psrf: [nfree]. */
int mc3b_gelman_rubin(const double* Z, int64_t nfree, int64_t nchains,
                      int64_t M0, const int64_t* rows, int64_t ldr,
                      int64_t burnin, int64_t niter, double* work, double* psrf,
                      void* stream);

/* The two stages of mc3b_gelman_rubin, for chains spread over devices: every
 * device fills work[0, c, :] (mean) and work[1, c, :] (population variance,
 * gelman.py:75-76) for ITS chains [c_begin, c_end) from its own history rows; the
 * caller all-gathers the two [nchains, nfree] blocks (2 nchains nfree doubles -- not
 * the history) and every device evaluates W, B, V, sqrt(V/W) over all chains in chain
 * order (gelman.py:77-92): identical bits to the one-device call. */
int mc3b_gelman_rubin_moments(const double* Z, int64_t nfree, int64_t nchains,
                              int64_t M0, const int64_t* rows, int64_t ldr,
                              int64_t burnin, int64_t niter, int64_t c_begin,
                              int64_t c_end, double* work, void* stream);
int mc3b_gelman_rubin_psrf(const double* work, int64_t nfree, int64_t nchains,
                           int64_t niter, double* psrf, void* stream);

/* ------------------------------------------------------------------------
 * Wavelet likelihood   (replaces _dwt.c + wavelet.h)
 * ---------------------------------------------------------------------- */

/* Bytes of workspace mc3b_dwt_chisq needs for (nchains, n). */
int64_t mc3b_dwt_workspace(int64_t nchains, int64_t n);

/* Carter & Winn (2009) wavelet pseudo chi-squared, batched over chains, for
 * n = 2^k >= 4 only (the reference is undefined elsewhere, see DESIGN.md):
 * residual = data - model, D4 pyramid, per-scale sums, log terms
 * (_dwt.c:71-118).  gamma, sigma_r, sigma_w are params[c, npars-3 .. npars-1].
 * Model: built-in (model_id >= 0, evaluated from params[c, 0..nmodel) on x) or
 * given (model_id < 0, `model` is [nchains, ldm]).  Priors are NOT added here
 * (use mc3b_chisq_finish with nsplit = 1 or mc3b_metropolis). */
int mc3b_dwt_chisq(int model_id, const double* params, int64_t ldp,
                   int64_t nchains, int npars, int nmodel, const double* x,
                   const double* model, int64_t ldm, const double* data,
                   int64_t n, void* workspace, double* chisq, void* stream);

/* mc3b_dwt_chisq for a user model (_dwt.c:71-118 with the model of chain.py:317
 * evaluated on the device): the model reads params[c, 0..nmodel), its nx inputs xs
 * [host] (nx device pointers of n points) and its nk constants (fp64, device; NULL
 * when nk = 0), and its values go straight into the D4 pyramid, never to memory.
 * Same workspace (mc3b_dwt_workspace), checks and results as a built-in model; nx
 * and nk must equal the handle's, nmodel <= npars - 3.  The wavelet likelihood is
 * fp64: the handle must be the model's fp64 module (MC3B_ERR_ARG otherwise). */
int mc3b_user_model_dwt_chisq(const mc3b_user_model_t* m, const double* params,
                              int64_t ldp, int64_t nchains, int npars,
                              const double* const* xs /*[host] nx device pointers*/,
                              int nx, const double* consts, int nk,
                              const double* data, int64_t n, void* workspace,
                              double* chisq, void* stream);

/* _dwt.daub4: forward (isign >= 0) or inverse (isign < 0) D4 transform of a
 * length-n2 array, n2 = 2^k >= 4; workspace holds n2 doubles; in and out
 * must not alias.  Zero padding to 2^k is the caller's (stats.dwt_daub4 does it). */
int mc3b_daub4(const double* in, int64_t n2, int isign, void* workspace,
               double* out, void* stream);

/* ------------------------------------------------------------------------
 * Time-series diagnostics   (replace _time_averaging.c and _binarray.c)
 * ---------------------------------------------------------------------- */

/* Bytes of workspace for mc3b_binrms on n points. */
int64_t mc3b_binrms_workspace(int64_t n, int64_t maxbins, int64_t binstep);

/* _time_averaging.binrms: for bin sizes b = 1, 1+binstep, ... <= maxbins:
 * rms of the bin means, its lower/upper errors (asymptotic for more than 35
 * bins, inverse-gamma credible region otherwise), the Gaussian extrapolation
 * stderr and b.  Outputs have (maxbins-1)/binstep + 1 entries. */
int mc3b_binrms(const double* data, int64_t n, int64_t maxbins,
                int64_t binstep, void* workspace, double* rms, double* rmslo,
                double* rmshi, double* stderr_, double* binsz, void* stream);

/* _binarray.binarray: n/binsize bin means; with uncert != NULL, 1/sigma^2
 * weighted means and binstd = sqrt(1/sum(1/sigma^2)) (binstd may be NULL
 * otherwise). */
int mc3b_binarray(const double* data, int64_t n, int64_t binsize,
                  const double* uncert, double* bindata, double* binstd,
                  void* stream);

/* ------------------------------------------------------------------------
 * Posterior statistics   (replace the scipy/numpy path of stats.py:433-467, 764-802)
 * ---------------------------------------------------------------------- */

/* Bytes of workspace for mc3b_hpd. */
int64_t mc3b_hpd_workspace(int nfree);

/* Highest-posterior-density statistics of the marginals of posterior [n, nfree]
 * (row-major fp64), per column as the reference's cred_region + marginal_statistics
 * ('max_like'): Gaussian kernel density with Scott's bandwidth (scipy.stats.
 * gaussian_kde) on every (n/120000)-th sample, traced at 100 points inside
 * [max(mean - 6 std, min), min(mean + 6 std, max)], resampled linearly to 3000
 * points, density threshold where the descending running sum reaches `quantile`
 * of the total.  out [3, nfree]: mode, lowest and highest point above the
 * threshold. */
int mc3b_hpd(const double* posterior, int64_t n, int nfree, double quantile,
             void* workspace, double* out, void* stream);

/* ------------------------------------------------------------------------
 * Roofline denominators
 * ---------------------------------------------------------------------- */

/* Register-resident FMA chains on every SM: runs `iters` dependent FMAs per
 * accumulator; *flops receives the flop count of the launch (2 per FMA).
 * Time it with events to get the FP64 / FP32 pipe peak. */
int mc3b_fma_peak(int dtype, int64_t iters, double* sink, double* flops /*[host]*/,
                  void* stream);

/* Same, with the operand kinds and parallelism of the model kernel (fp64):
 * variant 1 = 8 chains/thread with constant-bank operands, 2 = 4 chains/thread
 * at 6 CTAs of 128 threads per SM, 3 = 2 chains, 4 = 1 chain at 8 CTAs of 128.
 * Used to read the FP64 dependent-issue latency off the device. */
int mc3b_fma_peak_variant(int variant, int64_t iters, double* sink,
                          double* flops /*[host]*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MC3B200_H */
