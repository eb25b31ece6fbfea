// mc3_b200 -- the D4 kernels of the wavelet likelihood that read the model.
// Device code only: dwt.cu instantiates them for the built-in models, jit.cu has NVRTC
// instantiate them for a user model (fp64 modules; the header travels inside the library
// as a string, csrc/jit_headers.inc written by build.py).  The passes after the first
// read coefficients, not the model: they are the library's own (dwt.cu, SRC_ARRAY).
//
//   k_dwt_reg_model  register stage (4 levels), x/data staged once per CTA
//   k_dwt_pass       one warp per chain, 8 chains per CTA sharing the x/data tile.
//                    A tile of T inputs + halo H = 2^(L+1)-2 (taken modulo n, which
//                    reproduces the periodic wrap) goes through L levels inside
//                    shared memory; the T/2^L smooth outputs go to a workspace, the
//                    per-level detail sums stay in registers across the tiles of a
//                    span -> sums[chain, level, span].
//   k_dwt_last       finishes the pyramid of the <=512 remaining coefficients in
//                    shared memory, adds the span sums in fixed order and evaluates
//                    the likelihood terms.
//
// A model of NX > 1 per-point inputs (models.cuh ninputs_of) reads input j from xs[j];
// a model of run-time constants (takes_consts) loads them from uconst.
#pragma once
#include "models.cuh"
#ifndef M_PI                   // NVRTC has no math.h: its value there
#define M_PI 3.14159265358979323846
#endif

// NVRTC: a named namespace, so that the instantiations have names the loader can
// look up (jit.cu); the library keeps them local to dwt.cu.
#ifdef __CUDACC_RTC__
namespace mc3b_jit {
#else
namespace {
#endif

constexpr int CH = 8;          // chains (warps) per CTA
constexpr int T = 512;         // inputs per tile
constexpr int LMAX = 6;        // levels per pass
constexpr int LASTMAX = 512;   // coefficients finished by k_dwt_last
constexpr int MAXSPAN = 64;
constexpr int MAXLEV = 40;

__device__ __constant__ double kC[4] = {0.4829629131445341, 0.83651630373780772, 0.22414386804201339,
                                        -0.12940952255126034};

enum { SRC_MODEL = 0, SRC_GIVEN = 1, SRC_ARRAY = 2 };

// compile-time flag for the block lambdas (NVRTC has no <type_traits>)
template <bool B> struct dwt_flag { static constexpr bool value = B; };

// load(p), or load(p, k) with the constants of the argument block a (takes_consts)
template <class M, class A> __device__ __forceinline__ void dwt_load(M& m, const double* p, const A& a) {
    if constexpr (takes_consts<M>::value) m.load(p, a.uconst);
    else m.load(p);
}

struct PassArgs {
    const double* params; int64_t ldp; int64_t nchains;
    const double* x; const double* data;         // SRC_MODEL / SRC_GIVEN
    const double* rows; int64_t ldr;              // SRC_GIVEN: model rows; SRC_ARRAY: input coefficients
    int64_t n_in;                                 // input length (2^k)
    int L;                                        // levels in this pass
    int lev0;                                     // levels done before this pass
    int spans, tiles_per_span;
    double* out; int64_t ldo;                     // smooth output rows
    double* sums;                                 // [nchains, MAXLEV, MAXSPAN]
};
// The argument blocks of a user model's kernels: the block of the built-in ones, then the
// model's inputs (xs[0] = x) and its constants (nullptr when it has none).  The built-in
// kernels keep the smaller block: a larger one changes their code.
struct PassArgsX : PassArgs { const double* xs[MC3B_MAX_INPUTS]; const double* uconst; };

constexpr int PB0 = T + (2 << LMAX);              // doubles of a staged row / of a warp's buf0
// dynamic shared memory of k_dwt_pass for a model of nx inputs: x, data, the warps'
// buffers, then inputs 2..nx
inline size_t pass_smem(int nx) {
    return (size_t)(2 * PB0 + CH * (PB0 * 3 / 2) + (nx - 1) * PB0) * sizeof(double);
}

// A: PassArgs, or PassArgsX for a user model
template <int SRC, class M, class A>
__global__ void __launch_bounds__(CH * 32) k_dwt_pass(A a) {
    constexpr int NX = ninputs_of<M>::value;
    extern __shared__ __align__(16) double smem[];
    const int H = (2 << a.L) - 2;
    const int len0 = T + H;
    double* sx = smem;                               // [len0] (SRC_MODEL)
    double* sd = sx + (T + (2 << LMAX));             // [len0]
    double* wbuf = sd + (T + (2 << LMAX));           // per warp: buf0[len0max] + buf1[len0max/2]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int B0 = T + (2 << LMAX), B1 = B0 / 2;
    double* buf0 = wbuf + (size_t)warp * (B0 + B1);
    double* buf1 = buf0 + B0;
    double* sxe = wbuf + (size_t)CH * (B0 + B1);     // inputs 2..NX: [NX-1][B0] (SRC_MODEL)

    int64_t c = (int64_t)blockIdx.x * CH + warp;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;
    M mdl;
    if (SRC == SRC_MODEL) dwt_load(mdl, a.params + c * a.ldp, a);
    const double c0 = kC[0], c1 = kC[1], c2 = kC[2], c3 = kC[3];
    double acc[LMAX];
#pragma unroll
    for (int l = 0; l < LMAX; l++) acc[l] = 0.0;
    const int64_t mask = a.n_in - 1;

    for (int ts = 0; ts < a.tiles_per_span; ts++) {
        const int64_t tile = (int64_t)blockIdx.y * a.tiles_per_span + ts;
        const int64_t g0 = tile * T;
        if (SRC == SRC_MODEL) {
            __syncthreads();
            for (int i = threadIdx.x; i < len0; i += CH * 32) {
                const int64_t g = (g0 + i) & mask;
                sx[i] = a.x[g];
                if constexpr (NX > 1) {
#pragma unroll
                    for (int j = 1; j < NX; j++) sxe[(j - 1) * B0 + i] = a.xs[j][g];
                }
                sd[i] = a.data[g];
            }
            __syncthreads();
            if constexpr (NX == 1) {
                for (int i = lane; i < len0; i += 32) buf0[i] = sd[i] - mdl.eval_safe(sx[i]);
            } else {
                for (int i = lane; i < len0; i += 32) {
                    double v[NX];
                    v[0] = sx[i];
#pragma unroll
                    for (int j = 1; j < NX; j++) v[j] = sxe[(j - 1) * B0 + i];
                    buf0[i] = sd[i] - mdl.eval_safe(v);
                }
            }
        } else if (SRC == SRC_GIVEN) {
            const double* m = a.rows + c * a.ldr;
            for (int i = lane; i < len0; i += 32) {
                const int64_t g = (g0 + i) & mask;
                buf0[i] = a.data[g] - m[g];
            }
        } else {
            const double* m = a.rows + c * a.ldr;
            for (int i = lane; i < len0; i += 32) buf0[i] = m[(g0 + i) & mask];
        }
        __syncwarp();
        double* in = buf0;
        double* ot = buf1;
        int len = len0;
#pragma unroll
        for (int l = 1; l <= LMAX; l++) {
            if (l <= a.L) {
                const int lo = (len - 2) >> 1;
                const int own = T >> l;
                double s2 = 0.0;
                for (int j = lane; j < lo; j += 32) {
                    const double a0 = in[2 * j], a1 = in[2 * j + 1], a2 = in[2 * j + 2], a3 = in[2 * j + 3];
                    ot[j] = c0 * a0 + c1 * a1 + c2 * a2 + c3 * a3;
                    if (j < own) {
                        const double d = c3 * a0 - c2 * a1 + c1 * a2 - c0 * a3;
                        s2 = fma(d, d, s2);
                    }
                }
                acc[l - 1] += s2;
                __syncwarp();
                double* t = in; in = ot; ot = t;
                len = lo;
            }
        }
        if (live) {
            double* o = a.out + c * a.ldo + (g0 >> a.L);
            for (int j = lane; j < (T >> a.L); j += 32) o[j] = in[j];
        }
        __syncwarp();
    }
#pragma unroll
    for (int l = 0; l < LMAX; l++) {
        if (l < a.L) {
            double v = acc[l];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0 && live) a.sums[(c * MAXLEV + (a.lev0 + l)) * MAXSPAN + blockIdx.y] = v;
        }
    }
}

// ---- register stage: 4 levels per pass without the shared-memory round trips --
// A warp takes blocks of 512 consecutive inputs of its chain (read modulo n).
// The block is loaded/evaluated coalesced, transposed once through a padded
// shared-memory row so that lane l owns inputs [16 l, 16 l + 16), and the four
// levels then run in registers: each level needs two values of the next lane
// (shuffle) and halves the lane's values (16 -> 8 -> 4 -> 2 -> 1).  Lane 31 has
// no right neighbour, so the last 2 of the 32 level-4 outputs are not valid:
// blocks advance by 480 inputs (30 outputs) and an output is counted by the
// block that owns its first input.  Shared-memory traffic drops from ~64 to 16
// bytes per input; the FP64 pipe becomes the limiter.
constexpr int RB = 512;             // inputs per block
constexpr int RADV = 480;           // block advance (30 lanes x 16)

struct RegArgs {
    const double* params; int64_t ldp; int64_t nchains;
    const double* x; const double* data;
    const double* rows; int64_t ldr;
    int64_t n_in;
    int lev0;
    int64_t nblocks; int blocks_per_span;
    double* out; int64_t ldo;
    double* sums;
};
struct RegArgsX : RegArgs { const double* xs[MC3B_MAX_INPUTS]; const double* uconst; };

// The model's first pass: the 8 chains of a CTA walk the same blocks, so x and data are
// staged ONCE per CTA (double-buffered, padded rows of 18 so that a lane's 16
// consecutive values are conflict-free 16-byte reads) and every warp evaluates
// its own chain's residuals straight into the lane-contiguous registers -- no
// per-warp transpose.  L1/shared-memory wavefronts per block and warp: ~80
// instead of 128.  A model of NX inputs stages NX + 1 rows (46 KB at NX = 4).
constexpr int RPAD = 18;                         // doubles per 16-value row

// A: RegArgs, or RegArgsX for a user model
template <class M, class A>
__global__ void __launch_bounds__(CH * 32) k_dwt_reg_model(A a) {
    constexpr int NX = ninputs_of<M>::value;
    __shared__ __align__(16) double sxd[2][NX + 1][32 * RPAD];   // inputs, then data
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t c = (int64_t)blockIdx.x * CH + warp;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;
    M mdl;
    dwt_load(mdl, a.params + c * a.ldp, a);
    const double c0 = kC[0], c1 = kC[1], c2 = kC[2], c3 = kC[3];
    const int64_t mask = a.n_in - 1;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    const int64_t b_begin = (int64_t)blockIdx.y * a.blocks_per_span;
    int64_t b_end = b_begin + a.blocks_per_span;
    if (b_end > a.nblocks) b_end = a.nblocks;
    auto fill = [&](int64_t b, int buf) {
        const int64_t g0 = b * RADV;
#pragma unroll
        for (int q = 0; q < RB / (CH * 32); q++) {
            const int idx = q * CH * 32 + threadIdx.x;
            const int64_t g = (g0 + idx) & mask;
            const int pos = (idx >> 4) * RPAD + (idx & 15);
            sxd[buf][0][pos] = a.x[g];
            if constexpr (NX > 1) {
#pragma unroll
                for (int j = 1; j < NX; j++) sxd[buf][j][pos] = a.xs[j][g];
            }
            sxd[buf][NX][pos] = a.data[g];
        }
    };
    if (b_begin < b_end) fill(b_begin, 0);
    // One block; INTERIOR (compile time): every output the block owns exists, so the
    // squares are summed without a per-element select (the ALU pipe was as busy as the
    // FP64 pipe: profiles/r2_dwt_reg_model.md).
    auto do_block = [&](int64_t b, int buf, auto interior_tag) {
        constexpr bool interior = decltype(interior_tag)::value;
        const int64_t g0 = b * RADV;
        double v[18];
        const double2* px = reinterpret_cast<const double2*>(&sxd[buf][0][lane * RPAD]);
        const double2* pd = reinterpret_cast<const double2*>(&sxd[buf][NX][lane * RPAD]);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const double2 xv = px[k], dv = pd[k];
            if constexpr (NX == 1) {
                v[2 * k] = dv.x - mdl.eval_safe(xv.x);
                v[2 * k + 1] = dv.y - mdl.eval_safe(xv.y);
            } else {
                double u0[NX], u1[NX];
                u0[0] = xv.x;
                u1[0] = xv.y;
#pragma unroll
                for (int j = 1; j < NX; j++) {
                    const double2 xj = reinterpret_cast<const double2*>(&sxd[buf][j][lane * RPAD])[k];
                    u0[j] = xj.x;
                    u1[j] = xj.y;
                }
                v[2 * k] = dv.x - mdl.eval_safe(u0);
                v[2 * k + 1] = dv.y - mdl.eval_safe(u1);
            }
        }
        int cnt = 16;
#pragma unroll
        for (int l = 0; l < 4; l++) {
            v[cnt] = __shfl_down_sync(0xffffffffu, v[0], 1);
            v[cnt + 1] = __shfl_down_sync(0xffffffffu, v[1], 1);
            const int half = cnt >> 1;
            const int64_t lev_pos0 = (g0 >> (l + 1)) + (int64_t)lane * half;
            const int64_t lev_n = a.n_in >> (l + 1);
            double s2 = 0.0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                if (j < half) {
                    const double a0 = v[2 * j], a1 = v[2 * j + 1], a2 = v[2 * j + 2], a3 = v[2 * j + 3];
                    const double sm = fma(c3, a3, fma(c2, a2, fma(c1, a1, c0 * a0)));
                    const double d = fma(-c0, a3, fma(c1, a2, fma(-c2, a1, c3 * a0)));
                    if (interior) s2 = fma(d, d, s2);
                    else s2 = fma(d, (lev_pos0 + j < lev_n) ? d : 0.0, s2);
                    v[j] = sm;
                }
            }
            acc[l] += (lane < 30) ? s2 : 0.0;
            cnt = half;
        }
        const int64_t o = (g0 >> 4) + lane;
        if (live && lane < 30 && (interior || o < (a.n_in >> 4))) a.out[c * a.ldo + o] = v[0];
    };
    for (int64_t b = b_begin; b < b_end; b++) {
        const int buf = (int)((b - b_begin) & 1);
        __syncthreads();                             // tile b is complete; tile b-1 is no longer read
        if (b + 1 < b_end) fill(b + 1, buf ^ 1);
        if (b * RADV + RB <= a.n_in) do_block(b, buf, dwt_flag<true>{});
        else do_block(b, buf, dwt_flag<false>{});
    }
#pragma unroll
    for (int l = 0; l < 4; l++) {
        double t = acc[l];
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0 && live) a.sums[(c * MAXLEV + (a.lev0 + l)) * MAXSPAN + blockIdx.y] = t;
    }
}

struct LastArgs {
    const double* params; int64_t ldp; int npars; int64_t nchains;
    const double* x; const double* data;
    const double* rows; int64_t ldr;
    int n0;                      // coefficients to finish (4..512, 2^j)
    int lev0;                    // levels done by the passes
    int kbits;                   // n = 2^kbits
    const double* sums;          // [nchains, MAXLEV, MAXSPAN]
    int spans_of_level[MAXLEV];  // spans that hold level l (levels done by the passes)
    double* chisq;
};
struct LastArgsX : LastArgs { const double* xs[MC3B_MAX_INPUTS]; const double* uconst; };
constexpr int CHL = 4;           // chains (warps) per CTA of k_dwt_last

// A: LastArgs, or LastArgsX for a user model
template <int SRC, class M, class A>
__global__ void __launch_bounds__(CHL * 32) k_dwt_last(A a) {
    constexpr int NX = ninputs_of<M>::value;
    __shared__ double wb[CHL][LASTMAX + LASTMAX / 2];
    __shared__ double lev_s2[CHL][MAXLEV];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t c = (int64_t)blockIdx.x * CHL + warp;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;
    double* in = wb[warp];
    double* ot = in + LASTMAX;
    const double c0 = kC[0], c1 = kC[1], c2 = kC[2], c3 = kC[3];
    if (SRC == SRC_MODEL) {
        M mdl;
        dwt_load(mdl, a.params + c * a.ldp, a);
        if constexpr (NX == 1) {
            for (int i = lane; i < a.n0; i += 32) in[i] = a.data[i] - mdl.eval_safe(a.x[i]);
        } else {
            for (int i = lane; i < a.n0; i += 32) {
                double v[NX];
                v[0] = a.x[i];
#pragma unroll
                for (int j = 1; j < NX; j++) v[j] = a.xs[j][i];
                in[i] = a.data[i] - mdl.eval_safe(v);
            }
        }
    } else if (SRC == SRC_GIVEN) {
        const double* m = a.rows + c * a.ldr;
        for (int i = lane; i < a.n0; i += 32) in[i] = a.data[i] - m[i];
    } else {
        const double* m = a.rows + c * a.ldr;
        for (int i = lane; i < a.n0; i += 32) in[i] = m[i];
    }
    __syncwarp();
    int lev = a.lev0;
    for (int nn = a.n0; nn >= 4; nn >>= 1, lev++) {
        const int nh = nn >> 1;
        double s2 = 0.0;
        for (int j = lane; j < nh; j += 32) {
            const double a0 = in[2 * j], a1 = in[2 * j + 1], a2 = in[(2 * j + 2) & (nn - 1)],
                         a3 = in[(2 * j + 3) & (nn - 1)];
            ot[j] = c0 * a0 + c1 * a1 + c2 * a2 + c3 * a3;
            const double d = c3 * a0 - c2 * a1 + c1 * a2 - c0 * a3;
            s2 = fma(d, d, s2);
        }
        for (int o = 16; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        if (lane == 0) lev_s2[warp][lev] = s2;
        __syncwarp();
        double* t = in; in = ot; ot = t;
    }
    // levels done by the passes: add their span sums in span order
    for (int l = lane; l < a.lev0; l += 32) {
        double s = 0.0;
        const int ns = a.spans_of_level[l];
        const double* p = a.sums + (c * MAXLEV + l) * MAXSPAN;
        for (int k = 0; k < ns; k++) s += p[k];
        lev_s2[warp][l] = s;
    }
    __syncwarp();
    if (lane == 0 && live) {                        // _dwt.c:96-110
        const double* p = a.params + c * a.ldp;
        const double gamma = p[a.npars - 3], sr = p[a.npars - 2], sw = p[a.npars - 1];
        const double g = 0.72134752;
        const double sS2 = sr * sr * pow(2.0, -gamma) * g + sw * sw;
        double chi = in[0] * in[0] / sS2 + in[1] * in[1] / sS2 + 2.0 * log(2.0 * M_PI * sS2);
        const int Msc = a.kbits;
        for (int m = 1; m < Msc; m++) {
            const double sW2 = sr * sr * pow(2.0, -gamma * m) + sw * sw;
            const double cnt = (double)(1 << m);
            chi += lev_s2[warp][Msc - 1 - m] / sW2 + cnt * log(2.0 * M_PI * sW2);
        }
        a.chisq[c] = chi;
    }
}

}  // namespace

#ifndef __CUDACC_RTC__
// dwt.cu: the wavelet chi-squared of a user model (jit.cu).  Its first pass -- pass 0, or
// the last pass when n <= 512 -- runs on the kernels of the model's module (reg =
// k_dwt_reg_model, pass = k_dwt_pass<SRC_MODEL>, whose dynamic shared-memory attribute the
// loader set to pass_smem(nx), last = k_dwt_last<SRC_MODEL>); every later pass on the
// library's own.  xs: nx device pointers, consts: the model's constants or nullptr.
struct DwtUserModel {
    const void* reg; const void* pass; const void* last;
    int nx, nmodel;
    const double* const* xs;
    const double* consts;
};
int mc3b_dwt_chisq_user(const DwtUserModel& u, const double* params, int64_t ldp, int64_t nchains, int npars,
                        const double* data, int64_t n, void* workspace, double* chisq, cudaStream_t st);
#endif
