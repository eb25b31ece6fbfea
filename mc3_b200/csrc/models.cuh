// mc3_b200 -- built-in model functions, evaluated per (chain, data point).
//
// The reference has no built-in models: its `func` is user Python evaluated
// once per chain-step (mc3/chain.py:316-319, ~90% of its run time).  These
// functors are the CUDA side of BASELINE.json's north_star item (2); their
// numpy twins for the oracle live in oracle/models.py (same formulas, same
// parameter order).  load() runs once per chain per launch and hoists every
// per-chain constant; eval() is the per-point cost.
#pragma once
#include "common.cuh"

// Branch-free fp64 sine: 14 FP64-pipe instructions against ~35 (plus a divergent
// sin/cos kernel choice) of the CUDA library's sin().  Reduction modulo pi with a
// two-constant Cody-Waite step (each FMA rounds once, so the reduced argument
// carries <= 4e-16 absolute error for any |a| < 1e9), odd polynomial of degree 17
// on [-pi/2, pi/2] (near-minimax fit, max error 3.6e-17 + rounding), sign from
// the parity of the quotient.  Measured against numpy.sin in
// tests/test_gpu_kernels.py::test_fast_sin_accuracy.  Huge or non-finite
// arguments take the library path.
__device__ __constant__ double kSinC[12] = {
    0.3183098861837907,          // 1/pi
    -3.141592653589793,          // -pi (high part)
    -1.2246467991473532e-16,     // -pi (low part)
    2.7314447669863995e-15, -7.643970296798572e-13, 1.6058977312464087e-10, -2.5052107616996182e-08,
    2.7557319219163234e-06, -0.00019841269841254974, 0.008333333333333316, -0.16666666666666666, 0.0};
#define MC3B_SIN_MAGIC 6755399441055744.0               // 1.5 * 2^52

// sin(a), no branches; `magic` holds MC3B_SIN_MAGIC in a register (so the FMA
// below can take 1/pi from a uniform register).  Low word of t = rint(a/pi).
__device__ __forceinline__ double fast_sin_core(double a, double magic) {
    const double t = fma(a, kSinC[0], magic);
    const double q = t - magic;
    double r = fma(q, kSinC[1], a);
    r = fma(q, kSinC[2], r);
    const double s = r * r;
    double p = fma(s, kSinC[3], kSinC[4]);
    p = fma(p, s, kSinC[5]);
    p = fma(p, s, kSinC[6]);
    p = fma(p, s, kSinC[7]);
    p = fma(p, s, kSinC[8]);
    p = fma(p, s, kSinC[9]);
    p = fma(p, s, kSinC[10]);
    const double v = fma(r * s, p, r);
    return __hiloint2double(__double2hiint(v) ^ (__double2loint(t) << 31), __double2loint(v));
}
// sin and cos of the same argument (shared reduction); cos(r) = 1 - s/2 + s^2 Q(s),
// Q of degree 6 (near-minimax, max error 7e-17 on [-pi/2, pi/2]).
__device__ __constant__ double kCosC[8] = {
    4.6464359591124806e-14, -1.1466252259718479e-11, 2.0876681558867395e-09, -2.7557318573366175e-07,
    2.480158729891355e-05, -0.0013888888888884767, 0.04166666666666666, 0.0};

__device__ __forceinline__ void fast_sincos_core(double a, double& sn, double& cs) {
    const double t = fma(a, kSinC[0], MC3B_SIN_MAGIC);
    const double q = t - MC3B_SIN_MAGIC;
    double r = fma(q, kSinC[1], a);
    r = fma(q, kSinC[2], r);
    const double s = r * r;
    double p = fma(s, kSinC[3], kSinC[4]);
    double h = fma(s, kCosC[0], kCosC[1]);
#pragma unroll
    for (int i = 5; i <= 10; i++) p = fma(p, s, kSinC[i]);
#pragma unroll
    for (int i = 2; i <= 6; i++) h = fma(h, s, kCosC[i]);
    const double v = fma(r * s, p, r);
    const double w = fma(s * s, h, fma(s, -0.5, 1.0));
    const int flip = __double2loint(t) << 31;
    sn = __hiloint2double(__double2hiint(v) ^ flip, __double2loint(v));
    cs = __hiloint2double(__double2hiint(w) ^ flip, __double2loint(w));
}

// The fast path is valid for |a| < 1e9 (finite); callers check with this.
__device__ __forceinline__ int sin_arg_key(double a) { return __double2hiint(a) & 0x7fffffff; }
#define MC3B_SIN_KEY_LIMIT 0x41cdcd65

__device__ __forceinline__ double fast_sin(double a) {
    if (sin_arg_key(a) >= MC3B_SIN_KEY_LIMIT) return sin(a);   // |a| >= 1e9, inf, nan
    return fast_sin_core(a, MC3B_SIN_MAGIC);
}

template <typename T> struct mathx;
template <> struct mathx<double> {
    static __device__ __forceinline__ double sin_(double v) { return fast_sin(v); }
    static __device__ __forceinline__ double exp_(double v) { return exp(v); }
};
template <> struct mathx<float> {
    static __device__ __forceinline__ float sin_(float v) { return sinf(v); }
    static __device__ __forceinline__ float exp_(float v) { return expf(v); }
};

// y = sum_k p[k] x^k, NP coefficients (Horner).  get_started's quad() is NP=3.
// Model interface used by the kernels:
//   load(p)      once per chain per launch
//   eval(x)      per point, branch-free; may be invalid for extreme arguments,
//                in which case flagged() turns true
//   flagged()    eval() met an argument outside its valid range since clear()
//   eval_safe(x) always valid (slow path); clear() resets the flag
template <typename T, int NP> struct PolyModel {
    static constexpr bool GUARD = false;
    static constexpr bool TILE_STATE = false;
    __device__ __forceinline__ bool flagged() const { return false; }
    __device__ __forceinline__ void clear() {}
    __device__ __forceinline__ T eval_safe(T x) const { return eval(x); }
    T c[NP];
    __device__ __forceinline__ void load(const double* p) {
#pragma unroll
        for (int k = 0; k < NP; k++) c[k] = (T)p[k];
    }
    __device__ __forceinline__ T eval(T x) const {
        T y = c[NP - 1];
#pragma unroll
        for (int k = NP - 2; k >= 0; k--) y = fma(y, x, c[k]);
        return y;
    }
};

// y = p0 sin(2 pi x / p1 + p2) + p3 + p4 x        (BASELINE config 2)
template <typename T> struct SineModel {
    static constexpr bool GUARD = false;
    static constexpr bool TILE_STATE = false;
    __device__ __forceinline__ bool flagged() const { return false; }
    __device__ __forceinline__ void clear() {}
    T a, k, ph, c, s;
    __device__ __forceinline__ void load(const double* p) {
        a = (T)p[0]; k = (T)(6.283185307179586476925287 / p[1]); ph = (T)p[2];
        c = (T)p[3]; s = (T)p[4];
    }
    __device__ __forceinline__ T eval(T x) const {
        return fma(a, mathx<T>::sin_(fma(x, k, ph)), fma(s, x, c));
    }
    __device__ __forceinline__ T eval_safe(T x) const { return eval(x); }
};
// fp64: branch-free sine inside the point loop (so the unrolled points
// interleave); the largest |argument| seen is tracked with two integer ops and
// checked once per tile by the kernel, which then redoes the tile with eval_safe.
template <> struct SineModel<double> {
    static constexpr bool GUARD = true;
    static constexpr bool TILE_STATE = false;
    double a, k, ph, c, s, magic;
    int keymax;
#ifdef MC3B_SIN_REGCONST
    double K[11];
#define KS(i) K[i]
#else
#define KS(i) kSinC[i]
#endif
    __device__ __forceinline__ void load(const double* p) {
        a = p[0]; k = 6.283185307179586476925287 / p[1]; ph = p[2]; c = p[3]; s = p[4];
        magic = MC3B_SIN_MAGIC;
        asm volatile("" : "+d"(magic));          // keep it in a register
#ifdef MC3B_SIN_REGCONST
#pragma unroll
        for (int i = 0; i < 11; i++) { K[i] = kSinC[i]; asm volatile("" : "+d"(K[i])); }
#endif
        keymax = 0;
    }
    __device__ __forceinline__ double eval(double x) {
        const double arg = fma(x, k, ph);
        keymax = max(keymax, sin_arg_key(arg));
        return fma(a, fast_sin_core(arg, magic), fma(s, x, c));
    }
    template <int U> __device__ __forceinline__ void evalN(const double (&x)[U], double (&y)[U]) {
        double arg[U], t[U], q[U], r[U], s2[U], p[U];
#pragma unroll
        for (int u = 0; u < U; u++) arg[u] = fma(x[u], k, ph);
#pragma unroll
        for (int u = 0; u < U; u++) t[u] = fma(arg[u], KS(0), magic);
#pragma unroll
        for (int u = 0; u < U; u++) keymax = max(keymax, sin_arg_key(arg[u]));
#pragma unroll
        for (int u = 0; u < U; u++) q[u] = t[u] - magic;
#pragma unroll
        for (int u = 0; u < U; u++) r[u] = fma(q[u], KS(1), arg[u]);
#pragma unroll
        for (int u = 0; u < U; u++) r[u] = fma(q[u], KS(2), r[u]);
#pragma unroll
        for (int u = 0; u < U; u++) s2[u] = r[u] * r[u];
#pragma unroll
        for (int u = 0; u < U; u++) p[u] = fma(s2[u], KS(3), KS(4));
#pragma unroll
        for (int cidx = 5; cidx <= 10; cidx++) {
#pragma unroll
            for (int u = 0; u < U; u++) p[u] = fma(p[u], s2[u], KS(cidx));
        }
#pragma unroll
        for (int u = 0; u < U; u++) s2[u] = r[u] * s2[u];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const double v = fma(s2[u], p[u], r[u]);
            r[u] = __hiloint2double(__double2hiint(v) ^ (__double2loint(t[u]) << 31), __double2loint(v));
        }
#pragma unroll
        for (int u = 0; u < U; u++) y[u] = fma(a, r[u], fma(s, x[u], c));
    }
    __device__ __forceinline__ bool flagged() const { return keymax >= MC3B_SIN_KEY_LIMIT; }
    __device__ __forceinline__ void clear() { keymax = 0; }
    __device__ __forceinline__ double eval_safe(double x) const {
        return fma(a, sin(fma(x, k, ph)), fma(s, x, c));
    }
};

// Sinusoid on a uniform grid x_i = x_0 + i dx (fp64, one chain per lane walking
// the points of a tile in order, four at a time).  sin(k x_i + ph) is not
// evaluated per point: four interleaved sequences (points i = 0,1,2,3 mod 4)
// each advance by D = 4 k dx with Reinsch's form of the three-term recurrence,
//     du <- du - 4 sin^2(D/2) s ;  s <- s + du        (du = s_k - s_{k-1}),
// which keeps full accuracy for small D where 2 cos D would not.  The sequences
// carry A sin (amplitude folded in), so the model value is one ADDITION
// (A sin + line): a DFMA that reads three fresh vector registers occupies the
// FP64 pipe for 3 cycles instead of 2 (profiles/peakprobe.py variants 5/6;
// profiles/sass_rf_model.py reproduces the kernel time from the SASS), so the
// form with the fewest three-register FMAs wins, not only the fewest
// instructions.  Per point: 2 (sine) + 1 (line) + 1 (sum) + 2 (residual from the
// pre-scaled data tile, square) = 6 FP64 instructions instead of 20.
//
// Accuracy: every tile restarts the sequences (three one-step rotations from the
// tile's first point), so rounding accumulates over TILE/4 = 32 steps: an error e
// made m steps earlier shows as e sin((m+1)D)/sin D: <= 2e-15 A for k dx < 0.01,
// <= 8e-14 A up to 2.5 rad per sample (profiles/recurrence_error.py) unless D
// is within ~0.14 rad of pi (period ~ 8 samples, 1e-13); such chains, and model
// arguments beyond 1e9, are flagged and take the direct evaluation (GUARD).
// The tile's first point itself comes from fast_sincos_core every 8th tile and
// from one rotation by TILE k dx in between (error ~1e-16 per rotation).
struct SineGridModel {
    static constexpr bool GUARD = true;
    static constexpr bool TILE_STATE = true;
    static constexpr bool PREMUL = true;     // the kernel scales the data tile by 1/sigma once
    static constexpr int REANCHOR = 8;
    double a, k, ph, c0, sl, cd1, sd1, sD, hk, nkap, dth, cdT, sdT, S0, C0;
    double s[4], du[4];
    int keymax, keybase, tcount;
    __device__ __forceinline__ void load(const double* p, double dx, int tile) {
        a = p[0]; k = 6.283185307179586476925287 / p[1]; ph = p[2]; c0 = p[3]; sl = p[4];
        dth = k * dx;
        double sh, ch;
        fast_sincos_core(dth, sd1, cd1);
        fast_sincos_core(2.0 * dth, sh, ch);
        fast_sincos_core((double)tile * dth, sdT, cdT);
        sD = 2.0 * sh * ch;                  // sin D,  D = 4 dth
        hk = 2.0 * sh * sh;                  // 1 - cos D, no cancellation
        nkap = -2.0 * hk;                    // -4 sin^2(D/2)
        // |dth| beyond the fast range, or D too close to pi: always the direct path
        keybase = (sin_arg_key((double)tile * dth) >= MC3B_SIN_KEY_LIMIT || ch * ch < 0.005)
                      ? MC3B_SIN_KEY_LIMIT : 0;
        keymax = keybase;
        tcount = 0;
    }
    // x0: first point of the tile; npts: points of the tile (tiles of a CTA are contiguous)
    __device__ __forceinline__ void begin_tile(double x0, int npts) {
        const double th = fma(x0, k, ph);
        keymax = max(keymax, max(sin_arg_key(th), sin_arg_key(fma((double)npts, dth, th))));
        if (tcount == 0) {
            fast_sincos_core(th, S0, C0);
            S0 *= a; C0 *= a;
        } else {
            const double sn = fma(C0, sdT, S0 * cdT);
            C0 = fma(-S0, sdT, C0 * cdT);
            S0 = sn;
        }
        tcount = (tcount + 1 == REANCHOR) ? 0 : tcount + 1;
        double c[4];
        s[0] = S0; c[0] = C0;
#pragma unroll
        for (int u = 1; u < 4; u++) {
            s[u] = fma(c[u - 1], sd1, s[u - 1] * cd1);
            c[u] = fma(-s[u - 1], sd1, c[u - 1] * cd1);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) du[u] = fma(c[u], sD, s[u] * hk);   // A sin(th_u) - A sin(th_u - D)
    }
    template <int U> __device__ __forceinline__ void evalN(const double (&x)[U], double (&y)[U]) {
        static_assert(U == 4, "four interleaved sequences");
#pragma unroll
        for (int u = 0; u < U; u++) y[u] = fma(sl, x[u], c0) + s[u];
#pragma unroll
        for (int u = 0; u < U; u++) {
            du[u] = fma(nkap, s[u], du[u]);
            s[u] += du[u];
        }
    }
    __device__ __forceinline__ double eval(double x) const { return eval_safe(x); }
    __device__ __forceinline__ bool flagged() const { return keymax >= MC3B_SIN_KEY_LIMIT; }
    __device__ __forceinline__ void clear() { keymax = keybase; }
    __device__ __forceinline__ double eval_safe(double x) const {
        return fma(a, sin(fma(x, k, ph)), fma(sl, x, c0));
    }
};

// y = p0 exp(-0.5 ((x - p1)/p2)^2) + p3           (Gaussian line)
template <typename T> struct GaussModel {
    static constexpr bool GUARD = false;
    static constexpr bool TILE_STATE = false;
    __device__ __forceinline__ bool flagged() const { return false; }
    __device__ __forceinline__ void clear() {}
    __device__ __forceinline__ T eval_safe(T x) const { return eval(x); }
    T a, mu, is, c;
    __device__ __forceinline__ void load(const double* p) {
        a = (T)p[0]; mu = (T)p[1]; is = (T)(1.0 / p[2]); c = (T)p[3];
    }
    __device__ __forceinline__ T eval(T x) const {
        T d = (x - mu) * is;
        return fma(a, mathx<T>::exp_((T)(-0.5) * d * d), c);
    }
};

// y = p3 - p0 [ |x - p1| < p2/2 ]                 (transit-like box, config 3)
template <typename T> struct BoxModel {
    static constexpr bool GUARD = false;
    static constexpr bool TILE_STATE = false;
    __device__ __forceinline__ bool flagged() const { return false; }
    __device__ __forceinline__ void clear() {}
    __device__ __forceinline__ T eval_safe(T x) const { return eval(x); }
    T lo, base, t0, h;
    __device__ __forceinline__ void load(const double* p) {
        base = (T)p[3]; lo = (T)(p[3] - p[0]); t0 = (T)p[1]; h = (T)(0.5 * p[2]);
    }
    __device__ __forceinline__ T eval(T x) const { return (fabs(x - t0) < h) ? lo : base; }
};

template <class M, typename = void> struct premul_of { static constexpr bool value = false; };
template <class M> struct premul_of<M, decltype((void)M::PREMUL)> { static constexpr bool value = M::PREMUL; };
// Per-point inputs a model reads (M::NX; 1 unless the model says otherwise): a model of
// NX > 1 inputs has eval(const T (&v)[NX]) and eval_safe likewise.
template <class M, typename = void> struct ninputs_of { static constexpr int value = 1; };
template <class M> struct ninputs_of<M, decltype((void)M::NX)> { static constexpr int value = M::NX; };
// A model that declares M::NC (a user model of run-time constants, or of a prepare step) is
// loaded with load(p, k): its parameters, then the NC constants k[0..NC).  Others: load(p).
template <class M, typename = void> struct takes_consts { static constexpr bool value = false; };
template <class M> struct takes_consts<M, decltype((void)M::NC)> { static constexpr bool value = true; };

// y[u] = model(x[u]) for U points at once.  Models may provide their own evalN
// (stage-by-stage over the U points, so that in-order issue sees U independent
// dependency chains); the default just loops.
template <class M, typename T, int U>
__device__ __forceinline__ auto eval_points(M& m, const T (&x)[U], T (&y)[U], int) -> decltype(m.evalN(x, y), void()) {
    m.evalN(x, y);
}
template <class M, typename T, int U>
__device__ __forceinline__ void eval_points(M& m, const T (&x)[U], T (&y)[U], long) {
#pragma unroll
    for (int u = 0; u < U; u++) y[u] = m.eval(x[u]);
}
// ... and for a model of NX > 1 inputs: x[j][u] is input j of point u.
template <class M, typename T, int NX, int U>
__device__ __forceinline__ void eval_points(M& m, const T (&x)[NX][U], T (&y)[U]) {
#pragma unroll
    for (int u = 0; u < U; u++) {
        T v[NX];
#pragma unroll
        for (int j = 0; j < NX; j++) v[j] = x[j][u];
        y[u] = m.eval(v);
    }
}
// m.eval_safe at one point, v[j] = input j (the plain call for a model of one input).
template <class M, typename T, int NX>
__device__ __forceinline__ T eval_safe_at(const M& m, const T (&v)[NX]) {
    if constexpr (NX == 1) return m.eval_safe(v[0]);
    else return m.eval_safe(v);
}

// Dispatch a generic lambda-like functor F<Model> over (model_id, nmodel).
#define MC3B_DISPATCH_MODEL(T, model_id, nmodel, CALL)                                   \
    switch (model_id) {                                                                  \
    case MC3B_MODEL_POLYNOMIAL:                                                          \
        switch (nmodel) {                                                                \
        case 1: { using M = PolyModel<T, 1>; CALL; } break;                              \
        case 2: { using M = PolyModel<T, 2>; CALL; } break;                              \
        case 3: { using M = PolyModel<T, 3>; CALL; } break;                              \
        case 4: { using M = PolyModel<T, 4>; CALL; } break;                              \
        case 5: { using M = PolyModel<T, 5>; CALL; } break;                              \
        case 6: { using M = PolyModel<T, 6>; CALL; } break;                              \
        case 7: { using M = PolyModel<T, 7>; CALL; } break;                              \
        case 8: { using M = PolyModel<T, 8>; CALL; } break;                              \
        default: mc3b_set_error("polynomial needs 1..8 coefficients, got %d", nmodel);   \
                 return MC3B_ERR_ARG;                                                    \
        } break;                                                                         \
    case MC3B_MODEL_SINUSOID: { using M = SineModel<T>; CALL; } break;                   \
    case MC3B_MODEL_GAUSSIAN: { using M = GaussModel<T>; CALL; } break;                  \
    case MC3B_MODEL_BOX: { using M = BoxModel<T>; CALL; } break;                         \
    default: mc3b_set_error("unknown model id %d", model_id); return MC3B_ERR_ARG;       \
    }

static inline int mc3b_model_nparams(int model_id, int nmodel) {
    switch (model_id) {
    case MC3B_MODEL_POLYNOMIAL: return nmodel;
    case MC3B_MODEL_SINUSOID: return 5;
    case MC3B_MODEL_SINUSOID_GRID: return 5;
    case MC3B_MODEL_GAUSSIAN: return 4;
    case MC3B_MODEL_BOX: return 4;
    }
    return -1;
}
