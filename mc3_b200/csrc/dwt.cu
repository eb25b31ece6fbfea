// mc3_b200 -- wavelet likelihood (replaces src_c/_dwt.c + include/wavelet.h).
//
// dwt_chisq for a whole population: residual = data - model, Daubechies-4
// pyramid (periodic at every level, wavelet.h:16-51, 109-117), and only what
// _dwt.c:96-110 consumes: the sum of squared detail coefficients of every level
// and the last two smooth coefficients.  The n-point residual of a chain is
// never written to memory.  The kernels that read the model (k_dwt_reg_model,
// k_dwt_pass, k_dwt_last) are in dwt_kernel.cuh, shared with the user models of
// jit.cu; this file has the passes over given rows or coefficients (k_dwt_reg),
// the schedule, the launches and the standalone transform.
//
// For n = 2^20: reg(4 levels) -> 2^16, reg -> 2^12, pass(L=3) -> 512, last.  Bound:
// FP64 pipe (about 8 FMA-class instructions per input point over all levels + model).
#include <type_traits>
#include "dwt_kernel.cuh"

namespace {

// The register stage (dwt_kernel.cuh) over given model rows or over the coefficients of
// an earlier pass: every warp reads its own chain's row and transposes it.
template <int SRC, class M>
__global__ void __launch_bounds__(CH * 32) k_dwt_reg(RegArgs a) {
    __shared__ double tr[CH][RB + RB / 16];          // padded transpose rows (stride 17)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t c = (int64_t)blockIdx.x * CH + warp;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;
    M mdl;
    if (SRC == SRC_MODEL) mdl.load(a.params + c * a.ldp);
    const double* row = (SRC == SRC_MODEL) ? nullptr : a.rows + c * a.ldr;
    const double c0 = kC[0], c1 = kC[1], c2 = kC[2], c3 = kC[3];
    const int64_t mask = a.n_in - 1;
    double* T_ = tr[warp];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    const int64_t b_begin = (int64_t)blockIdx.y * a.blocks_per_span;
    int64_t b_end = b_begin + a.blocks_per_span;
    if (b_end > a.nblocks) b_end = a.nblocks;
    // One block.  INTERIOR: the 512 inputs do not wrap and every output the block
    // owns exists (no index masking, ownership is just lane < 30).
    auto do_block = [&](int64_t b, auto interior_tag) {
        constexpr bool INTERIOR = decltype(interior_tag)::value;
        const int64_t g0 = b * RADV;
        const double* px = (SRC == SRC_MODEL) ? a.x + g0 : nullptr;
        const double* pd = (SRC == SRC_ARRAY) ? nullptr : a.data + g0;
        const double* pr = (SRC == SRC_MODEL) ? nullptr : row + g0;
#pragma unroll 4
        for (int i = 0; i < 16; i++) {
            const int idx = i * 32 + lane;
            double r;
            if (INTERIOR) {
                if (SRC == SRC_MODEL) r = pd[idx] - mdl.eval_safe(px[idx]);
                else if (SRC == SRC_GIVEN) r = pd[idx] - pr[idx];
                else r = pr[idx];
            } else {
                const int64_t g = (g0 + idx) & mask;
                if (SRC == SRC_MODEL) r = a.data[g] - mdl.eval_safe(a.x[g]);
                else if (SRC == SRC_GIVEN) r = a.data[g] - row[g];
                else r = row[g];
            }
            T_[idx + (idx >> 4)] = r;
        }
        __syncwarp();
        double v[18];
#pragma unroll
        for (int k = 0; k < 16; k++) v[k] = T_[lane * 17 + k];
        __syncwarp();
        int cnt = 16;                                  // values this lane holds
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
                    if (INTERIOR) s2 = fma(d, d, s2);
                    else s2 = fma(d, (lev_pos0 + j < lev_n) ? d : 0.0, s2);
                    v[j] = sm;                         // j <= 2j: safe in-place
                }
            }
            // an output belongs to the block that holds its first input: lanes 0..29
            acc[l] += (lane < 30) ? s2 : 0.0;
            cnt = half;
        }
        const int64_t o = (g0 >> 4) + lane;
        if (live && lane < 30 && (INTERIOR || o < (a.n_in >> 4))) a.out[c * a.ldo + o] = v[0];
    };
    for (int64_t b = b_begin; b < b_end; b++) {
        if (b * RADV + RB <= a.n_in) do_block(b, std::true_type{});
        else do_block(b, std::false_type{});
    }
#pragma unroll
    for (int l = 0; l < 4; l++) {
        double t = acc[l];
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0 && live) a.sums[(c * MAXLEV + (a.lev0 + l)) * MAXSPAN + blockIdx.y] = t;
    }
}

// ---- standalone transform (one array) ---------------------------------------
__global__ void k_d4_fwd(const double* src, double* smooth, double* detail, int64_t nn) {
    const int64_t nh = nn >> 1;
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nh) return;
    const double a0 = src[2 * j], a1 = src[2 * j + 1], a2 = src[(2 * j + 2) & (nn - 1)],
                 a3 = src[(2 * j + 3) & (nn - 1)];
    smooth[j] = kC[0] * a0 + kC[1] * a1 + kC[2] * a2 + kC[3] * a3;
    detail[j] = kC[3] * a0 - kC[2] * a1 + kC[1] * a2 - kC[0] * a3;
}

// wavelet.h:38-44: out[2i+2], out[2i+3] from smooth s[i], s[i+1], detail d[i], d[i+1];
// out[0], out[1] from s[nh-1], d[nh-1], s[0], d[0].
__global__ void k_d4_inv(const double* s, const double* d, double* out, int64_t nn) {
    const int64_t nh = nn >> 1;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nh) return;
    const int64_t im = (i + nh - 1) & (nh - 1);       // i-1 with wrap
    const double sm = s[im], dm = d[im], s0 = s[i], d0 = d[i];
    out[2 * i] = kC[2] * sm + kC[1] * dm + kC[0] * s0 + kC[3] * d0;
    out[2 * i + 1] = kC[3] * sm - kC[0] * dm + kC[1] * s0 - kC[2] * d0;
}

int ilog2(int64_t n) { int k = 0; while ((1LL << k) < n) k++; return k; }

struct Schedule {
    int npass; int L[8]; int64_t nin[8]; int spans[8]; int tps[8]; int kind[8];   // kind 1 = register stage
    int64_t nblocks[8];
    int n0, lev0;
};

Schedule make_schedule(int64_t n) {
    Schedule s; s.npass = 0; s.lev0 = 0;
    int64_t cur = n;
    while (cur > LASTMAX) {
        if (cur >= 16 * LASTMAX) {                   // register stage: 4 levels, blocks of 512 advancing by 480
            const int64_t nb = ceil_div64(cur, RADV);
            const int spans = (int)(nb < MAXSPAN ? nb : MAXSPAN);
            s.kind[s.npass] = 1; s.L[s.npass] = 4; s.nin[s.npass] = cur; s.spans[s.npass] = spans;
            s.nblocks[s.npass] = nb; s.tps[s.npass] = (int)ceil_div64(nb, spans);
            s.npass++;
            s.lev0 += 4;
            cur >>= 4;
            continue;
        }
        int L = ilog2(cur / LASTMAX);
        if (L > LMAX) L = LMAX - 1;
        const int64_t tiles = cur / T;
        int spans = (int)(tiles < MAXSPAN ? tiles : MAXSPAN);
        s.kind[s.npass] = 0; s.nblocks[s.npass] = 0;
        s.L[s.npass] = L; s.nin[s.npass] = cur; s.spans[s.npass] = spans; s.tps[s.npass] = (int)(tiles / spans);
        s.npass++;
        s.lev0 += L;
        cur >>= L;
    }
    s.n0 = (int)cur;
    return s;
}

}  // namespace

extern "C" int64_t mc3b_dwt_workspace(int64_t nchains, int64_t n) {
    if (nchains <= 0 || n < 4) return 0;
    Schedule s = make_schedule(n);
    int64_t words = 1;
    if (s.npass > 0) {
        words += nchains * (n >> s.L[0]);                     // ping
        words += nchains * (s.npass > 1 ? (n >> (s.L[0] + s.L[1])) : 0);   // pong
        words += nchains * (int64_t)MAXLEV * MAXSPAN;         // span sums
    }
    return words * 8;
}

// u: a user model (SRC_MODEL, M unused), whose first pass runs on the kernels of its module;
// nullptr for the built-in M
template <int SRC, class M>
static int dwt_run(const Schedule& sc, int kbits, const double* params, int64_t ldp, int64_t nchains, int npars,
                   const double* x, const double* model, int64_t ldm, const double* data, int64_t n, double* ws,
                   double* chisq, cudaStream_t st, const DwtUserModel* u = nullptr) {
    const double* xs[MC3B_MAX_INPUTS] = {};
    for (int j = 0; u && j < u->nx; j++) xs[j] = u->xs[j];
    const double* uconst = u ? u->consts : nullptr;
    double* ping = ws;
    double* pong = ping + (sc.npass > 0 ? nchains * (n >> sc.L[0]) : 0);
    double* sums = pong + (sc.npass > 1 ? nchains * (n >> (sc.L[0] + sc.L[1])) : 0);
    LastArgsX la;
    for (int l = 0; l < MAXLEV; l++) la.spans_of_level[l] = 0;
    const unsigned groups = (unsigned)ceil_div64(nchains, CH);
    const double* cur_rows = model; int64_t cur_ld = ldm;
    int lev0 = 0;
    for (int p = 0; p < sc.npass; p++) {
        if (sc.kind[p] == 1) {
            RegArgsX r;
            r.params = params; r.ldp = ldp; r.nchains = nchains; r.x = x; r.data = data;
            r.rows = cur_rows; r.ldr = cur_ld; r.n_in = sc.nin[p]; r.lev0 = lev0;
            r.nblocks = sc.nblocks[p]; r.blocks_per_span = sc.tps[p];
            r.out = (p % 2 == 0) ? ping : pong; r.ldo = sc.nin[p] >> 4; r.sums = sums;
            for (int j = 0; j < MC3B_MAX_INPUTS; j++) r.xs[j] = xs[j];
            r.uconst = uconst;
            // spans actually needed with whole blocks per span
            const int spans = (int)ceil_div64(sc.nblocks[p], sc.tps[p]);
            dim3 grid(groups, (unsigned)spans);
            void* args[] = {&r};
            if (p == 0 && u) MC3B_CUDA(cudaLaunchKernel(u->reg, grid, dim3(CH * 32), args, 0, st));
            else if (p == 0 && SRC == SRC_MODEL) k_dwt_reg_model<M, RegArgs><<<grid, CH * 32, 0, st>>>(r);
            else if (p == 0) k_dwt_reg<SRC, M><<<grid, CH * 32, 0, st>>>(r);
            else k_dwt_reg<SRC_ARRAY, BoxModel<double>><<<grid, CH * 32, 0, st>>>(r);
            MC3B_CHECK_LAUNCH("k_dwt_reg");
            for (int l = 0; l < 4; l++) la.spans_of_level[lev0 + l] = spans;
            lev0 += 4;
            cur_rows = r.out; cur_ld = r.ldo;
            continue;
        }
        PassArgsX a;
        a.params = params; a.ldp = ldp; a.nchains = nchains; a.x = x; a.data = data;
        a.rows = cur_rows; a.ldr = cur_ld; a.n_in = sc.nin[p]; a.L = sc.L[p]; a.lev0 = lev0;
        a.spans = sc.spans[p]; a.tiles_per_span = sc.tps[p];
        a.out = (p % 2 == 0) ? ping : pong; a.ldo = sc.nin[p] >> sc.L[p]; a.sums = sums;
        for (int j = 0; j < MC3B_MAX_INPUTS; j++) a.xs[j] = xs[j];
        a.uconst = uconst;
        dim3 grid(groups, (unsigned)sc.spans[p]);
        const size_t sm = pass_smem(1);
        void* args[] = {&a};
        if (p == 0 && u) {
            MC3B_CUDA(cudaLaunchKernel(u->pass, grid, dim3(CH * 32), args, pass_smem(u->nx), st));
        } else if (p == 0) {
            MC3B_CUDA(cudaFuncSetAttribute(k_dwt_pass<SRC, M, PassArgs>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            k_dwt_pass<SRC, M, PassArgs><<<grid, CH * 32, sm, st>>>(a);
        } else {
            MC3B_CUDA(cudaFuncSetAttribute(k_dwt_pass<SRC_ARRAY, M, PassArgs>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)sm));
            k_dwt_pass<SRC_ARRAY, M, PassArgs><<<grid, CH * 32, sm, st>>>(a);
        }
        MC3B_CHECK_LAUNCH("k_dwt_pass");
        for (int l = 0; l < sc.L[p]; l++) la.spans_of_level[lev0 + l] = sc.spans[p];
        lev0 += sc.L[p];
        cur_rows = a.out; cur_ld = a.ldo;
    }
    la.params = params; la.ldp = ldp; la.npars = npars; la.nchains = nchains; la.x = x; la.data = data;
    la.rows = cur_rows; la.ldr = cur_ld; la.n0 = sc.n0; la.lev0 = lev0; la.kbits = kbits; la.sums = sums;
    la.chisq = chisq;
    for (int j = 0; j < MC3B_MAX_INPUTS; j++) la.xs[j] = xs[j];
    la.uconst = uconst;
    const unsigned lgroups = (unsigned)ceil_div64(nchains, CHL);
    void* args[] = {&la};
    if (sc.npass == 0 && u) MC3B_CUDA(cudaLaunchKernel(u->last, dim3(lgroups), dim3(CHL * 32), args, 0, st));
    else if (sc.npass == 0) k_dwt_last<SRC, M, LastArgs><<<lgroups, CHL * 32, 0, st>>>(la);
    else k_dwt_last<SRC_ARRAY, M, LastArgs><<<lgroups, CHL * 32, 0, st>>>(la);
    MC3B_CHECK_LAUNCH("k_dwt_last");
    return MC3B_OK;
}

// the checks every wavelet chi-squared runs: kbits = log2 n
static int dwt_check(const double* params, int64_t ldp, int64_t nchains, int npars, const double* data, int64_t n,
                     void* workspace, double* chisq, int* kbits) {
    MC3B_CHECK_ARG(params && data && chisq && workspace && nchains > 0, "bad arguments");
    MC3B_CHECK_ARG(n >= 4 && (n & (n - 1)) == 0, "dwt_chisq needs n = 2^k >= 4 (got %lld)", (long long)n);
    MC3B_CHECK_ARG(npars >= 3 && npars <= ldp, "wavelet chisq needs at least three parameters");
    *kbits = ilog2(n);
    MC3B_CHECK_ARG(*kbits < MAXLEV, "n too large");
    return MC3B_OK;
}

extern "C" int mc3b_dwt_chisq(int model_id, const double* params, int64_t ldp, int64_t nchains, int npars, int nmodel,
                              const double* x, const double* model, int64_t ldm, const double* data, int64_t n,
                              void* workspace, double* chisq, void* stream) {
    int kbits = 0;
    if (int rc = dwt_check(params, ldp, nchains, npars, data, n, workspace, chisq, &kbits)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    Schedule sc = make_schedule(n);
    double* ws = (double*)workspace;
    if (model_id < 0) {
        MC3B_CHECK_ARG(model != nullptr && ldm >= n, "model rows missing");
        using M = BoxModel<double>;   // unused by SRC_GIVEN / SRC_ARRAY
        return dwt_run<SRC_GIVEN, M>(sc, kbits, params, ldp, nchains, npars, x, model, ldm, data, n, ws, chisq, st);
    }
    MC3B_CHECK_ARG(x != nullptr, "built-in model needs x");
    if (model_id == MC3B_MODEL_SINUSOID_GRID) model_id = MC3B_MODEL_SINUSOID;
    MC3B_CHECK_ARG(mc3b_model_nparams(model_id, nmodel) == nmodel && nmodel <= npars - 3,
                   "model %d does not take %d parameters", model_id, nmodel);
    MC3B_DISPATCH_MODEL(double, model_id, nmodel,
                        return (dwt_run<SRC_MODEL, M>(sc, kbits, params, ldp, nchains, npars, x, model, ldm, data, n,
                                                      ws, chisq, st)));
    return MC3B_OK;
}

int mc3b_dwt_chisq_user(const DwtUserModel& u, const double* params, int64_t ldp, int64_t nchains, int npars,
                        const double* data, int64_t n, void* workspace, double* chisq, cudaStream_t st) {
    int kbits = 0;
    if (int rc = dwt_check(params, ldp, nchains, npars, data, n, workspace, chisq, &kbits)) return rc;
    MC3B_CHECK_ARG(u.nmodel <= npars - 3, "the model takes %d parameters, more than npars - 3 = %d", u.nmodel,
                   npars - 3);
    for (int j = 0; j < u.nx; j++) MC3B_CHECK_ARG(u.xs[j] != nullptr, "null pointer (input %d)", j);
    // M is unused: pass 0 (or the last pass) runs on u's kernels, later passes on SRC_ARRAY
    return dwt_run<SRC_MODEL, BoxModel<double>>(make_schedule(n), kbits, params, ldp, nchains, npars, u.xs[0],
                                                 nullptr, 0, data, n, (double*)workspace, chisq, st, &u);
}

extern "C" int mc3b_daub4(const double* in, int64_t n2, int isign, void* workspace, double* out, void* stream) {
    MC3B_CHECK_ARG(in && out && workspace, "null pointer");
    MC3B_CHECK_ARG(n2 >= 4 && (n2 & (n2 - 1)) == 0, "daub4 needs n = 2^k >= 4");
    MC3B_CHECK_ARG(in != out, "daub4: in and out must not alias");
    cudaStream_t st = (cudaStream_t)stream;
    double* t0 = (double*)workspace;            // two scratch halves of n2/2
    double* t1 = t0 + n2 / 2;
    if (isign >= 0) {
        // level nn: smooth -> scratch, detail -> its final slot out[nn/2 .. nn)
        const double* src = in;
        double* dst = t0;
        for (int64_t nn = n2; nn >= 4; nn >>= 1) {
            const int64_t nh = nn >> 1;
            double* sm = (nn == 4) ? out : dst;
            k_d4_fwd<<<(unsigned)ceil_div64(nh, 256), 256, 0, st>>>(src, sm, out + nh, nn);
            MC3B_CHECK_LAUNCH("k_d4_fwd");
            src = dst;
            dst = (dst == t0) ? t1 : t0;
        }
    } else {
        // level nn: smooth from the previous level (or in[0..2)), detail from in[nn/2 .. nn)
        const double* s = in;
        double* dst = t0;
        for (int64_t nn = 4; nn <= n2; nn <<= 1) {
            const int64_t nh = nn >> 1;
            double* o = (nn == n2) ? out : dst;
            k_d4_inv<<<(unsigned)ceil_div64(nh, 256), 256, 0, st>>>(s, in + nh, o, nn);
            MC3B_CHECK_LAUNCH("k_d4_inv");
            s = o;
            dst = (dst == t0) ? t1 : t0;
        }
    }
    return MC3B_OK;
}
