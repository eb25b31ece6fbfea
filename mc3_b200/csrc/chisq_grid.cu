// mc3_b200 -- the headline kernel: sinusoid + line on a uniform abscissa grid with
// one uncertainty for all points (BASELINE config 2), fused with chi-squared and,
// optionally, the Metropolis step.  Bound: FP64 pipe.
#include "chisq_args.cuh"

namespace {

// ---- sinusoid + line on a uniform abscissa grid ------------------------------
// With x_i = x_0 + i dx the abscissa is never streamed, and with one uncertainty
// for all points (USIG, BASELINE config 2: sigma = 0.5) neither are the weights:
//   chisq = sigma^-2 sum_i (A sin(k x_i + ph) + c0 + sl x_i - d_i)^2.
// Only the data tile is staged (TMA bulk copy, NSTAGE deep, full/empty mbarriers:
// no CTA-wide barrier in the tile loop).  Six FP64 instructions per chain-point,
//   t  = Lb + s                      block base of the line + A sin
//   y  = fma(dL4, j, t)              exact line of step j (j an immediate): the line
//                                    is never a running sum, so offsets of 1e5 sigma
//                                    keep 1e-10 on chi-squared
//   r  = y - d ;  q = fma(r, r, q)
//   du = fma(nkap, s, du) ; s = s + du      Reinsch recurrence (models.cuh SineGridModel)
// each reading at most two fresh vector registers.  What bounds the loop is the
// register file, not the FP64 pipe's issue rate: one 64-bit operand per cycle and
// scheduler (profiles/r2_fp64_probe.md: DADD/DFMA with two fresh registers 2.04
// cycles, three fresh 3.03, a shared multiplier 2.2, + 1.2 per LDS.128; DMMA.8x8x4
// runs on the same pipe at 16 cycles, so the tensor form of the line gains nothing).
// Four interleaved sequences (points 0..3 mod 4) per chain, one chain per lane.
// Sequences restart every RESTART tiles from the first point of the interval, which
// comes from fast_sincos_core every REANCHOR-th restart and one rotation in
// between.  Accuracy as SineGridModel; the same guard sends stiff or huge-argument
// chains to the direct evaluation.
// Per-point uncertainties (!USIG): the stage also holds 1/sigma; every warp scales
// the data tile into a private buffer once (d/sigma, warp-synchronous) and the
// residual is fma(y, 1/sigma, -d/sigma).
namespace grid {
constexpr int TILE = 128;           // points per TMA stage and per schedule unit
#ifndef MC3B_GRID_NSTAGE
#define MC3B_GRID_NSTAGE 4
#endif
constexpr int NSTAGE = MC3B_GRID_NSTAGE;
#ifndef MC3B_GRID_RESTART
#define MC3B_GRID_RESTART 4
#endif
constexpr int RESTART = MC3B_GRID_RESTART;   // tiles between restarts of the sequences
constexpr int REANCHOR = 4;         // restarts between direct sincos evaluations of the anchor
}

// 4 CTAs per SM: 120 registers hold the sequences and the per-chain constants without
// spilling (6 CTAs at 80 registers measured 0.1829 ms, 4 at 120: 0.1778 ms at config 2)
#ifndef MC3B_GRID_MINB
#define MC3B_GRID_MINB 4
#endif
template <bool USIG>
__global__ void __launch_bounds__(WARPS * 32, MC3B_GRID_MINB) k_sinegrid(ChisqArgs<double> a) {
    using namespace grid;
    asm volatile("griddepcontrol.launch_dependents;");   // the next proposal kernel may start its draws
    __shared__ __align__(128) double sd[NSTAGE][TILE];
    __shared__ __align__(128) double sw[USIG ? 1 : NSTAGE][USIG ? 2 : TILE];
    __shared__ __align__(128) double pw[USIG ? 1 : WARPS][USIG ? 2 : TILE];      // per-warp d/sigma
    __shared__ __align__(8) uint64_t full[NSTAGE], empty[NSTAGE];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t c = ((int64_t)blockIdx.x * WARPS + warp) * 32 + lane;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;                   // idle lanes shadow the last chain

    // piecewise-uniform abscissa (tile origins a.xt, include/mc3b200.h tile_x): every tile is
    // anchored on its own origin; the plan may hold a few tiles that do not exist
    const bool seg = a.xt != nullptr;
    const double x0 = a.x[0];
    const double dx = seg ? a.dxg : (a.x[a.n - 1] - x0) / (double)(a.n - 1);
    const double* p = a.params + c * a.ldp;
    const double amp = p[0], k = 6.283185307179586476925287 / p[1], ph = p[2], c0 = p[3], sl = p[4];
    const double dth = k * dx;
    double cd1, sd1, cdT, sdT, sh, ch;
    fast_sincos_core(dth, sd1, cd1);
    fast_sincos_core(2.0 * dth, sh, ch);
    fast_sincos_core((double)(RESTART * TILE) * dth, sdT, cdT);
    const double sD = 2.0 * sh * ch;                // sin D, D = 4 dth
    const double hk = 2.0 * sh * sh;                // 1 - cos D
    double nkap = -2.0 * hk;                        // -4 sin^2(D/2)
    double dL4 = 4.0 * sl * dx;
    asm volatile("" : "+d"(dL4), "+d"(nkap));       // loop constants stay registers (no re-multiplication)
    // direct evaluation for this chain: |RESTART T dth| beyond the fast range, or D within ~0.14 rad of pi
    const int keybase = (sin_arg_key((double)(RESTART * TILE) * dth) >= MC3B_SIN_KEY_LIMIT || ch * ch < 0.005)
                            ? MC3B_SIN_KEY_LIMIT : 0;
    auto direct = [&](double x) { return fma(amp, sin(fma(x, k, ph)), fma(sl, x, c0)); };

    const int64_t nfull = seg ? a.ntiles : a.n / TILE;
    int64_t tb, te;
    if (a.nsched > 0) { tb = a.tstart[blockIdx.y]; te = a.tstart[blockIdx.y + 1]; }
    else { tb = (a.n / TILE) * blockIdx.y / gridDim.y; te = (a.n / TILE) * (blockIdx.y + 1) / gridDim.y; }
    if (tb > nfull) tb = nfull;
    if (te > nfull) te = nfull;
    const int64_t nt = te - tb;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    auto issue = [&](int64_t t, int s) {
        mbar_expect_tx(&full[s], (USIG ? 1u : 2u) * TILE * sizeof(double));
        bulk_g2s(sd[s], a.d + t * TILE, TILE * sizeof(double), &full[s]);
        if constexpr (!USIG) bulk_g2s(sw[s], a.w + t * TILE, TILE * sizeof(double), &full[s]);
    };
    if (threadIdx.x == 0)
        for (int s = 0; s < NSTAGE && s < nt; s++) issue(tb + s, s);

    double acc = 0.0, S0 = 0.0, C0 = 0.0;
    double s[4], du[4], Lu[4], q[4];
    int rcount = 0, key = 0;
    for (int64_t it = 0; it < nt; it++) {
        const int st = (int)(it % NSTAGE);
        const uint32_t par = (uint32_t)((it / NSTAGE) & 1);
        const int tr = seg ? 0 : (int)(it % RESTART);   // tile within the restart interval
        const double xt = seg ? a.xt[tb + it] : fma((double)((tb + it) * TILE), dx, x0);
        if (tr == 0) {
            // ---- restart: anchors of the four sequences (no data needed yet) ----
            const double th = fma(xt, k, ph);
            key = max(keybase, max(sin_arg_key(th), sin_arg_key(fma((double)(RESTART * TILE), dth, th))));
            if (rcount == 0 || seg) {
                fast_sincos_core(th, S0, C0);
                S0 *= amp; C0 *= amp;
            } else {
                const double sn = fma(C0, sdT, S0 * cdT);
                C0 = fma(-S0, sdT, C0 * cdT);
                S0 = sn;
            }
            rcount = (rcount + 1 == REANCHOR) ? 0 : rcount + 1;
            double cc[4];
            s[0] = S0; cc[0] = C0;
#pragma unroll
            for (int u = 1; u < 4; u++) {
                s[u] = fma(cc[u - 1], sd1, s[u - 1] * cd1);
                cc[u] = fma(-s[u - 1], sd1, cc[u - 1] * cd1);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                du[u] = fma(cc[u], sD, s[u] * hk);       // A sin(th_u) - A sin(th_u - D)
                Lu[u] = fma(sl, fma((double)u, dx, xt), c0);   // line at the first point of each sequence
            }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) q[u] = 0.0;
        mbar_wait(&full[st], par);
        const double* dt = sd[st];                  // what the residual subtracts
        const double* wt = sw[USIG ? 0 : st];
        if constexpr (!USIG) {
            __syncwarp();                           // the warp is done with its previous tile
#pragma unroll
            for (int i = lane; i < TILE; i += 32) pw[warp][i] = sd[st][i] * sw[st][i];
            __syncwarp();
            dt = pw[warp];
        }
        if (key < MC3B_SIN_KEY_LIMIT) {
            // 32 steps of 4 points per tile, in blocks of 8 steps: the line of step m is
            // Lu + m dL4 with ONE rounding (block base by FMA, step offset an immediate),
            // never a running sum -- offsets of 1e5 sigma keep 1e-10 on chi-squared
            double mb = (double)(tr * (TILE / 4));
#pragma unroll 1
            for (int o = 0; o < TILE; o += 32) {
                double Lb[4];
#pragma unroll
                for (int u = 0; u < 4; u++) Lb[u] = fma(dL4, mb, Lu[u]);
                mb += 8.0;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int i = o + 4 * j;
                    const double2 d01 = *reinterpret_cast<const double2*>(&dt[i]);
                    const double2 d23 = *reinterpret_cast<const double2*>(&dt[i + 2]);
                    const double d[4] = {d01.x, d01.y, d23.x, d23.y};
                    double r[4];
                    if constexpr (USIG) {
#pragma unroll
                        for (int u = 0; u < 4; u++)
                            r[u] = (j == 0 ? Lb[u] + s[u] : fma(dL4, (double)j, Lb[u] + s[u])) - d[u];
                    } else {
                        const double2 w01 = *reinterpret_cast<const double2*>(&wt[i]);
                        const double2 w23 = *reinterpret_cast<const double2*>(&wt[i + 2]);
                        const double w[4] = {w01.x, w01.y, w23.x, w23.y};
#pragma unroll
                        for (int u = 0; u < 4; u++)
                            r[u] = fma(j == 0 ? Lb[u] + s[u] : fma(dL4, (double)j, Lb[u] + s[u]), w[u], -d[u]);
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) q[u] = fma(r[u], r[u], q[u]);
#pragma unroll
                    for (int u = 0; u < 4; u++) du[u] = fma(nkap, s[u], du[u]);
#pragma unroll
                    for (int u = 0; u < 4; u++) s[u] += du[u];
                }
            }
        } else {                                    // guarded chains: library sine per point
            double qd = 0.0;
            for (int i = 0; i < TILE; i++) {
                const double r = USIG ? direct(fma((double)i, dx, xt)) - sd[st][i]
                                      : (direct(fma((double)i, dx, xt)) - sd[st][i]) * sw[USIG ? 0 : st][USIG ? 0 : i];
                qd = fma(r, r, qd);
            }
            q[0] = qd;
        }
        acc += (q[0] + q[1]) + (q[2] + q[3]);
        // ---- stage hand-back: this warp is done with tile `it`; the producer refills
        // the stage of the PREVIOUS tile (every warp has long left it) -------------
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);
        if (threadIdx.x == 0 && it >= 1 && it - 1 + NSTAGE < nt) {
            const int sp = (int)((it - 1) % NSTAGE);
            mbar_wait(&empty[sp], (uint32_t)(((it - 1) / NSTAGE) & 1));
            issue(tb + it - 1 + NSTAGE, sp);
        }
    }

    if (seg) {                                      // points that fill no tile: shared out over the splits
        const int64_t nl = a.n - nfull * TILE;
        const int64_t lb = nfull * TILE + nl * blockIdx.y / gridDim.y, le = nfull * TILE + nl * (blockIdx.y + 1) / gridDim.y;
        double t = 0.0;
        for (int64_t i = lb; i < le; i++) {
            const double r = USIG ? direct(a.x[i]) - a.d[i] : (direct(a.x[i]) - a.d[i]) * a.w[i];
            t = fma(r, r, t);
        }
        acc += t;
    } else if (blockIdx.y == gridDim.y - 1) {       // ragged tail, straight from global memory
        double t = 0.0;
        for (int64_t i = nfull * TILE; i < a.n; i++) {
            const double r = USIG ? direct(a.x[i]) - a.d[i] : (direct(a.x[i]) - a.d[i]) * a.w[i];
            t = fma(r, r, t);
        }
        acc += t;
    }
    const double w0 = USIG ? a.w[0] : 1.0;
    if (live) a.partial[(int64_t)blockIdx.y * a.ldpartial + c] = USIG ? acc * (w0 * w0) : acc;
#ifndef MC3B_NO_FUSE_CODE
    if (a.f.on) fused_metropolis(a.f, a.partial, a.ldpartial, a.nchains, WARPS * 32);
#endif
}

// ---- the same model on point PAIRS mirrored about block centres ----------------
// One uncertainty for all points.  In a block of 16 points with centre phase th_c
// (between points 7 and 8) the pair p = 0..7 sits at offsets -+dl, dl = p + 1/2:
//   A sin(th_c +- dl h) = Sc cos(dl h) +- Cc sin(dl h)      (Sc, Cc = A sin/cos th_c)
//   line(x_c +- dl dx)  = L_c +- sl dx dl
// so with e = (d+ + d-)/2 and o = (d+ - d-)/2, both chain-independent and prepared
// ONCE per data set by mc3b_fold_data (stored negated),
//   u = Sc cp[p] + (L_c - e)          = (r+ + r-)/2
//   v = Cc sp[p] + (sl dx dl - o)     = (r+ - r-)/2
//   r+^2 + r-^2 = 2 (u^2 + v^2).
// Six FP64 instructions per PAIR (t = L_c + ne; u = fma; q = fma(u,u,q); t' = fma(gs,
// dl, no), dl an immediate; v = fma; q = fma(v,v,q)) plus five per block (rotation of
// (Sc, Cc) by 16 h, block line): 3.3 per chain-point instead of 6, every one of them
// with at most two fresh register operands, and the same rounding-error class as the
// per-point evaluation (no subtraction of large sums: profiles/fold_error.py).  The
// tables cp/sp[p] = cos/sin((p + 1/2) h) live in 32 registers per chain.  Anchors as in
// k_sinegrid: (Sc, Cc) restart every RESTART tiles from a rotation of the previous
// anchor, every REANCHOR-th from fast_sincos_core; 32 block rotations in between.
// Rotations are stable for any step, so only huge arguments take the direct path.
// Per-chain constants of the kernel: every CTA of a chain group (105 data splits at
// config 2) would derive the same numbers through a division and four dependent
// sine/cosine evaluations before it can touch its first tile (ncu, round 2: a third of
// all warp time).  k_fold_consts derives them once per chain and launch; the CTAs
// then start with one round of coalesced loads.  Same formulas, same bits.
namespace fold {
constexpr int BLK = 16, NP = BLK / 2;
constexpr int NCONST = 2 * NP + 11;     // k, cp[NP], sp[NP], c16, s16, cdT, sdT, Kcc, Kc2, Kss, Ksd2, c128, s128
static_assert(NCONST == MC3B_FOLD_WORK, "include/mc3b200.h: MC3B_FOLD_WORK");
struct Consts { double k, cp[NP], sp[NP], c16, s16, cdT, sdT; };
__device__ __forceinline__ void derive(double period, double dx, Consts& K) {
    using namespace grid;
    K.k = 6.283185307179586476925287 / period;
    const double dth = K.k * dx;
    double s1, c1;
    fast_sincos_core(0.5 * dth, K.sp[0], K.cp[0]);
    fast_sincos_core(dth, s1, c1);
#pragma unroll
    for (int i = 1; i < NP; i++) {
        K.cp[i] = fma(-K.sp[i - 1], s1, K.cp[i - 1] * c1);
        K.sp[i] = fma(K.cp[i - 1], s1, K.sp[i - 1] * c1);
    }
    fast_sincos_core((double)BLK * dth, K.s16, K.c16);
    fast_sincos_core((double)(RESTART * TILE) * dth, K.sdT, K.cdT);
}
}  // namespace fold

__global__ void __launch_bounds__(128) k_fold_consts(const double* __restrict__ params, int64_t ldp, int64_t nchains,
                                                     const double* __restrict__ x, int64_t n, double dxg,
                                                     double* __restrict__ out, int64_t ld) {
    asm volatile("griddepcontrol.launch_dependents;");
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    using fold::NP;
    const double dx = dxg != 0.0 ? dxg : (x[n - 1] - x[0]) / (double)(n - 1);
    fold::Consts K;
    fold::derive(params[c * ldp + 1], dx, K);
    double* o = out + c;
    o[0] = K.k;
    double kcc = 0.0, kc = 0.0, kss = 0.0, ksd = 0.0;       // sums over the pair offsets (k_sinefold<MOM>)
#pragma unroll
    for (int i = 0; i < NP; i++) {
        o[(1 + i) * ld] = K.cp[i]; o[(1 + NP + i) * ld] = K.sp[i];
        kcc = fma(K.cp[i], K.cp[i], kcc); kc += K.cp[i];
        kss = fma(K.sp[i], K.sp[i], kss); ksd = fma(K.sp[i], (double)i + 0.5, ksd);
    }
    o[(1 + 2 * NP) * ld] = K.c16; o[(2 + 2 * NP) * ld] = K.s16;
    o[(3 + 2 * NP) * ld] = K.cdT; o[(4 + 2 * NP) * ld] = K.sdT;
    o[(5 + 2 * NP) * ld] = kcc; o[(6 + 2 * NP) * ld] = 2.0 * kc;
    o[(7 + 2 * NP) * ld] = kss; o[(8 + 2 * NP) * ld] = 2.0 * ksd;
    double s128, c128;                                      // one tile on (k_sinemma)
    fast_sincos_core((double)grid::TILE * (K.k * dx), s128, c128);
    o[(9 + 2 * NP) * ld] = c128; o[(10 + 2 * NP) * ld] = s128;
}

// ---- MOM: the same sum from sufficient statistics -------------------------------------
// Expanding the squares of u and v over a block's eight pairs,
//   sum_p u_p^2 + v_p^2 = Sc (Sc Kcc + 2 Lc Kc - 2 Pe) + Cc (Cc Kss + 2 g Ksd - 2 Po)
//                         + [8 Lc^2 + 170 g^2 - 2 Lc E1 - 2 g O1 + E2 + O2]
//   Pe = sum_p cp_p e_p,  Po = sum_p sp_p o_p,  Kcc = sum cp^2, Kc = sum cp, Kss = sum sp^2, Ksd = sum sp dl
// only Pe and Po touch the data: ONE FMA per point; the bracket needs the data only
// through three moments per 128-point tile (prepared once by mc3b_moment_prepare,
// like the pairs themselves, which it stores centred on a reference line and scaled by
// -2).  28 FP64 instructions per 16-point block: 1.75 per chain-point.
// The price: chi-squared is what is left after sums of size (|s| + |L'| + |d'|)^2 cancel,
// so its relative error is eps_eff amp, amp = (|s|max + |L'| + |d'|)^2 / (sigma^2 chisq),
// eps_eff < 3e-15 (profiles/moment_error.py, against long double).  The Metropolis
// epilogue therefore checks amp <= amp_max for every chain (MomentFix below) and
// re-evaluates the chains that fail it point by point, so that every chi-squared that
// leaves the kernel is within the 1e-10 contract; the host watches the count and
// returns to k_sinefold<MOM=false> when it is not rare (high signal-to-noise data).
struct MomentFix {
    const ChisqArgs<double>& a;
    // `act`: this thread owns a chain whose proposal is inside the bounds; nxt = its data chi-squared.
    // Returns the CTA's count of chains sent to the point-by-point evaluation.
    __device__ __forceinline__ int operator()(bool act, int64_t cl, double& nxt) const {
        const double* p = a.params + cl * a.ldp;
        double pa = 0.0, pc = 0.0, ps = 0.0;
        if (act) { pa = p[0]; pc = p[3]; ps = p[4]; }
        return guard(act, p, pa, pc, ps, a.w[0], nxt);
    }
    // the same with the chain's amplitude, intercept and slope (p[0], p[3], p[4]; read when act)
    // and the weight w0 in registers
    __device__ __forceinline__ int guard(bool act, const double* p, double pa, double pc, double ps, double w0,
                                         double& nxt) const {
        const MomentArgs& m = a.m;
        bool bad = false;
        if (act) {
            // |L'| <= sqrt(n) max(|L'(xlo)|, |L'(xhi)|): a line is extremal at the ends of its range
            const double n = (double)a.n;
            const double c0 = pc - m.c0ref, sl = ps - m.slref;
            const double lmax = fmax(fabs(fma(sl, m.xlo, c0)), fabs(fma(sl, m.xhi, c0)));
            const double mag = (fabs(pa) + lmax) * sqrt(n) + sqrt(m.d2tot);
            bad = !(mag * mag * (w0 * w0) <= m.amp_max * nxt);        // NaN: exact path too
        }
        const int hits = __syncthreads_count(bad);
        if (!hits) return 0;
        // rare: the flagged chains one at a time, in thread order, the whole CTA over the data
        __shared__ double prm[5], red[WARPS];
        __shared__ uint32_t mask[WARPS];
        const uint32_t bal = __ballot_sync(0xffffffffu, bad);
        if ((threadIdx.x & 31) == 0) mask[threadIdx.x >> 5] = bal;
        __syncthreads();
        for (int w = 0; w < WARPS; w++) {
            uint32_t mk = mask[w];
            while (mk) {
                const int t = w * 32 + __ffs(mk) - 1;
                mk &= mk - 1;
                if ((int)threadIdx.x == t)
                    for (int j = 0; j < 5; j++) prm[j] = p[j];
                __syncthreads();
                const double amp = prm[0], k = 6.283185307179586476925287 / prm[1], ph = prm[2], c0 = prm[3], sl = prm[4];
                double q = 0.0;
                for (int64_t i = threadIdx.x; i < a.n; i += WARPS * 32) {
                    const double x = a.x[i];
                    const double r = fma(amp, sin(fma(x, k, ph)), fma(sl, x, c0)) - a.d[i];
                    q = fma(r, r, q);
                }
                for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
                if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
                __syncthreads();
                if ((int)threadIdx.x == t) {
                    double tot = 0.0;
                    for (int j = 0; j < WARPS; j++) tot += red[j];
                    nxt = tot * (w0 * w0);
                }
                __syncthreads();
            }
        }
        return hits;
    }
    __device__ __forceinline__ int32_t* counter() const { return a.m.guard_hits; }
    // Guard record of the fused epilogue (include/mc3b200.h mc3b_moment_t.record): the host reads
    // the count of generation g without a copy on the stream.  hits: guard_hits once every hit of
    // the launch is in (fused_metropolis_end); one aligned 64-bit store, stamp in the high word.
    __device__ __forceinline__ bool recording() const { return a.m.record != nullptr; }
    __device__ __forceinline__ void record(int64_t g, int hits) const {
        const unsigned long long v = ((unsigned long long)(uint32_t)g << 32) | (uint32_t)hits;
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(a.m.record + (g & (MC3B_GUARD_RECORDS - 1))), "l"(v)
                     : "memory");
    }
};

#ifndef MC3B_FOLD_MINB
#define MC3B_FOLD_MINB 4
#endif
#ifndef MC3B_MOM_ACC
#define MC3B_MOM_ACC 1
#endif
template <bool PRE, bool MOM>
__global__ void __launch_bounds__(WARPS * 32, MC3B_FOLD_MINB) k_sinefold(ChisqArgs<double> a) {
    using namespace grid;
    using fold::BLK; using fold::NP;
    static_assert(PRE || !MOM, "the moment form takes its constants from k_fold_consts");
    asm volatile("griddepcontrol.launch_dependents;");
    __shared__ __align__(128) double sf[NSTAGE][TILE];
    __shared__ __align__(32) double sm[MOM ? NSTAGE : 1][4];        // tile moments
    __shared__ __align__(8) uint64_t full[NSTAGE], empty[NSTAGE];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t c = ((int64_t)blockIdx.x * WARPS + warp) * 32 + lane;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;

    // piecewise-uniform abscissa: the plan was made for n / TILE tiles, a few of which may not exist
    const bool seg = a.xt != nullptr;
    const int64_t nfull = seg ? a.ntiles : a.n / TILE;
    int64_t tb, te;
    if (a.nsched > 0) { tb = a.tstart[blockIdx.y]; te = a.tstart[blockIdx.y + 1]; }
    else { tb = (a.n / TILE) * blockIdx.y / gridDim.y; te = (a.n / TILE) * (blockIdx.y + 1) / gridDim.y; }
    if (tb > nfull) tb = nfull;
    if (te > nfull) te = nfull;
    const int64_t nt = te - tb;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    const double* folded = MOM ? a.m.folded : a.fold;
    auto issue = [&](int64_t t, int s) {
        mbar_expect_tx(&full[s], (TILE + (MOM ? 4 : 0)) * sizeof(double));
        bulk_g2s(sf[s], folded + t * TILE, TILE * sizeof(double), &full[s]);
        if constexpr (MOM) bulk_g2s(sm[s], a.m.tiles + t * 4, 4 * sizeof(double), &full[s]);
    };
    if (threadIdx.x == 0)
        for (int s = 0; s < NSTAGE && s < nt; s++) issue(tb + s, s);

    const double x0 = a.x[0];
    const double dx = seg ? a.dxg : (a.x[a.n - 1] - x0) / (double)(a.n - 1);
    const double* p = a.params + c * a.ldp;
    const double amp = p[0], ph = p[2], c0 = p[3], sl = p[4];
    // MOM: the line relative to the reference line the data were centred on
    const double c0r = MOM ? c0 - a.m.c0ref : c0, slr = MOM ? sl - a.m.slref : sl;
    fold::Consts K;
    double Kcc = 0.0, Kc2 = 0.0, Kss = 0.0, gK = 0.0;
    if constexpr (PRE) {
        if (a.consts_wait) asm volatile("griddepcontrol.wait;" ::: "memory");   // k_fold_consts has completed
        const double* kc = a.consts + c;
        K.k = kc[0];
#pragma unroll
        for (int i = 0; i < NP; i++) { K.cp[i] = kc[(1 + i) * a.ldc]; K.sp[i] = kc[(1 + NP + i) * a.ldc]; }
        K.c16 = kc[(1 + 2 * NP) * a.ldc]; K.s16 = kc[(2 + 2 * NP) * a.ldc];
        K.cdT = kc[(3 + 2 * NP) * a.ldc]; K.sdT = kc[(4 + 2 * NP) * a.ldc];
        if constexpr (MOM) {
            Kcc = kc[(5 + 2 * NP) * a.ldc]; Kc2 = kc[(6 + 2 * NP) * a.ldc];
            Kss = kc[(7 + 2 * NP) * a.ldc]; gK = kc[(8 + 2 * NP) * a.ldc];
        }
    } else {
        fold::derive(p[1], dx, K);
    }
    const double k = K.k, c16 = K.c16, s16 = K.s16, cdT = K.cdT, sdT = K.sdT;
    const double (&cp)[NP] = K.cp;
    const double (&sp)[NP] = K.sp;
    const double dth = k * dx;
    double gs = slr * dx;
    double dL16 = (double)BLK * gs;
    asm volatile("" : "+d"(gs), "+d"(dL16));
    gK *= gs;                                       // 2 g Ksd
    const int keybase = sin_arg_key((double)(RESTART * TILE) * dth) >= MC3B_SIN_KEY_LIMIT ? MC3B_SIN_KEY_LIMIT : 0;
    auto direct = [&](double x) { return fma(amp, sin(fma(x, k, ph)), fma(sl, x, c0)); };

    double acc = 0.0, S0 = 0.0, C0 = 0.0, Sc = 0.0, Cc = 0.0;
    int rcount = 0, key = 0;
    for (int64_t it = 0; it < nt; it++) {
        const int st = (int)(it % NSTAGE);
        const uint32_t par = (uint32_t)((it / NSTAGE) & 1);
        const int tr = (int)(it % RESTART);
        // centre of the tile's first block: x0 + (first point + 7.5) dx, one rounding; on a
        // piecewise-uniform abscissa every tile has its own origin and its own anchor
        const double xc = seg ? fma(7.5, dx, a.xt[tb + it]) : fma((double)((tb + it) * TILE) + 7.5, dx, x0);
        if (tr == 0 || seg) {
            const double th = fma(xc, k, ph);
            key = max(keybase, max(sin_arg_key(th), sin_arg_key(fma((double)(RESTART * TILE), dth, th))));
            if (rcount == 0 || seg) {
                fast_sincos_core(th, S0, C0);
                S0 *= amp; C0 *= amp;
            } else {
                const double sn = fma(C0, sdT, S0 * cdT);
                C0 = fma(-S0, sdT, C0 * cdT);
                S0 = sn;
            }
            rcount = (rcount + 1 == REANCHOR) ? 0 : rcount + 1;
            Sc = S0; Cc = C0;
        }
        const double Lt = fma(slr, xc, c0r);        // line at the centre of the first block
        double q[4] = {0.0, 0.0, 0.0, 0.0};
        mbar_wait(&full[st], par);
        if (key < MC3B_SIN_KEY_LIMIT) {
            const double* ft = sf[st];
#pragma unroll
            for (int b = 0; b < TILE / BLK; b++) {
                const double Lc = b == 0 ? Lt : fma(dL16, (double)b, Lt);
                if constexpr (!MOM) {
#pragma unroll
                    for (int pp = 0; pp < NP; pp++) {
                        const double2 f2 = *reinterpret_cast<const double2*>(&ft[b * BLK + 2 * pp]);
                        const double u = fma(Sc, cp[pp], Lc + f2.x);
                        const double v = fma(Cc, sp[pp], fma(gs, (double)pp + 0.5, f2.y));
                        q[(2 * pp) & 3] = fma(u, u, q[(2 * pp) & 3]);
                        q[(2 * pp + 1) & 3] = fma(v, v, q[(2 * pp + 1) & 3]);
                    }
                } else {
                    constexpr int NA = MC3B_MOM_ACC;                        // partial sums per block (ILP)
                    double pe[NA], po[NA];
#pragma unroll
                    for (int i = 0; i < NA; i++) { pe[i] = 0.0; po[i] = 0.0; }
                    pe[0] = Lc * Kc2; po[0] = gK;                           // 2 Lc Kc - 2 Pe ; 2 g Ksd - 2 Po
#pragma unroll
                    for (int pp = 0; pp < NP; pp++) {
                        const double2 f2 = *reinterpret_cast<const double2*>(&ft[b * BLK + 2 * pp]);
                        pe[pp % NA] = fma(cp[pp], f2.x, pe[pp % NA]);
                        po[pp % NA] = fma(sp[pp], f2.y, po[pp % NA]);
                    }
#pragma unroll
                    for (int i = NA / 2; i > 0; i >>= 1)
#pragma unroll
                        for (int j = 0; j < i; j++) { pe[j] += pe[j + i]; po[j] += po[j + i]; }
                    q[0] = fma(Sc, fma(Sc, Kcc, pe[0]), q[0]);
                    q[1] = fma(Cc, fma(Cc, Kss, po[0]), q[1]);
                }
                const double sn = fma(Cc, s16, Sc * c16);
                Cc = fma(-Sc, s16, Cc * c16);
                Sc = sn;
            }
            if constexpr (MOM) {
                // line and data terms of the whole tile from its three moments:
                //   64 Lm^2 + 87376 g^2 - 2 Lm M0 - 2 g M1 + M2,  Lm = line at the tile centre
                const double4 mo = *reinterpret_cast<const double4*>(sm[st]);
                const double Lm = fma(gs, 56.0, Lt);
                q[2] = fma(Lm, fma(Lm, 64.0, mo.x), mo.z);
                q[3] = gs * fma(gs, 87376.0, mo.y);
            }
        } else {                                    // guarded chains: library sine per point, raw data
            double qd = 0.0;
            const double xt = seg ? a.xt[tb + it] : fma((double)((tb + it) * TILE), dx, x0);
            const double* dt = a.d + (tb + it) * TILE;
            for (int i = 0; i < TILE; i++) {
                const double r = direct(fma((double)i, dx, xt)) - dt[i];
                qd = fma(r, r, qd);
            }
            q[0] = 0.5 * qd;
        }
        acc += (q[0] + q[1]) + (q[2] + q[3]);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);
        if (threadIdx.x == 0 && it >= 1 && it - 1 + NSTAGE < nt) {
            const int sq = (int)((it - 1) % NSTAGE);
            mbar_wait(&empty[sq], (uint32_t)(((it - 1) / NSTAGE) & 1));
            issue(tb + it - 1 + NSTAGE, sq);
        }
    }

    acc *= 2.0;
    if (seg) {                                      // points that fill no tile: shared out over the splits
        const int64_t nl = a.n - nfull * TILE;
        const int64_t lb = nfull * TILE + nl * blockIdx.y / gridDim.y, le = nfull * TILE + nl * (blockIdx.y + 1) / gridDim.y;
        double t = 0.0;
        for (int64_t i = lb; i < le; i++) {
            const double r = direct(a.x[i]) - a.d[i];
            t = fma(r, r, t);
        }
        acc += t;
    } else if (blockIdx.y == gridDim.y - 1) {       // ragged tail, straight from global memory
        double t = 0.0;
        for (int64_t i = nfull * TILE; i < a.n; i++) {
            const double r = direct(a.x[i]) - a.d[i];
            t = fma(r, r, t);
        }
        acc += t;
    }
    const double w0 = a.w[0];
    if (live) a.partial[(int64_t)blockIdx.y * a.ldpartial + c] = acc * (w0 * w0);
#ifndef MC3B_NO_FUSE_CODE
    if (a.f.on) {
        if constexpr (MOM) fused_metropolis(a.f, a.partial, a.ldpartial, a.nchains, WARPS * 32, MomentFix{a});
        else fused_metropolis(a.f, a.partial, a.ldpartial, a.nchains, WARPS * 32);
    }
#endif
}

// ---- k_sinemma: the moment form with Pe, Po as FP64 tensor-core products ----------------
// Pe[chain, block] = sum_p cos(dl_p h_chain) e[p, block] is an [8 chains x 8 pairs] x [8 pairs x
// 8 blocks] product per 128-point tile: two mma.m8n8k4 (k = pairs 0-3, 4-7), two more for
// Po.  DMMA runs on the FP64 FMA units at the same flop rate (profiles/r2_fp64_probe.md), but
// an m8n8k4 reads four operand registers for 256 FMAs where 128 DFMAs read 384, needs 4
// instructions instead of 128, and its B fragments are four conflict-free LDS.64 per lane
// and tile instead of 64 LDS.128 -- the DFMA form is bound by exactly those (operand reads,
// issue slots, shared-memory latency), not by the pipe.
// Mapping: a warp owns 8 chains (lane l: chain l >> 2) and, per tile, lane l ends up with Pe, Po
// of blocks 2 (l & 3) and 2 (l & 3) + 1 of its chain: the per-block work (rotation of (Sc, Cc),
// block line, the four FMAs that fold Pe, Po into the sum) is spread over the chain's four
// lanes, and each lane keeps ONE chain's constants.  The CTA covers its 128 chains in four
// passes of 32 over the split's tiles (the TMA ring just keeps turning: the tile sequence
// repeats), so the launch shape, the partial rows and the Metropolis epilogue are those of
// k_sinefold.
#ifndef MC3B_MMA_MINB
#define MC3B_MMA_MINB 4
#endif
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(WARPS * 32, MC3B_MMA_MINB) k_sinemma(ChisqArgs<double> a) {
    using namespace grid;
    using fold::BLK; using fold::NP;
    static_assert(WARPS == 4 && TILE == 128 && NP == 8, "four warps x 8 chains x 4 passes = 128 chains; one n8 tile");
    // One iteration = up to NT4 consecutive tiles (one TMA stage): the per-iteration work
    // (barrier waits, addresses, anchors) is paid once per 4 x 128 points x 8 chains per warp.
    constexpr int NT4 = 4;
    static_assert(NT4 == RESTART, "an iteration is one restart interval of the anchors");
    asm volatile("griddepcontrol.launch_dependents;");
    __shared__ __align__(128) double sf[NSTAGE][NT4 * TILE];
    __shared__ __align__(32) double sm[NSTAGE][NT4 * 4];
    __shared__ __align__(8) uint64_t full[NSTAGE], empty[NSTAGE];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q4 = lane & 3;
    const bool seg = a.xt != nullptr;
    const int64_t nfull = seg ? a.ntiles : a.n / TILE;
    int64_t tb, te;
    if (a.nsched > 0) { tb = a.tstart[blockIdx.y]; te = a.tstart[blockIdx.y + 1]; }
    else { tb = (a.n / TILE) * blockIdx.y / gridDim.y; te = (a.n / TILE) * (blockIdx.y + 1) / gridDim.y; }
    if (tb > nfull) tb = nfull;
    if (te > nfull) te = nfull;
    const int64_t nt = te - tb;
    const int64_t npi = (nt + NT4 - 1) / NT4, nit = 4 * npi;      // iterations per pass; four passes over the same tiles

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    auto issue = [&](int64_t it, int s) {
        const int64_t t = tb + (it % npi) * NT4;
        const int64_t cnt = te - t < NT4 ? te - t : NT4;
        mbar_expect_tx(&full[s], (uint32_t)(cnt * (TILE + 4) * sizeof(double)));
        bulk_g2s(sf[s], a.m.folded + t * TILE, (uint32_t)(cnt * TILE * sizeof(double)), &full[s]);
        bulk_g2s(sm[s], a.m.tiles + t * 4, (uint32_t)(cnt * 4 * sizeof(double)), &full[s]);
    };
    if (threadIdx.x == 0)
        for (int s = 0; s < NSTAGE && s < nit; s++) issue(s, s);

    const double x0 = a.x[0];
    const double dx = seg ? a.dxg : (a.x[a.n - 1] - x0) / (double)(a.n - 1);
    const double w0 = a.w[0];
    if (a.consts_wait) asm volatile("griddepcontrol.wait;" ::: "memory");       // k_fold_consts has completed

    int64_t it = 0;
    for (int pass = 0; pass < 4; pass++) {
        int64_t c = (int64_t)blockIdx.x * (WARPS * 32) + pass * 32 + warp * 8 + g;
        const bool live = c < a.nchains;
        if (!live) c = a.nchains - 1;
        const double* p = a.params + c * a.ldp;
        const double amp = p[0], ph = p[2], c0 = p[3], sl = p[4];
        const double c0r = c0 - a.m.c0ref, slr = sl - a.m.slref;
        const double* kc = a.consts + c;
        const double k = kc[0];
        const double cpa0 = kc[(1 + q4) * a.ldc], cpa1 = kc[(5 + q4) * a.ldc];                 // A fragments
        const double spa0 = kc[(1 + NP + q4) * a.ldc], spa1 = kc[(5 + NP + q4) * a.ldc];
        const double c16 = kc[(1 + 2 * NP) * a.ldc], s16 = kc[(2 + 2 * NP) * a.ldc];
        const double cdT = kc[(3 + 2 * NP) * a.ldc], sdT = kc[(4 + 2 * NP) * a.ldc];
        const double Kcc = kc[(5 + 2 * NP) * a.ldc], Kc2 = kc[(6 + 2 * NP) * a.ldc];
        const double Kss = kc[(7 + 2 * NP) * a.ldc];
        const double c128 = kc[(9 + 2 * NP) * a.ldc], s128 = kc[(10 + 2 * NP) * a.ldc];
        const double dth = k * dx;
        const double gs = slr * dx, dL16 = (double)BLK * gs, dL128 = (double)TILE * gs;
        const double gK = kc[(8 + 2 * NP) * a.ldc] * gs;                                        // 2 g Ksd
        const int keybase = sin_arg_key((double)(NT4 * TILE) * dth) >= MC3B_SIN_KEY_LIMIT ? MC3B_SIN_KEY_LIMIT : 0;
        auto direct = [&](double x) { return fma(amp, sin(fma(x, k, ph)), fma(sl, x, c0)); };
        const double boff = (double)(2 * q4 * BLK) + 7.5;       // centre of this lane's first block of a tile, in points

        double acc = 0.0, S0 = 0.0, C0 = 0.0;
        int rcount = 0;
        for (int64_t ji = 0; ji < npi; ji++, it++) {
            const int st = (int)(it % NSTAGE);
            const uint32_t par = (uint32_t)((it / NSTAGE) & 1);
            const int64_t t0 = tb + ji * NT4;
            const int cnt = (int)(te - t0 < NT4 ? te - t0 : NT4);
            // anchor of the iteration: this lane's first block of its first tile
            const double xo = seg ? a.xt[t0] : fma((double)(t0 * TILE), dx, x0);
            const double xc = fma(boff, dx, xo);
            const double th = fma(xc, k, ph);
            int key = max(keybase, max(sin_arg_key(th), sin_arg_key(fma((double)(NT4 * TILE), dth, th))));
            if (rcount == 0 || seg) {
                fast_sincos_core(th, S0, C0);
                S0 *= amp; C0 *= amp;
            } else {
                const double sn = fma(C0, sdT, S0 * cdT);
                C0 = fma(-S0, sdT, C0 * cdT);
                S0 = sn;
            }
            rcount = (rcount + 1 == REANCHOR) ? 0 : rcount + 1;
            double Sc = S0, Cc = C0;
            const double L00 = fma(slr, xc, c0r);       // line at the centre of that block
            double q = 0.0;
            mbar_wait(&full[st], par);
#pragma unroll
            for (int u = 0; u < NT4; u++) {
                if (u < cnt) {                          // (uniform over the CTA: the MMAs stay warp-wide)
                    double L0 = u == 0 ? L00 : fma(dL128, (double)u, L00);
                    if (u > 0) {
                        if (seg) {                      // tiles of a piecewise-uniform abscissa have their own origins
                            const double xcu = fma(boff, dx, a.xt[t0 + u]);
                            const double thu = fma(xcu, k, ph);
                            key = max(key, sin_arg_key(thu));
                            fast_sincos_core(thu, Sc, Cc);
                            Sc *= amp; Cc *= amp;
                            L0 = fma(slr, xcu, c0r);
                        } else {                        // one tile on
                            const double sn = fma(Cc, s128, Sc * c128);
                            Cc = fma(-Sc, s128, Cc * c128);
                            Sc = sn;
                        }
                    }
                    const double L1 = L0 + dL16;
                    const double* ft = sf[st] + u * TILE;
                    double pe0 = L0 * Kc2, pe1 = L1 * Kc2, po0 = gK, po1 = gK;     // 2 Lc Kc - 2 Pe ; 2 g Ksd - 2 Po
                    dmma884(pe0, pe1, cpa0, ft[lane]);
                    dmma884(po0, po1, spa0, ft[64 + lane]);
                    dmma884(pe0, pe1, cpa1, ft[32 + lane]);
                    dmma884(po0, po1, spa1, ft[96 + lane]);
                    const double S1 = fma(Cc, s16, Sc * c16), C1 = fma(-Sc, s16, Cc * c16);   // the second block
                    q = fma(Sc, fma(Sc, Kcc, pe0), q);
                    q = fma(Cc, fma(Cc, Kss, po0), q);
                    q = fma(S1, fma(S1, Kcc, pe1), q);
                    q = fma(C1, fma(C1, Kss, po1), q);
                    if (u == q4) {
                        // line and data terms of tile u from its three moments (one of the chain's lanes each):
                        //   64 Lm^2 + 87376 g^2 - 2 Lm M0 - 2 g M1 + M2,  Lm = line at the tile centre
                        const double4 mo = *reinterpret_cast<const double4*>(sm[st] + 4 * u);
                        const double Lm = fma(gs, 63.5 - boff, L0);
                        q += fma(Lm, fma(Lm, 64.0, mo.x), mo.z) + gs * fma(gs, 87376.0, mo.y);
                    }
                }
            }
            if (key >= MC3B_SIN_KEY_LIMIT) {            // guarded chains: library sine per point, raw data
                double qd = 0.0;
                for (int u = 0; u < cnt; u++) {
                    const double xou = seg ? a.xt[t0 + u] : fma((double)((t0 + u) * TILE), dx, x0);
                    const double* dt = a.d + (t0 + u) * TILE;
                    for (int i = q4; i < TILE; i += 4) {
                        const double r = direct(fma((double)i, dx, xou)) - dt[i];
                        qd = fma(r, r, qd);
                    }
                }
                q = 0.5 * qd;
            }
            acc += q;
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[st]);
            if (threadIdx.x == 0 && it >= 1 && it - 1 + NSTAGE < nit) {
                const int sq = (int)((it - 1) % NSTAGE);
                mbar_wait(&empty[sq], (uint32_t)(((it - 1) / NSTAGE) & 1));
                issue(it - 1 + NSTAGE, sq);
            }
        }
        acc *= 2.0;
        // points outside the tiles (ragged tail: last split; piecewise-uniform: shared out over the
        // splits), every fourth point to each of the chain's lanes
        {
            int64_t lb = nfull * TILE, le = a.n;
            if (seg) {
                const int64_t nl = a.n - nfull * TILE;
                lb = nfull * TILE + nl * blockIdx.y / gridDim.y; le = nfull * TILE + nl * (blockIdx.y + 1) / gridDim.y;
            } else if (blockIdx.y != gridDim.y - 1) le = lb;
            double t = 0.0;
            for (int64_t i = lb + q4; i < le; i += 4) {
                const double r = direct(a.x[i]) - a.d[i];
                t = fma(r, r, t);
            }
            acc += t;
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (live && q4 == 0) a.partial[(int64_t)blockIdx.y * a.ldpartial + c] = acc * (w0 * w0);
    }
#ifndef MC3B_NO_FUSE_CODE
    if (a.f.on) fused_metropolis(a.f, a.partial, a.ldpartial, a.nchains, WARPS * 32, MomentFix{a});
#endif
}

// mc3b_moment_finish: what the fused epilogue does for a launch WITHOUT the Metropolis step --
// rows of k_sinefold<MOM> added in split order, the guard, the point-by-point
// re-evaluation of the chains that fail it, then the prior terms (as k_chisq_finish).
__global__ void __launch_bounds__(WARPS * 32) k_moment_finish(ChisqArgs<double> a, int nsplit, int npars,
                                                              const double* __restrict__ prior,
                                                              const double* __restrict__ plo,
                                                              const double* __restrict__ pup, double* __restrict__ chisq) {
    const int64_t c = (int64_t)blockIdx.x * (WARPS * 32) + threadIdx.x;
    const bool mine = c < a.nchains;
    double acc = 0.0;
    if (mine)
        for (int s = 0; s < nsplit; s++) acc += a.partial[(int64_t)s * a.ldpartial + c];
    const int hits = MomentFix{a}(mine, c, acc);
    if (threadIdx.x == 0 && hits && a.m.guard_hits) atomicAdd(a.m.guard_hits, hits);
    if (!mine) return;
    if (prior != nullptr) {
        double pr = 0.0;
        for (int j = 0; j < npars; j++) {
            const double lo = plo[j], up = pup[j];
            if (lo > 0.0 && up > 0.0) {
                const double off = a.params[c * a.ldp + j] - prior[j];
                const double t = off / (off > 0.0 ? up : lo);
                pr += t * t;
            }
        }
        acc += pr;
    }
    chisq[c] = acc;
}

// out[16 b + 2 p] = -(d[16 b + 8 + p] + d[16 b + 7 - p])/2, out[16 b + 2 p + 1] = -(d[hi] - d[lo])/2
__global__ void k_fold(const double* __restrict__ d, int64_t nblk16, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nblk16 * 16) return;
    const int64_t b = i >> 4;
    const int j = (int)(i & 15), pp = j >> 1;
    const double lo = d[b * 16 + 7 - pp], hi = d[b * 16 + 8 + pp];
    out[i] = (j & 1) ? -0.5 * (hi - lo) : -0.5 * (hi + lo);
}

// mc3b_moment_prepare: one warp per 128-point tile; lane l holds pairs 2 (l & 3), +1 of
// block l >> 2.  d' = d - (c0ref + slref x_i); folded[.] = -2 e, -2 o (e, o = half sum and
// half difference of a pair); tiles[t] = {-2 sum e, -2 (16 sum_b (b - 3.5) E1_b + sum dl o),
// sum e^2 + o^2, 0}.  Fixed-order shuffles: same bits on every run.
// layout 1 (k_sinemma): the tile as the four B fragments of mma.m8n8k4 -- entry
// eo*64 + ks*32 + 4 b + q holds pair p = 4 ks + q of block b (eo = 0: -2 e, 1: -2 o), so
// that lane l = 4 b + q of a warp reads its element of fragment (eo, ks) at offset l.
__global__ void __launch_bounds__(128) k_moment_prepare(const double* __restrict__ d, int64_t ntiles, double x0, double dx,
                                                        const double* __restrict__ tile_x, double c0ref, double slref,
                                                        double* __restrict__ folded, double* __restrict__ tiles, int layout) {
    const int64_t t = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (t >= ntiles) return;
    const int lane = threadIdx.x & 31, b = lane >> 2;
    const double xo = tile_x ? tile_x[t] : fma((double)(t * 128), dx, x0);      // abscissa of the tile's first point
    double m0 = 0.0, m1 = 0.0, m2 = 0.0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int pp = 2 * (lane & 3) + h;
        const int64_t ilo = t * 128 + b * 16 + 7 - pp, ihi = t * 128 + b * 16 + 8 + pp;
        const double lo = d[ilo] - fma(slref, fma((double)(b * 16 + 7 - pp), dx, xo), c0ref);
        const double hi = d[ihi] - fma(slref, fma((double)(b * 16 + 8 + pp), dx, xo), c0ref);
        const double e = 0.5 * (hi + lo), o = 0.5 * (hi - lo);
        if (layout == 0) {
            folded[t * 128 + b * 16 + 2 * pp] = -2.0 * e;
            folded[t * 128 + b * 16 + 2 * pp + 1] = -2.0 * o;
        } else {
            folded[t * 128 + (pp >> 2) * 32 + b * 4 + (pp & 3)] = -2.0 * e;
            folded[t * 128 + 64 + (pp >> 2) * 32 + b * 4 + (pp & 3)] = -2.0 * o;
        }
        m0 += e;
        m1 += fma(16.0 * ((double)b - 3.5), e, ((double)pp + 0.5) * o);
        m2 += fma(e, e, o * o);
    }
    for (int s = 16; s > 0; s >>= 1) {
        m0 += __shfl_xor_sync(0xffffffffu, m0, s);
        m1 += __shfl_xor_sync(0xffffffffu, m1, s);
        m2 += __shfl_xor_sync(0xffffffffu, m2, s);
    }
    if (lane == 0) {
        double4 o4 = make_double4(-2.0 * m0, -2.0 * m1, m2, 0.0);
        *reinterpret_cast<double4*>(tiles + t * 4) = o4;
    }
}

// ---- spectral form: the whole chi-squared from a precomputed spectrum of the data ----------
// With t = x - xc, d' = d - (c0ref + slref x), the line relative to the reference line written
// about the centre, L' = a + b t, and S_g(w) = sum_n g_n e^{i w x_n},
//   sigma^2 chisq = A^2 [n/2 - Re(e^{2 i ph} S_1(2w))/2] + 2 A Im(e^{i ph} [a S_1(w) + b S_t(w) - S_d'(w)])
//                 + n a^2 + 2 a b St + b^2 St2 - 2 a Sd - 2 b Std + D2
// (St = sum t, St2 = sum t^2, Sd = sum d', Std = sum t d', D2 = sum d'^2, all measured).  The data
// enter only through S at the chain's own frequency; per node w_j of a grid Delta apart the table
// holds T_g[j][k] = sum_n g_n t_n^k e^{i w_j x_n} / k!, and
//   S_g(w_j + delta) = e^{i delta xc} sum_k (i delta)^k T_g[j][k]          (complex Horner)
// with truncation error <= (|delta| R)^{K+1} / (K+1)! sum |g|, R = max |t|.  S_t needs no table of
// its own: T_t[j][k] = (k + 1) T_1[j][k + 1], so the band's nodes hold T_1 to order K + 1.
// Layout (doubles): spec::HEAD sums {n, St, St2, Sd, Std, D2, 0, 0}; per node of the band,
// K + 2 complex T_1 then K + 1 complex T_d'; per node of the doubled band, K + 1 complex T_1.
namespace spec {
constexpr int HEAD = MC3B_SPECTRAL_HEAD;
}

// One CTA per node (the band's, then the doubled band's) plus one for the sums; every thread
// adds the points i = tid mod 256 in order, then lanes (xor tree) and warps (in order): the
// bits depend on neither the SM count nor the device.
template <int K>
__global__ void __launch_bounds__(256) k_spectral_table(const double* __restrict__ x, const double* __restrict__ d,
                                                        int64_t n, double c0ref, double slref, double xc, double w1,
                                                        double w2, double delta, int n1, int n2,
                                                        double* __restrict__ out) {
    constexpr int NV = 4 * K + 6;
    __shared__ double red[8][NV];
    const int j = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool band1 = j < n1, sums = j == n1 + n2;
    const double om = band1 ? fma((double)j, delta, w1) : fma((double)(j - n1), delta, w2);
    double v[NV];                   // re T_1[0..K+1], im T_1[0..K+1], re T_d'[0..K], im T_d'[0..K]
#pragma unroll
    for (int k = 0; k < NV; k++) v[k] = 0.0;
    if (sums) {
        for (int64_t i = threadIdx.x; i < n; i += 256) {
            const double xv = x[i], t = xv - xc, dp = d[i] - fma(slref, xv, c0ref);
            v[1] += t; v[2] = fma(t, t, v[2]); v[3] += dp; v[4] = fma(t, dp, v[4]); v[5] = fma(dp, dp, v[5]);
        }
    } else {
        for (int64_t i = threadIdx.x; i < n; i += 256) {
            const double xv = x[i], t = xv - xc;
            double pr, pi;
            sincos(om * xv, &pi, &pr);
            const double dp = band1 ? d[i] - fma(slref, xv, c0ref) : 0.0;
#pragma unroll
            for (int k = 0; k < K + 2; k++) {
                v[k] += pr; v[K + 2 + k] += pi;
                if (band1 && k <= K) { v[2 * K + 4 + k] = fma(dp, pr, v[2 * K + 4 + k]); v[3 * K + 5 + k] = fma(dp, pi, v[3 * K + 5 + k]); }
                pr *= t; pi *= t;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NV; k++) {
        double s = v[k];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) red[warp][k] = s;
    }
    __syncthreads();
    const int k = threadIdx.x;
    if (k >= NV) return;
    double s = 0.0;
    for (int w = 0; w < 8; w++) s += red[w][k];
    if (sums) {
        if (k < spec::HEAD) out[k] = k == 0 ? (double)n : (k < 6 ? s : 0.0);
        return;
    }
    const int kk = k < 2 * K + 4 ? k % (K + 2) : (k - 2 * K - 4) % (K + 1);
    const int im = k < 2 * K + 4 ? k / (K + 2) : (k - 2 * K - 4) / (K + 1);
    double fact = 1.0;
    for (int i = 2; i <= kk; i++) fact *= (double)i;
    double* tab = out + spec::HEAD;
    if (band1) {
        const int64_t e = (int64_t)j * (2 * K + 3) + (k < 2 * K + 4 ? kk : K + 2 + kk);
        tab[2 * e + im] = s / fact;
    } else if (k < 2 * K + 4 && kk <= K) {
        const int64_t e = (int64_t)n1 * (2 * K + 3) + (int64_t)(j - n1) * (K + 1) + kk;
        tab[2 * e + im] = s / fact;
    }
}

// One thread per chain, no data stream: three complex Horner sums of K + 1 terms and three
// sincos, whatever n is.  The row is that of a one-split launch of the tile kernels, and as
// unguarded: a chain whose frequency (or twice it) falls outside the table gets NaN, which
// MomentFix (fused epilogue or mc3b_moment_finish) sends to the point-by-point evaluation
// together with the chains whose amplification is too large.
// What is constant during a run (the table's sums, the weight) is requested at entry, before the
// chain's parameters arrive, together with an L2 prefetch of one 128-byte line of the table per
// launched thread (the whole table at config 2's 4096 chains; only its first lines for small
// populations).  The Horner sums are unrolled and the table loads written ahead of the first FMA.
// Launched with WARPS * 32 threads.  The register cap (without it ptxas settles on 72 registers
// and spills) holds the whole table row of a chain at K = 9 (31 complex values, 124 registers);
// at K = 15 the row (49 complex values) does not fit and ptxas issues it in more than one batch.
template <int K>
__global__ void __maxnreg__(168) k_spectral_chisq(ChisqArgs<double> a) {
    asm volatile("griddepcontrol.launch_dependents;");   // the next proposal kernel may start its draws
    const MomentArgs& m = a.m;
    const double* h = m.spec;                       // n, St, St2, Sd, Std, D2
    const double h0 = h[0], h1 = h[1], h2 = h[2], h3 = h[3], h4 = h[4], h5 = h[5];
    const double w0 = a.w[0];
    {
        const int64_t bytes = 8 * (spec::HEAD + 2 * ((int64_t)m.sn1 * (2 * K + 3) + (int64_t)m.sn2 * (K + 1)));
        const int64_t at = ((int64_t)blockIdx.x * (WARPS * 32) + threadIdx.x) * 128;
        if (at < bytes) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(m.spec) + at));
    }
    int64_t c = (int64_t)blockIdx.x * (WARPS * 32) + threadIdx.x;
    const bool live = c < a.nchains;
    if (!live) c = a.nchains - 1;
    const double* p = a.params + c * a.ldp;
    const double amp = p[0], om = 6.283185307179586476925287 / p[1], ph = p[2], p3 = p[3], p4 = p[4];
#ifndef MC3B_NO_FUSE_CODE
    __shared__ double vbuf[STAGE_DOUBLES];
    const MomentFix fix{a};
    FusedEntry fe;
    if (a.f.on) fe = fused_metropolis_load(a.f, fix, vbuf, c);
#endif
    const double b = p4 - m.slref;
    const double ac = fma(b, m.sxc, p3 - m.c0ref);             // L' at the centre
    const double j1 = rint((om - m.sw1) / m.sdelta), j2 = rint((2.0 * om - m.sw2) / m.sdelta);
    double q = __longlong_as_double(0x7ff8000000000000LL);
    if (j1 >= 0.0 && j1 < (double)m.sn1 && j2 >= 0.0 && j2 < (double)m.sn2) {
        const double d1 = om - fma(j1, m.sdelta, m.sw1), d2 = fma(2.0, om, -fma(j2, m.sdelta, m.sw2));
        const double2* tab = reinterpret_cast<const double2*>(m.spec + spec::HEAD);
        const double2* T = tab + (int64_t)j1 * (2 * K + 3);
        const double2* U = tab + (int64_t)m.sn1 * (2 * K + 3) + (int64_t)j2 * (K + 1);
        double2 t[K + 2], td[K + 1], u[K + 1];
#pragma unroll
        for (int k = 0; k < K + 2; k++) t[k] = T[k];
#pragma unroll
        for (int k = 0; k <= K; k++) { td[k] = T[K + 2 + k]; u[k] = U[k]; }
        // H = sum_k (i d1)^k [a T_1[k] + b (k+1) T_1[k+1] - T_d'[k]],  G = sum_k (i d2)^k U[k]
        double hr = 0.0, hi = 0.0, gr = 0.0, gi = 0.0;
#pragma unroll
        for (int k = K; k >= 0; k--) {
            const double bk = b * (double)(k + 1);
            const double cr = fma(ac, t[k].x, fma(bk, t[k + 1].x, -td[k].x));
            const double ci = fma(ac, t[k].y, fma(bk, t[k + 1].y, -td[k].y));
            const double nr = fma(-d1, hi, cr);
            hi = fma(d1, hr, ci); hr = nr;
            const double mr = fma(-d2, gi, u[k].x);
            gi = fma(d2, gr, u[k].y); gr = mr;
        }
        double sp, cp, s1, c1, s2, c2;
        sincos(ph, &sp, &cp);
        sincos(d1 * m.sxc, &s1, &c1);
        sincos(d2 * m.sxc, &s2, &c2);
        const double er = fma(cp, c1, -sp * s1), ei = fma(sp, c1, cp * s1);      // e^{i ph} e^{i d1 xc}
        const double im1 = fma(er, hi, ei * hr);
        const double pr = (cp - sp) * (cp + sp), pi = 2.0 * sp * cp;              // e^{2 i ph}
        const double fr = fma(pr, c2, -pi * s2), fi = fma(pr, s2, pi * c2);      // ... e^{i d2 xc}
        const double re2 = fma(fr, gr, -fi * gi);
        const double line = fma(ac, fma(h0, ac, 2.0 * fma(b, h1, -h3)), fma(b, fma(b, h2, -2.0 * h4), h5));
        q = fma(amp * amp, 0.5 * (h0 - re2), fma(2.0 * amp, im1, line)) * (w0 * w0);
    }
    if (live) a.partial[c] = q;
#ifndef MC3B_NO_FUSE_CODE
    if (a.f.on)
        fused_metropolis_apply(a.f, fe, vbuf, c, live, q, fix, [&](bool act, double& nxt) {
            return fix.guard(act, p, amp, p3, p4, w0, nxt);
        });
#endif
}

}  // namespace

int mc3b_launch_spectral_chisq(const ChisqArgs<double>& a, unsigned groups, cudaStream_t st) {
    if (a.m.sorder == 9) k_spectral_chisq<9><<<groups, WARPS * 32, 0, st>>>(a);
    else k_spectral_chisq<15><<<groups, WARPS * 32, 0, st>>>(a);
    MC3B_CHECK_LAUNCH("k_spectral_chisq");
    return MC3B_OK;
}

int mc3b_launch_spectral_prepare(const double* x, const double* d, int64_t n, double c0ref, double slref,
                                 const mc3b_spectral_t& s, cudaStream_t st) {
    const unsigned nb = (unsigned)(s.n1 + s.n2 + 1);
    if (s.order == 9)
        k_spectral_table<9><<<nb, 256, 0, st>>>(x, d, n, c0ref, slref, s.xc, s.w1, s.w2, s.delta, s.n1, s.n2, s.table);
    else
        k_spectral_table<15><<<nb, 256, 0, st>>>(x, d, n, c0ref, slref, s.xc, s.w1, s.w2, s.delta, s.n1, s.n2, s.table);
    MC3B_CHECK_LAUNCH("k_spectral_table");
    return MC3B_OK;
}

int mc3b_launch_sinefold(const ChisqArgs<double>& a0, double* work, unsigned groups, unsigned nsplit, cudaStream_t st) {
    const bool mom = a0.m.folded != nullptr;
    if (work == nullptr) {
        if (mom) { mc3b_set_error("the moment form needs the constants workspace (opts.work)"); return MC3B_ERR_ARG; }
        k_sinefold<false, false><<<dim3(groups, nsplit), WARPS * 32, 0, st>>>(a0);
        MC3B_CHECK_LAUNCH("k_sinefold");
        return MC3B_OK;
    }
    ChisqArgs<double> a = a0;
    a.consts = work; a.ldc = a.nchains; a.consts_wait = 0;
    k_fold_consts<<<(unsigned)((a.nchains + 127) / 128), 128, 0, st>>>(a.params, a.ldp, a.nchains, a.x, a.n,
                                                                        a.xt ? a.dxg : 0.0, work, a.ldc);
    MC3B_CHECK_LAUNCH("k_fold_consts");
    static const bool pdl = !(getenv("MC3B_FOLD_PDL") && atoi(getenv("MC3B_FOLD_PDL")) == 0);
    if (pdl) {
        // programmatic dependent launch: the CTAs set up their barriers and start the first
        // bulk copies while k_fold_consts runs, and wait for it only before reading the constants
        a.consts_wait = 1;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(groups, nsplit); cfg.blockDim = dim3(WARPS * 32); cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        if (mom && a.m.layout == 1) MC3B_CUDA(cudaLaunchKernelEx(&cfg, k_sinemma, a));
        else if (mom) MC3B_CUDA(cudaLaunchKernelEx(&cfg, k_sinefold<true, true>, a));
        else MC3B_CUDA(cudaLaunchKernelEx(&cfg, k_sinefold<true, false>, a));
    } else if (mom && a.m.layout == 1) {
        k_sinemma<<<dim3(groups, nsplit), WARPS * 32, 0, st>>>(a);
    } else if (mom) {
        k_sinefold<true, true><<<dim3(groups, nsplit), WARPS * 32, 0, st>>>(a);
    } else {
        k_sinefold<true, false><<<dim3(groups, nsplit), WARPS * 32, 0, st>>>(a);
    }
    MC3B_CHECK_LAUNCH("k_sinefold");
    return MC3B_OK;
}

int mc3b_launch_moment_finish(const ChisqArgs<double>& a, int nsplit, int npars, const double* prior, const double* plo,
                              const double* pup, double* chisq, cudaStream_t st) {
    k_moment_finish<<<(unsigned)((a.nchains + WARPS * 32 - 1) / (WARPS * 32)), WARPS * 32, 0, st>>>(a, nsplit, npars, prior,
                                                                                                  plo, pup, chisq);
    MC3B_CHECK_LAUNCH("k_moment_finish");
    return MC3B_OK;
}

int mc3b_launch_moment_prepare(const double* d, int64_t nt, double x0, double dx, const double* tile_x, double c0ref,
                               double slref, double* folded, double* tiles, int layout, cudaStream_t st) {
    if (nt == 0) return MC3B_OK;
    k_moment_prepare<<<(unsigned)((nt + 3) / 4), 128, 0, st>>>(d, nt, x0, dx, tile_x, c0ref, slref, folded, tiles, layout);
    MC3B_CHECK_LAUNCH("k_moment_prepare");
    return MC3B_OK;
}

int mc3b_launch_fold(const double* d, int64_t n, double* out, cudaStream_t st) {
    const int64_t nb = n / 16;
    if (nb == 0) return MC3B_OK;
    k_fold<<<(unsigned)((nb * 16 + 255) / 256), 256, 0, st>>>(d, nb, out);
    MC3B_CHECK_LAUNCH("k_fold");
    return MC3B_OK;
}

int mc3b_launch_sinegrid(const ChisqArgs<double>& a, bool usig, unsigned groups, unsigned nsplit, cudaStream_t st) {
    if (usig) k_sinegrid<true><<<dim3(groups, nsplit), WARPS * 32, 0, st>>>(a);
    else k_sinegrid<false><<<dim3(groups, nsplit), WARPS * 32, 0, st>>>(a);
    MC3B_CHECK_LAUNCH("k_sinegrid");
    return MC3B_OK;
}
