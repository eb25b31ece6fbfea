// mc3_b200 -- per-chain device functions of the sampler (shared by the
// per-generation kernels of sampler.cu and the persistent kernels of small.cu and batch.cu).
#pragma once
#include "common.cuh"

namespace {

constexpr int MAXP = MC3B_MAX_PARS;

struct Draws {                      // what one chain consumes in one generation
    int64_t a, b, iz;
    double usj, gs, u;
};

__device__ __forceinline__ void box_muller(double u1, double u2, double& n0, double& n1) {
    const double r = sqrt(-2.0 * log(1.0 - u1));     // 1-u1 in (0,1]
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    n0 = r * c;
    n1 = r * s;
}

// Peer-memory exchange: generation flags (include/mc3b200.h, F_peers).
// Precondition: every CTA that stored into peers has executed a system fence (after a CTA
// barrier) before the event that let this thread know the generation is complete.
// ONE system fence here (it orders everything this thread has observed -- the other CTAs'
// fenced stores included -- before the flags), then relaxed stores: a release store per
// peer made every flag wait for the previous flag's round trip over NVLink (~3.3 us per
// peer: +9 / +15 / +29 us per generation at 2 / 4 / 8 GPUs, profiles/r2_bench_n*.json).
__device__ __forceinline__ void flags_publish(const mc3b_sampler_t& S, int64_t done) {
    __threadfence_system();
    for (int p = 0; p < S.world; p++)
        asm volatile("st.relaxed.sys.global.s64 [%0], %1;" ::"l"(S.F_peers[p] + S.rank), "l"((long long)done)
                     : "memory");
}
// every thread of the CTA calls it (one thread per peer polls, then a CTA barrier)
__device__ __forceinline__ void flags_wait(const mc3b_sampler_t& S, int64_t gen) {
    if ((int)threadIdx.x < S.world) {
        const int64_t* f = S.F_peers[S.rank] + threadIdx.x;
        long long v;
        do {
            asm volatile("ld.acquire.sys.global.s64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        } while (v < (long long)gen);
    }
    __syncthreads();
}

// The per-parameter vectors a chain walks in loops (bounds, steps, priors, free
// indices) staged in shared memory by the whole CTA in one round of loads, and the
// sampler description repointed to them: a thread per chain otherwise pays a
// chain of dependent L2 latencies per parameter.  buf: STAGE_DOUBLES doubles.
// The peer pointer tables (X_peers, Z_peers, F_peers: [world] pointers in global memory)
// are staged too: the Metropolis step stores nfree values into every device, and a
// table read from global memory inside those loops cost one L2 round trip per (value,
// peer) -- +3.3 us per peer and generation at config 2 (profiles/r2_bench_n*.json).
constexpr int MAXW = 16;            // devices whose peer pointers are staged (more: read from global)
constexpr int STAGE_PEERS = 7 * MAXP + MAXP / 2;       // offset of the pointer slots in the staging buffer
constexpr int STAGE_DOUBLES = STAGE_PEERS + 3 * MAXW;
__device__ __forceinline__ void stage_peers_load(const mc3b_sampler_t& T, double* buf, int tid, int nthreads) {
    if (T.X_peers == nullptr || T.world > MAXW) return;
    void** slot = reinterpret_cast<void**>(buf + STAGE_PEERS);
    for (int i = tid; i < 3 * T.world; i += nthreads) {
        const int v = i / T.world, p = i - v * T.world;
        if (v == 0) slot[p] = T.X_peers[p];
        else if (v == 1) { if (T.Z_peers) slot[MAXW + p] = T.Z_peers[p]; }
        else if (T.F_peers) slot[2 * MAXW + p] = T.F_peers[p];
    }
}
__device__ __forceinline__ void stage_peers_point(mc3b_sampler_t& S, double* buf) {
    if (S.X_peers == nullptr || S.world > MAXW) return;
    void** slot = reinterpret_cast<void**>(buf + STAGE_PEERS);
    S.X_peers = reinterpret_cast<double* const*>(slot);
    if (S.Z_peers) S.Z_peers = reinterpret_cast<double* const*>(slot + MAXW);
    if (S.F_peers) S.F_peers = reinterpret_cast<int64_t* const*>(slot + 2 * MAXW);
}
// The CTA's share of the per-parameter vectors and of the free indices, NT threads: every
// load is issued before the first shared-memory store (a store between two loads would hold
// the second behind it, since the source is a generic pointer that may alias shared memory).
__device__ __forceinline__ const double* stage_src(const mc3b_sampler_t& T, int v) {
    return v == 0 ? T.pstep : v == 1 ? T.pmin : v == 2 ? T.pmax : v == 3 ? T.params0
         : v == 4 ? T.prior : v == 5 ? T.priorlow : T.priorup;
}
template <int NT>
__device__ __forceinline__ void stage_vectors_load(const mc3b_sampler_t& T, double* buf, int tid) {
    constexpr int NV = (7 * MAXP + NT - 1) / NT, NI = (MAXP + NT - 1) / NT;
    const int np = T.npars, nf = T.nfree;
    double val[NV];
    int32_t fr[NI];
#pragma unroll
    for (int r = 0; r < NV; r++) {
        const int i = tid + r * NT, v = i / np, k = i - v * np;
        const double* src = stage_src(T, v);
        val[r] = i < 7 * np && src ? src[k] : 0.0;
    }
#pragma unroll
    for (int r = 0; r < NI; r++) fr[r] = tid + r * NT < nf ? T.ifree[tid + r * NT] : 0;
#pragma unroll
    for (int r = 0; r < NV; r++) {
        const int i = tid + r * NT, v = i / np, k = i - v * np;
        if (i < 7 * np && stage_src(T, v)) buf[v * MAXP + k] = val[r];
    }
    int32_t* ifr = reinterpret_cast<int32_t*>(buf + 7 * MAXP);
#pragma unroll
    for (int r = 0; r < NI; r++)
        if (tid + r * NT < nf) ifr[tid + r * NT] = fr[r];
}
// S repointed to the staged copies (after a CTA barrier)
__device__ __forceinline__ void stage_point(mc3b_sampler_t& S, double* buf) {
    S.pstep = buf; S.pmin = buf + MAXP; S.pmax = buf + 2 * MAXP; S.params0 = buf + 3 * MAXP;
    if (S.prior) { S.prior = buf + 4 * MAXP; S.priorlow = buf + 5 * MAXP; S.priorup = buf + 6 * MAXP; }
    S.ifree = reinterpret_cast<int32_t*>(buf + 7 * MAXP);
    stage_peers_point(S, buf);
}
// the whole CTA of NT = blockDim.x threads
template <int NT>
__device__ __forceinline__ void stage_vectors(mc3b_sampler_t& S, double* buf) {
    stage_vectors_load<NT>(S, buf, threadIdx.x);
    stage_peers_load(S, buf, threadIdx.x, NT);
    __syncthreads();
    stage_point(S, buf);
}

// The proposal works on the free parameters in chunks of PCHUNK held in registers: the loads
// of a chunk (the chain's row, the partner or snooker rows) are issued together, before any
// store to nextp, and nothing of a chain's proposal lives in local memory.
constexpr int PCHUNK = 2;
static_assert(MAXP % PCHUNK == 0, "the parameter vectors are whole chunks");

// The random numbers chain c consumes in generation gen (chain.py:185, 197-203,
// 223-229, 257): a function of (seed, chain, generation) only -- not of the chains'
// states, so a proposal kernel launched as a programmatic dependent of the previous
// generation's model kernel draws them while that kernel is still running.
// chain_draws: partner indices, snooker draws and u; chain_normals: the support draws of
// the free parameters j0 .. j0 + PCHUNK - 1 (j0 a multiple of PCHUNK), scaled by pstep.
template <bool REPLAY>
__device__ __forceinline__ void chain_draws(const mc3b_sampler_t& S, const mc3b_draws_t& D, int64_t gen,
                                            int64_t zsize, int64_t c, Draws& dr) {
    dr.iz = -1; dr.usj = 1.0; dr.gs = 0.0;

    if (REPLAY) {
        dr.a = dr.b = 0;
        if (S.sampler != MC3B_MRW) { dr.a = D.a[c]; dr.b = D.b[c]; }
        if (S.sampler == MC3B_SNOOKER) { dr.iz = D.iz[c]; dr.usj = D.usj[c]; dr.gs = D.gs[c]; }
        dr.u = D.u[c];
    } else {
        const Philox ph(S.seed);
        const uint32_t cid = (uint32_t)c, g0 = (uint32_t)gen, g1 = (uint32_t)((uint64_t)gen >> 32);
        const uint4 w0 = ph(cid, 0u, g0, g1), w1 = ph(cid, 1u, g0, g1), w2 = ph(cid, 2u, g0, g1);
        if (S.sampler == MC3B_DEMC) {               // chain.py:223-229
            int64_t r1 = 1 + ubelow(w0.x, w0.y, S.nchains - 1);
            if (r1 == c) r1 = 0;
            int64_t r2 = (r1 + 2 + ubelow(w0.z, w0.w, S.nchains - 2)) % S.nchains;
            if (r2 == c) r2 = (r1 + 1) % S.nchains;
            dr.a = r1; dr.b = r2;
        } else if (S.sampler == MC3B_SNOOKER) {     // chain.py:197-203
            int64_t i1 = ubelow(w0.x, w0.y, zsize);
            int64_t i2 = 1 + ubelow(w0.z, w0.w, zsize - 1);
            if (i2 == i1) i2 = 0;
            dr.a = i1; dr.b = i2;
            dr.usj = u01(w1.x, w1.y);
            dr.gs = 1.2 + u01(w1.z, w1.w);
            dr.iz = ubelow(w2.x, w2.y, zsize);
        } else {
            dr.a = dr.b = 0;
        }
        dr.u = u01(w2.z, w2.w);
    }
}
template <bool REPLAY>
__device__ __forceinline__ void chain_normals(const mc3b_sampler_t& S, const mc3b_draws_t& D, int64_t gen, int64_t c,
                                              int j0, double (&nrm)[PCHUNK]) {
    const int nfree = S.nfree;
    if (REPLAY) {
#pragma unroll
        for (int q = 0; q < PCHUNK; q++) nrm[q] = j0 + q < nfree ? D.normal[j0 + q] : 0.0;
    } else {
        const Philox ph(S.seed);
        const uint32_t cid = (uint32_t)c, g0 = (uint32_t)gen, g1 = (uint32_t)((uint64_t)gen >> 32);
#pragma unroll
        for (int q = 0; q < PCHUNK; q += 2) {       // per-chain support draw
            const int j = j0 + q;
            nrm[q] = nrm[q + 1] = 0.0;
            if (j < nfree) {
                const uint4 w = ph(cid, 3u + (uint32_t)(j >> 1), g0, g1);
                double n0, n1;
                box_muller(u01(w.x, w.y), u01(w.z, w.w), n0, n1);
                nrm[q] = n0 * S.pstep[S.ifree[j]];
                if (j + 1 < nfree) nrm[q + 1] = n1 * S.pstep[S.ifree[j + 1]];
            }
        }
    }
}

// Jump, bounds, shared parameters and the snooker factor from the draws and the
// population as of the start of generation gen (chain.py:195-255).  nrm0: the support
// draws of the first chunk (chain_normals, j0 = 0); the later chunks draw their own.
// have_x0: xv0 holds the first chunk of the chain's row, already read.
template <bool REPLAY>
__device__ __forceinline__ void propose_apply(const mc3b_sampler_t& S, const mc3b_draws_t& D, const Draws& dr,
                                              const double (&nrm0)[PCHUNK], int64_t gen, int64_t c,
                                              bool have_x0 = false, const double (&xv0)[PCHUNK] = {}) {
    const int nfree = S.nfree, npars = S.npars;
    // population as of the start of this generation (peer mode: half gen & 1)
    const double* Xg = S.X_peers ? S.X_peers[S.rank] + (gen & 1) * S.nchains * nfree : S.X;
    const double* x = Xg + c * nfree;
    const bool snooker = S.sampler == MC3B_SNOOKER, demc = S.sampler == MC3B_DEMC;
    // rows the jump takes its difference from: z1 - z2 (snooker), x1 - x2 (demc)
    const double* r1 = snooker ? S.Z + dr.a * nfree : Xg + dr.a * nfree;
    const double* r2 = snooker ? S.Z + dr.b * nfree : Xg + dr.b * nfree;
    const bool sjump = snooker && dr.usj < 0.1;
    const double* zrow = sjump ? S.Z + dr.iz * nfree : x;

    // snooker jump (chain.py:202-213): sums over every free parameter before the first jump
    bool same = true;
    double zp1 = 0.0, zp2 = 0.0, dd = 0.0;
    if (sjump) {
#pragma unroll 1
        for (int j0 = 0; j0 < nfree; j0 += PCHUNK) {
            double xv[PCHUNK], zv[PCHUNK], av[PCHUNK], bv[PCHUNK];
#pragma unroll
            for (int q = 0; q < PCHUNK; q++) {
                const bool in = j0 + q < nfree;
                xv[q] = in ? x[j0 + q] : 0.0; zv[q] = in ? zrow[j0 + q] : 0.0;
                av[q] = in ? r1[j0 + q] : 0.0; bv[q] = in ? r2[j0 + q] : 0.0;
            }
#pragma unroll
            for (int q = 0; q < PCHUNK; q++) {
                if (j0 + q < nfree) {
                    same = same && (zv[q] == xv[q]);
                    const double dz = __dsub_rn(xv[q], zv[q]);
                    zp1 = __dadd_rn(zp1, __dmul_rn(av[q], dz));
                    zp2 = __dadd_rn(zp2, __dmul_rn(bv[q], dz));
                    dd = __dadd_rn(dd, __dmul_rn(dz, dz));
                }
            }
        }
    }
    const double f = __dmul_rn(dr.gs, __dsub_rn(zp1, zp2));

    // chain.py:235-247 -- propose, bounds, shared parameters
    double* np_ = S.nextp + c * npars;
    int inb = 1;
#pragma unroll 1
    for (int j0 = 0; j0 < nfree; j0 += PCHUNK) {
        double xv[PCHUNK], av[PCHUNK], bv[PCHUNK], zv[PCHUNK], nrm[PCHUNK];
#pragma unroll
        for (int q = 0; q < PCHUNK; q++) {          // one batch of loads per chunk
            const bool in = j0 + q < nfree;
            xv[q] = !in ? 0.0 : j0 == 0 && have_x0 ? xv0[q] : x[j0 + q];
            av[q] = in && (snooker || demc) ? r1[j0 + q] : 0.0;
            bv[q] = in && (snooker || demc) ? r2[j0 + q] : 0.0;
            zv[q] = in && sjump ? zrow[j0 + q] : 0.0;
        }
        if (j0 == 0) {
#pragma unroll
            for (int q = 0; q < PCHUNK; q++) nrm[q] = nrm0[q];
            for (int k = 0; k < npars; k++) np_[k] = S.params0[k];
        } else {
            chain_normals<REPLAY>(S, D, gen, c, j0, nrm);
        }
#pragma unroll
        for (int q = 0; q < PCHUNK; q++) {
            const int j = j0 + q;
            if (j >= nfree) break;
            double jump;
            if (sjump) {
                jump = same ? __dmul_rn(dr.gs, __dsub_rn(bv[q], av[q]))
                            : __ddiv_rn(__dmul_rn(f, __dsub_rn(xv[q], zv[q])), dd);
            } else if (snooker || demc) {           // chain.py:214-217, 230-232
                jump = __dadd_rn(__dmul_rn(S.gamma, __dsub_rn(av[q], bv[q])), __dmul_rn(S.fepsilon, nrm[q]));
            } else {                                // mrw, chain.py:219-220
                jump = nrm[q];
            }
            const int k = S.ifree[j];
            double v = __dadd_rn(xv[q], jump);
            if (S.reflect) {                        // opt-in, non-reference behaviour
                const double lo = S.pmin[k], hi = S.pmax[k];
                for (int it = 0; it < 8 && (v < lo || v > hi); it++) v = v < lo ? 2.0 * lo - v : 2.0 * hi - v;
            }
            np_[k] = v;
            if (v < S.pmin[k] || v > S.pmax[k]) {
                inb = 0;
                atomicAdd(&S.outbounds[j], 1);
            }
        }
    }
    for (int k = 0; k < npars; k++)
        if (S.pstep[k] < 0.0) np_[k] = np_[-(int)S.pstep[k] - 1];
    double mrfactor = 1.0;
    if (sjump && inb) {                              // chain.py:251-255
        double cn = 0.0, nn = 0.0;
        for (int j = 0; j < nfree; j++) {
            const double dc = __dsub_rn(x[j], zrow[j]), dn = __dsub_rn(np_[S.ifree[j]], zrow[j]);
            cn = __dadd_rn(cn, __dmul_rn(dc, dc));
            nn = __dadd_rn(nn, __dmul_rn(dn, dn));
        }
        mrfactor = pow(nn / cn, 0.5 * (nfree - 1));
    }
    S.mrfactor[c] = mrfactor;
    S.u[c] = dr.u;
    S.inb[c] = inb;
}

// Proposal of chain c for generation gen (chain.py:185-247, 251-255).
template <bool REPLAY>
__device__ __forceinline__ void propose_chain(const mc3b_sampler_t& S, const mc3b_draws_t& D, int64_t gen,
                                              int64_t zsize, int64_t c) {
    Draws dr;
    double nrm[PCHUNK];
    chain_draws<REPLAY>(S, D, gen, zsize, c, dr);
    chain_normals<REPLAY>(S, D, gen, c, 0, nrm);
    propose_apply<REPLAY>(S, D, dr, nrm, gen, c);
}

// Data chi-squared of a proposal: the partial rows of the model kernel added in
// split order (fixed order = identical bits wherever the sum is taken).  CG: read
// through L2 (rows written by other SMs during the same kernel).
template <bool CG>
__device__ __forceinline__ double sum_partials(const double* partial, int64_t ldpartial, int nsplit, int64_t col) {
    double nxt = 0.0;
    const double* p = partial + col;
    int s = 0;
    for (; s + 32 <= nsplit; s += 32) {             // 32 loads in flight (the rows come from L2), added in order
        double v[32];
#pragma unroll
        for (int k = 0; k < 32; k++) v[k] = CG ? __ldcg(p + (int64_t)(s + k) * ldpartial) : p[(int64_t)(s + k) * ldpartial];
#pragma unroll
        for (int k = 0; k < 32; k++) nxt += v[k];
    }
    for (; s + 8 <= nsplit; s += 8) {
        double v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = CG ? __ldcg(p + (int64_t)(s + k) * ldpartial) : p[(int64_t)(s + k) * ldpartial];
#pragma unroll
        for (int k = 0; k < 8; k++) nxt += v[k];
    }
    for (; s < nsplit; s++) nxt += CG ? __ldcg(p + (int64_t)s * ldpartial) : p[(int64_t)s * ldpartial];
    return nxt;
}

// The Metropolis step of chain c (chain.py:257-289) in two halves.  metropolis_load reads
// what the step needs of the chain's state: none of it depends on the proposal's
// chi-squared, and during a launch only the chain's own thread writes it (k_propose wrote
// inb, mrfactor and u before), so a kernel may issue these loads at entry, in one batch, and
// apply the step once the chi-squared is known.
struct ChainState {
    int inb;
    int32_t nacc;
    double cur, mrf, u, best;
    double xv[PCHUNK];              // the chain's current row, first chunk
};
// x of chain c in generation gen (peer mode: half gen & 1 of this device)
__device__ __forceinline__ double* chain_row(const mc3b_sampler_t& S, int64_t gen, int64_t c) {
    if (S.X_peers) return S.X_peers[S.rank] + (gen & 1) * S.nchains * S.nfree + c * S.nfree;
    return S.X + c * S.nfree;
}
__device__ __forceinline__ ChainState metropolis_load(const mc3b_sampler_t& S, int64_t gen, int64_t c) {
    const int nfree = S.nfree;
    const double* x = chain_row(S, gen, c);
    const double* np_ = S.nextp + c * S.npars;
    ChainState st;
    st.inb = S.inb[c];
    st.cur = S.chisq_cur[c];
    st.mrf = S.mrfactor[c]; st.u = S.u[c]; st.best = S.best_chisq[c];
    st.nacc = S.naccept[c];
#pragma unroll
    for (int q = 0; q < PCHUNK; q++) st.xv[q] = q < nfree ? x[q] : 0.0;
    // the rest of both rows goes to L1 meanwhile, without holding registers across the step
    // (generic prefetch: no operation on a row in shared memory)
    asm volatile("prefetch.L1 [%0];" ::"l"(np_));
    asm volatile("prefetch.L1 [%0];" ::"l"(np_ + S.npars - 1));
    asm volatile("prefetch.L1 [%0];" ::"l"(x + nfree - 1));
    return st;
}

// nxt_data = data chi-squared of the proposal (unused when the proposal was out of bounds)
__device__ __forceinline__ void metropolis_apply(const mc3b_sampler_t& S, const ChainState& st, double nxt_data,
                                                 int64_t gen, int64_t zrow0, int64_t c) {
    const int nfree = S.nfree, npars = S.npars;
    const bool peer = S.X_peers != nullptr;
    double* x = chain_row(S, gen, c);
    const double* np_ = S.nextp + c * npars;
    double cur = st.cur;
    const double mrf = st.mrf, u = st.u, best = st.best;
    const int32_t nacc = st.nacc;
    bool accept = false, newbest = false;
    if (st.inb) {
        double nxt = nxt_data;
        if (S.prior != nullptr) {                    // stats.py:208-216 + stats.h:90-109
            double pr = 0.0;
            for (int k = 0; k < npars; k++) {
                const double lo = S.priorlow[k], up = S.priorup[k];
                if (lo > 0.0 && up > 0.0) {
                    const double off = np_[k] - S.prior[k];
                    const double t = off / (off > 0.0 ? up : lo);
                    pr += t * t;
                }
            }
            nxt += pr;
        }
        const double ratio = exp(0.5 * (cur - nxt)) * mrf;
        if (ratio > u) {                        // chain.py:257-274 (NaN rejects)
            accept = true;
            cur = nxt;
            S.chisq_cur[c] = nxt;
            S.naccept[c] = nacc + 1;
            if (nxt < best) {
                newbest = true;
                S.best_chisq[c] = nxt;
                S.best_gen[c] = gen;
            }
        }
    }
    const bool write = zrow0 >= 0 && zrow0 + c < S.zlen;
    const int64_t row = zrow0 + c;
    // the chain's next state v (chain.py:276-289) into best_x, x and the thinned history, or in peer
    // mode into half (gen+1)&1 of EVERY device (NVLink peer stores; thinned rows likewise when the
    // history is shared).  A chunk's loads are issued before its stores: the rows may alias as far
    // as the compiler knows, and a store between two loads would hold the second behind it.
    const int64_t dst = ((gen + 1) & 1) * S.nchains * nfree + c * nfree;
    if (accept || write || peer) {
#pragma unroll 1
        for (int j0 = 0; j0 < nfree; j0 += PCHUNK) {
            double v[PCHUNK];
#pragma unroll
            for (int q = 0; q < PCHUNK; q++) {
                const int j = j0 + q;
                v[q] = j >= nfree ? 0.0 : accept ? np_[S.ifree[j]] : j0 == 0 ? st.xv[q] : x[j];
            }
#pragma unroll
            for (int q = 0; q < PCHUNK; q++) {
                const int j = j0 + q;
                if (j >= nfree) break;
                if (newbest) S.best_x[c * nfree + j] = v[q];
                if (!peer) {
                    if (accept) x[j] = v[q];
                    if (write) S.Z[row * nfree + j] = v[q];
                } else {
                    for (int p = 0; p < S.world; p++) S.X_peers[p][dst + j] = v[q];
                    if (write) {
                        if (S.Z_peers) { for (int p = 0; p < S.world; p++) S.Z_peers[p][row * nfree + j] = v[q]; }
                        else S.Z[row * nfree + j] = v[q];
                    }
                }
            }
        }
    }
    // (no fence for the peer stores: the caller orders the CTA's peer stores with ONE system fence
    // after a CTA barrier, before it counts the group as done -- see fused_metropolis / k_metropolis)
    if (write) {
        S.log_post[row] = -0.5 * cur;
        S.zchain[row] = (int32_t)c;
    }
}
// both halves back to back
__device__ __forceinline__ void metropolis_chain(const mc3b_sampler_t& S, double nxt_data, int64_t gen, int64_t zrow0,
                                                 int64_t c) {
    metropolis_apply(S, metropolis_load(S, gen, c), nxt_data, gen, zrow0, c);
}

// Trial point t of round `round` of the initial population (mcmc_driver.py:229-262): v[0..npars)
// = params0 with the free entries drawn N(params0, pstep) (kickoff 0) or U(pmin, pmax) (kickoff 1)
// from Philox counter (t, slot, round, 0xFFFFFFFF), shared parameters filled.  Returns 1 when
// every parameter is inside [pmin, pmax] (mcmc_driver.py:252).
__device__ __forceinline__ int init_trial(const mc3b_sampler_t& S, int kickoff, int64_t t, int64_t round, double* v) {
    const Philox ph(S.seed);
    for (int k = 0; k < S.npars; k++) v[k] = S.params0[k];
    int good = 1;
    for (int j = 0; j < S.nfree; j += 2) {
        const uint4 w = ph((uint32_t)t, (uint32_t)(j >> 1), (uint32_t)round, 0xFFFFFFFFu);
        double d0, d1;
        if (kickoff == 0) box_muller(u01(w.x, w.y), u01(w.z, w.w), d0, d1);
        else { d0 = u01(w.x, w.y); d1 = u01(w.z, w.w); }
        for (int q = 0; q < 2 && j + q < S.nfree; q++) {
            const int k = S.ifree[j + q];
            const double d = q ? d1 : d0;
            v[k] = kickoff == 0 ? S.params0[k] + S.pstep[k] * d : S.pmin[k] + (S.pmax[k] - S.pmin[k]) * d;
        }
    }
    for (int k = 0; k < S.npars; k++)
        if (S.pstep[k] < 0.0) v[k] = v[-(int)S.pstep[k] - 1];
    for (int k = 0; k < S.npars; k++)
        if (v[k] > S.pmax[k] || v[k] < S.pmin[k]) good = 0;
    return good;
}

}  // namespace
