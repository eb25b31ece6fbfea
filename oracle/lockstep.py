"""ORACLE (test infrastructure only): numpy restatement of a production-mode
generation of the CUDA sampler, vectorised over chains.

It follows, statement by statement:

  Philox4x32-10, u01, ubelow            mc3_b200/csrc/common.cuh
  box_muller, chain_draws,              mc3_b200/csrc/sampler_dev.cuh
  chain_normals, propose_apply,
  metropolis_apply
  k_init_trials                         mc3_b200/csrc/sampler.cu
  zsize / history-row rules             mc3_b200/engine.py (_generation, _zrow0),
                                        sampler.cu k_propose, small.cu k_run_small
  initial population (draw order)       mc3_b200/engine.py Population.init_population

The jump arithmetic of propose_apply uses explicit round-to-nearest operations
(__dmul_rn / __dadd_rn / __dsub_rn / __ddiv_rn), so `propose` below reproduces it
bit for bit from the same inputs.  Box-Muller (log, sincospi), pow and exp are
not correctly rounded on the device; what depends on them agrees to a few ulps.

`propose` takes the population it reads as an argument, so one code path serves
both orders: the reference's sequential order (chains move in place, fed the
reference's recorded draws; tests/test_lockstep_cpu.py pins it to
tests/golden/mcmc_*.npz) and the lock-step order of production mode (every chain
reads the population as of the start of the generation).
"""
import numpy as np

MRW, DEMC, SNOOKER = 'mrw', 'demc', 'snooker'
_M32 = np.uint64(0xFFFFFFFF)


# ---------------------------------------------------------------------------
# random-number primitives (common.cuh)
# ---------------------------------------------------------------------------
def philox(seed, c0, c1, c2, c3):
    """Philox4x32-10 with key = (seed low word, seed high word); the counter words
    broadcast against each other.  Returns four uint64 arrays holding 32-bit words."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _M32 for c in np.broadcast_arrays(c0, c1, c2, c3))
    a, b = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    w0, w1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = m0*c0, m1*c2                     # 32 x 32 -> 64 bits: exact in uint64
        hi0, lo0 = p0 >> s32, p0 & _M32
        hi1, lo1 = p1 >> s32, p1 & _M32
        c0, c1, c2, c3 = hi1 ^ c1 ^ a, lo1, hi0 ^ c3 ^ b, lo0
        a, b = (a + w0) & _M32, (b + w1) & _M32
    return c0, c1, c2, c3


def u01(a, b):
    """53-bit uniform in [0, 1) from two 32-bit words, (a>>5, b>>6) (exact)."""
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    return ((a >> np.uint64(5)).astype(np.float64)*67108864.0
            + (b >> np.uint64(6)).astype(np.float64))*(1.0/9007199254740992.0)


def ubelow(a, b, n):
    """Integer in [0, n) from 64 random bits: the high word of ((a << 32) | b) * n,
    in Python integers.  Arrays in, int64 array out."""
    a, b, n = np.broadcast_arrays(np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64),
                                  np.asarray(n, dtype=np.int64))
    vals = [(((x << 32) | y)*m) >> 64 for x, y, m in zip(a.ravel().tolist(), b.ravel().tolist(),
                                                          n.ravel().tolist())]
    return np.array(vals, dtype=np.int64).reshape(a.shape)


def box_muller(u1, u2):
    """Two normals from two uniforms: r = sqrt(-2 log(1-u1)), (r cos 2 pi u2, r sin 2 pi u2)."""
    r = np.sqrt(-2.0*np.log(1.0 - u1))
    t = np.pi*(2.0*u2)
    return r*np.cos(t), r*np.sin(t)


# ---------------------------------------------------------------------------
# draws of one generation (sampler_dev.cuh chain_draws / chain_normals)
# ---------------------------------------------------------------------------
def chain_draws(seed, sampler, nchains, gen, zsize, chains=None):
    """Partner / snooker draws and u of `chains` (default: all) in generation gen:
    dict of arrays a, b, iz, usj, gs, u.  Counter = (chain, slot, gen lo, gen hi)."""
    c = np.arange(nchains, dtype=np.int64) if chains is None else np.asarray(chains, dtype=np.int64)
    g0, g1 = int(gen) & 0xFFFFFFFF, (int(gen) >> 32) & 0xFFFFFFFF
    w0 = philox(seed, c, 0, g0, g1)
    w1 = philox(seed, c, 1, g0, g1)
    w2 = philox(seed, c, 2, g0, g1)
    k = c.size
    d = dict(a=np.zeros(k, np.int64), b=np.zeros(k, np.int64), iz=np.full(k, -1, np.int64),
             usj=np.ones(k), gs=np.zeros(k))
    if sampler == DEMC:                               # chain.py:223-229
        r1 = 1 + ubelow(w0[0], w0[1], nchains - 1)
        r1 = np.where(r1 == c, 0, r1)
        r2 = (r1 + 2 + ubelow(w0[2], w0[3], nchains - 2)) % nchains
        r2 = np.where(r2 == c, (r1 + 1) % nchains, r2)
        d['a'], d['b'] = r1, r2
    elif sampler == SNOOKER:                          # chain.py:197-203
        i1 = ubelow(w0[0], w0[1], zsize)
        i2 = 1 + ubelow(w0[2], w0[3], zsize - 1)
        i2 = np.where(i2 == i1, 0, i2)
        d['a'], d['b'] = i1, i2
        d['usj'] = u01(w1[0], w1[1])
        d['gs'] = 1.2 + u01(w1[2], w1[3])
        d['iz'] = ubelow(w2[0], w2[1], zsize)
    elif sampler != MRW:
        raise ValueError(sampler)
    d['u'] = u01(w2[2], w2[3])
    return d


def chain_normals(seed, nchains, gen, pstep, ifree, chains=None):
    """Support draws [len(chains), nfree], scaled by pstep: slot 3 + j//2 gives the
    pair of free parameters (j, j+1)."""
    c = np.arange(nchains, dtype=np.int64) if chains is None else np.asarray(chains, dtype=np.int64)
    nfree = len(ifree)
    g0, g1 = int(gen) & 0xFFFFFFFF, (int(gen) >> 32) & 0xFFFFFFFF
    out = np.zeros((c.size, nfree))
    for j in range(0, nfree, 2):
        w = philox(seed, c, 3 + j//2, g0, g1)
        n0, n1 = box_muller(u01(w[0], w[1]), u01(w[2], w[3]))
        out[:, j] = n0*pstep[ifree[j]]
        if j + 1 < nfree:
            out[:, j + 1] = n1*pstep[ifree[j + 1]]
    return out


# ---------------------------------------------------------------------------
# the sampler description
# ---------------------------------------------------------------------------
class Spec:
    """What a generation needs besides the population: the vectors of the fit and
    the jump scales (engine.Population: gamma = fgamma 2.38 / sqrt(2 nfree))."""

    def __init__(self, params, pstep, pmin=None, pmax=None, prior=None, priorlow=None,
                 priorup=None, sampler=DEMC, fgamma=1.0, fepsilon=0.0, seed=0):
        self.params0 = np.array(params, dtype=float)
        npars = self.params0.size
        self.pstep = np.asarray(pstep, dtype=float)
        self.pmin = np.full(npars, -np.inf) if pmin is None else np.asarray(pmin, dtype=float)
        self.pmax = np.full(npars, np.inf) if pmax is None else np.asarray(pmax, dtype=float)
        z = np.zeros(npars)
        self.prior = z if prior is None else np.asarray(prior, dtype=float)
        self.priorlow = z if priorlow is None else np.asarray(priorlow, dtype=float)
        self.priorup = z if priorup is None else np.asarray(priorup, dtype=float)
        self.ifree = np.where(self.pstep > 0)[0]
        self.npars, self.nfree = npars, self.ifree.size
        self.sampler = sampler
        self.gamma = float(fgamma)*2.38/np.sqrt(2*self.nfree)
        self.fepsilon = float(fepsilon)
        self.seed = int(seed)


# ---------------------------------------------------------------------------
# proposal (sampler_dev.cuh propose_apply)
# ---------------------------------------------------------------------------
def propose(spec, X, Z, draws, normals, chains=None):
    """Proposals of `chains` (default: every row of X) read from the population X
    [nchains, nfree] and the history Z [>= zsize, nfree] as given.

    draws: chain_draws() of those chains; normals: [len(chains), nfree] support
    draws (already scaled by pstep).  Returns a dict:
      nextp [k, npars]   full vectors (fixed and shared slots filled)
      inb [k] bool, out [k, nfree] bool (per free parameter out of bounds)
      mrfactor [k], jump [k, nfree], sjump [k] bool
      exact [k] bool     the support term is exactly zero (DEMC with fepsilon = 0,
                         snooker jumps): the device's proposal is bit for bit this one
    """
    s = spec
    c = np.arange(X.shape[0]) if chains is None else np.asarray(chains, dtype=np.int64)
    k, nfree = c.size, s.nfree
    x = X[c]
    snooker, demc = s.sampler == SNOOKER, s.sampler == DEMC
    a, b = draws['a'], draws['b']
    if snooker:
        r1, r2 = Z[a], Z[b]
    elif demc:
        r1, r2 = X[a], X[b]
    else:
        r1 = r2 = np.zeros_like(x)
    sjump = snooker & (draws['usj'] < 0.1)
    iz = np.where(sjump, draws['iz'], 0)
    zrow = np.where(sjump[:, None], Z[iz], x)

    # snooker jump (chain.py:202-213): sums in free-parameter order
    same = np.all(zrow == x, axis=1)
    zp1, zp2, dd = np.zeros(k), np.zeros(k), np.zeros(k)
    for j in range(nfree):
        dz = x[:, j] - zrow[:, j]
        zp1 = zp1 + r1[:, j]*dz
        zp2 = zp2 + r2[:, j]*dz
        dd = dd + dz*dz
    gs = draws['gs']
    f = gs*(zp1 - zp2)

    jump = np.empty((k, nfree))
    with np.errstate(all='ignore'):
        for j in range(nfree):
            if snooker or demc:
                plain = s.gamma*(r1[:, j] - r2[:, j]) + s.fepsilon*normals[:, j]
            else:
                plain = normals[:, j]
            if snooker:
                sj = np.where(same, gs*(r2[:, j] - r1[:, j]), (f*(x[:, j] - zrow[:, j]))/dd)
                jump[:, j] = np.where(sjump, sj, plain)
            else:
                jump[:, j] = plain
    v = x + jump
    nextp = np.tile(s.params0, (k, 1))
    nextp[:, s.ifree] = v
    out = (v < s.pmin[s.ifree]) | (v > s.pmax[s.ifree])
    inb = ~np.any(out, axis=1)
    for q in range(s.npars):                          # shared parameters, in slot order
        if s.pstep[q] < 0:
            nextp[:, q] = nextp[:, -int(s.pstep[q]) - 1]
    mrf = np.ones(k)
    m = sjump & inb
    if np.any(m):                                     # chain.py:251-255
        cn, nn = np.zeros(k), np.zeros(k)
        for j in range(nfree):
            dc = x[:, j] - zrow[:, j]
            dn = nextp[:, s.ifree[j]] - zrow[:, j]
            cn = cn + dc*dc
            nn = nn + dn*dn
        with np.errstate(all='ignore'):
            mrf = np.where(m, (nn/cn)**(0.5*(nfree - 1)), 1.0)
    exact = sjump | (s.sampler != MRW and s.fepsilon == 0.0)
    return dict(nextp=nextp, inb=inb, out=out, mrfactor=mrf, jump=jump, sjump=sjump,
                exact=np.broadcast_to(exact, (k,)).copy(), x=x)


# ---------------------------------------------------------------------------
# Metropolis step (sampler_dev.cuh metropolis_apply)
# ---------------------------------------------------------------------------
def prior_terms(spec, nextp):
    """Gaussian two-sided prior terms of full vectors [k, npars]: sum over every
    parameter with priorlow > 0 and priorup > 0 of (off / (up if off > 0 else lo))^2.
    One-sided priors (priorlow < 0) add nothing here."""
    s = spec
    pr = np.zeros(nextp.shape[0])
    for q in range(s.npars):
        lo, up = s.priorlow[q], s.priorup[q]
        if lo > 0.0 and up > 0.0:
            off = nextp[:, q] - s.prior[q]
            t = off/np.where(off > 0.0, up, lo)
            pr = pr + t*t
    return pr


def log_margin(cur, nxt, mrf, u):
    """0.5 (cur - nxt) + log mrf - log u: the decision accepts where this is > 0
    (exp(0.5 (cur - nxt)) mrf > u)."""
    with np.errstate(all='ignore'):
        return 0.5*(cur - nxt) + np.log(mrf) - np.log(u)


def decide(cur, nxt, mrf, u):
    """exp(0.5 (cur - nxt)) * mrf > u; NaN rejects."""
    with np.errstate(all='ignore'):
        return np.exp(0.5*(cur - nxt))*mrf > u


class State:
    """Per-chain sampler state and counters of a restated run."""

    def __init__(self, X, cur, nfree):
        n = X.shape[0]
        self.X = np.array(X, dtype=float)
        self.cur = np.array(cur, dtype=float)
        self.naccept = np.zeros(n, np.int64)
        self.outbounds = np.zeros(nfree, np.int64)
        self.best_chisq = np.full(n, np.inf)
        self.best_gen = np.zeros(n, np.int64)
        self.best_x = np.zeros((n, nfree))


def metropolis(spec, st, chains, prop, nxt_data, u, gen, accept=None):
    """Apply the step of `chains` to State st: prior terms, decision (or the given
    `accept` mask), counters, per-chain best.  nxt_data: data chi-squared of the
    proposals (ignored where out of bounds).  Returns (accept mask, nxt)."""
    c = np.asarray(chains, dtype=np.int64)
    nxt = np.where(prop['inb'], nxt_data, np.nan) + prior_terms(spec, prop['nextp'])
    if accept is None:
        accept = prop['inb'] & decide(st.cur[c], nxt, prop['mrfactor'], u)
    accept = accept & prop['inb']
    st.outbounds += prop['out'].sum(axis=0)
    ca = c[accept]
    st.X[ca] = prop['nextp'][accept][:, spec.ifree]
    st.cur[ca] = nxt[accept]
    st.naccept[ca] += 1
    nb = accept & (nxt < st.best_chisq[c])
    cb = c[nb]
    st.best_chisq[cb] = nxt[nb]
    st.best_gen[cb] = gen
    st.best_x[cb] = prop['nextp'][nb][:, spec.ifree]
    return accept, nxt


# ---------------------------------------------------------------------------
# history layout (engine._zrow0, k_propose, k_run_small)
# ---------------------------------------------------------------------------
def zsize(M0, nchains, thinning, gen):
    """History rows a proposal of generation gen may read."""
    return M0 + (gen//thinning)*nchains


def zrow0(M0, nchains, thinning, gen):
    """First history row generation gen writes, or -1 when it writes none."""
    if (gen + 1) % thinning:
        return -1
    return M0 + ((gen + 1)//thinning - 1)*nchains


# ---------------------------------------------------------------------------
# initial population (k_init_trials, engine.init_population)
# ---------------------------------------------------------------------------
def init_trials(spec, kickoff, round_, nt):
    """Trial vectors [nt, npars] and their in-bounds flags: counter =
    (t, j//2, round, 0xFFFFFFFF).  kickoff 'normal': params0 + pstep * normal;
    'uniform': pmin + (pmax - pmin) * u."""
    s = spec
    t = np.arange(nt, dtype=np.int64)
    v = np.tile(s.params0, (nt, 1))
    for j in range(0, s.nfree, 2):
        w = philox(s.seed, t, j//2, round_, 0xFFFFFFFF)
        if kickoff == 'normal':
            d0, d1 = box_muller(u01(w[0], w[1]), u01(w[2], w[3]))
        else:
            d0, d1 = u01(w[0], w[1]), u01(w[2], w[3])
        for q, d in ((0, d0), (1, d1)):
            if j + q >= s.nfree:
                break
            k = s.ifree[j + q]
            if kickoff == 'normal':
                v[:, k] = s.params0[k] + s.pstep[k]*d
            else:
                v[:, k] = s.pmin[k] + (s.pmax[k] - s.pmin[k])*d
    for k in range(s.npars):
        if s.pstep[k] < 0:
            v[:, k] = v[:, -int(s.pstep[k]) - 1]
    ok = ~np.any((v > s.pmax) | (v < s.pmin), axis=1)
    return v, ok


def init_population(spec, kickoff, M0, chisq_fn):
    """The M0 initial rows in draw order, as engine.init_population takes them:
    batches of nt trials per round; the in-bounds ones up to the count still needed
    (+ max(8, need//100)) are evaluated, and those with a finite chi-squared are
    taken in draw order.  chisq_fn(P [k, npars]) -> chi-squared incl. priors.
    Returns (rows [M0, nfree], log_post [M0], list of (round, trial index))."""
    got = tried = rnd = 0
    rows, lps, picks = [], [], []
    while got < M0 and tried < 100*M0:
        nt = int(min(max(M0 - got, 64)*1.25 + 64, 100*M0 - tried))
        v, ok = init_trials(spec, kickoff, rnd, nt)
        inb = np.nonzero(ok)[0]
        need = M0 - got
        inb = inb[:need + max(8, need//100)]
        tried += int(inb[-1]) + 1 if inb.size else nt
        if inb.size:
            lp = -0.5*chisq_fn(v[inb])
            idx = np.nonzero(np.isfinite(lp))[0][:need]
            rows.append(v[inb[idx]][:, spec.ifree])
            lps.append(lp[idx])
            picks += [(rnd, int(t)) for t in inb[idx]]
            got += idx.size
        rnd += 1
    if got < M0:
        raise ValueError('cannot populate the initial sample')
    return np.concatenate(rows), np.concatenate(lps), picks
