"""Production-mode generations checked chain by chain against oracle/lockstep.py,
the numpy restatement of the lock-step sampler that tests/test_lockstep_cpu.py
pins to the reference's recorded runs.

Method: a Population runs with thinning = 1, so its history holds the whole
trajectory: X_0 = Z[:n], cur_0 = -2 log_post[:n] (set_initial), and after
generation g the chains' rows and chi-squared are rows M0 + g n ... of Z and
log_post.  For every generation the restatement recomputes each chain's Philox
draws and proposal from the DEVICE's state before the step, evaluates its
chi-squared in numpy, and checks what the device wrote: one ulp can never compound
into diverging chains, and a wrong partner, draw slot, prior, zsize, decision or
history row shows up at the first generation and chain it touches.

Tolerances:
  rows       bit for bit where the support term is exactly zero (DEMC and snooker
             with fepsilon = 0, snooker jumps: propose_apply rounds every operation
             explicitly); else within 4 eps (|x| + |jump|) per element (Box-Muller goes
             through the device's log and sincospi).
  log_post   rtol 1e-10 in fp64 (the chi-squared forms sit within 1.2e-11 of the
             exact sum), 1e-5 in fp32.
  marginal   a proposal within 4 eps (|x| + |jump|) of a bound, or a decision with
             |0.5 (cur - nxt) + log mrf - log u| < 1e-9 max(cur, nxt, 1) (fp64; 100x the
             chi-squared error) or 1e-5 max(cur, nxt, 1) (fp32; twice the margin error the
             log_post bound allows), is resolved by what the device did and counted; the
             counts are bounded (1e-3 of the chain-steps in fp64, 5 % in fp32).
"""
import contextlib
import os

import numpy as np
import pytest
import torch

from oracle import kernels as ok
from oracle import lockstep as ls
from oracle import models as om

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
TRUTH = np.array([1.0, 2.5, 1.0, 5.0, -0.2])      # amplitude = phase: p2 shares p0's value


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


@contextlib.contextmanager
def env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update({k: str(v) for k, v in kw.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ---------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------
def sine_fit(n, sigma=0.5, seed=1, x=None, uncert=None):
    """Sinusoid + line with a shared phase (p2 := p0), a fixed slope, a two-sided prior
    of unequal widths on the period, on the amplitude and on the shared phase, a
    one-sided prior on the offset (ignored by the chi-squared), and bounds on the
    amplitude and the offset that cut through the posterior."""
    rs = np.random.RandomState(seed)
    x = np.linspace(0.0, 10.0, n) if x is None else x
    unc = np.full(x.size, sigma) if uncert is None else uncert
    data = om.sinusoid(TRUTH, x) + rs.normal(0.0, 1.0, x.size)*unc
    return dict(
        data=data, uncert=unc, x=x, func='sinusoid', params=np.array([1.01, 2.505, 1.01, 5.01, -0.2]),
        pstep=np.array([1e-2, 1e-3, -1.0, 1e-2, 0.0]),
        pmin=np.array([0.99, 2.3, -np.pi, 4.994, -1.0]), pmax=np.array([1.035, 2.7, np.pi, 5.03, 1.0]),
        prior=np.array([1.0, 2.5, 1.0, 5.0, 0.0]), priorlow=np.array([0.02, 0.1, 0.03, 0.05, 0.0]),
        priorup=np.array([0.05, 0.2, 0.01, 0.0, 0.0]))


def poly_fit(n, seed=2):
    """Quartic on a jittered abscissa (the generic model kernel): p3 := p1, p4 fixed."""
    rs = np.random.RandomState(seed)
    x = np.sort(rs.uniform(-1.0, 1.0, n))
    pt = np.array([1.0, 0.5, -0.7, 0.5, 0.25])
    unc = rs.uniform(0.05, 0.15, n)
    data = om.polynomial(pt, x) + rs.normal(0.0, 1.0, n)*unc
    return dict(
        data=data, uncert=unc, x=x, func='polynomial', params=np.array([1.002, 0.498, -0.698, 0.498, 0.25]),
        pstep=np.array([2e-3, 2e-3, 3e-3, -2.0, 0.0]),
        pmin=np.array([0.998, -5.0, -0.705, -5.0, -5.0]), pmax=np.array([1.006, 5.0, 5.0, 5.0, 5.0]),
        prior=np.array([1.0, 0.5, 0.0, 0.5, 0.25]), priorlow=np.array([0.01, 0.02, 0.0, 0.0, 0.1]),
        priorup=np.array([0.03, 0.01, 0.0, 0.0, 0.2]))


def data_chisq_fn(f, model, batch_points=256*20000):
    """Data chi-squared of full vectors [k, npars] in numpy, batched over chains."""
    x, d, w = f['x'], f['data'], 1.0/f['uncert']

    def chi(P):
        out = np.empty(P.shape[0])
        b = max(1, min(256, batch_points//x.size))
        for i in range(0, P.shape[0], b):
            p = P[i:i + b].T[:, :, None]
            r = (model(p, x[None, :]) - d[None, :])*w[None, :]
            out[i:i + b] = np.einsum('ij,ij->i', r, r)
        return out
    return chi


def population(mc3, f, sampler, nchains, nzchain, seed, func=None, indparams=None, **kw):
    from mc3_b200.engine import Population
    func = func if func is not None else mc3.models.BUILTIN[f['func']]
    return Population(f['data'], f['uncert'], func, f['params'],
                      indparams if indparams is not None else [f['x']], {},
                      f['pstep'], f['pmin'], f['pmax'], f['prior'], f['priorlow'], f['priorup'],
                      nchains=nchains, sampler=sampler, fepsilon=kw.pop('fepsilon', 0.01), hsize=10,
                      thinning=kw.pop('thinning', 1), nzchain=nzchain, seed=seed, **kw)


def spec_of(pop, f, sampler, fepsilon=0.01):
    return ls.Spec(f['params'], f['pstep'], f['pmin'], f['pmax'], f['prior'], f['priorlow'], f['priorup'],
                   sampler, 1.0, fepsilon, pop.seed)


# ---------------------------------------------------------------------------
# the check
# ---------------------------------------------------------------------------
def _first(mask, g, what, detail=lambda c: ''):
    if np.any(mask):
        c = int(np.flatnonzero(mask)[0])
        raise AssertionError(f'generation {g}, chain {c}: {what} disagrees ({int(np.sum(mask))} chains) '
                             f'{detail(c)}')


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def history_states(pop, G):
    """(X_g, cur_g) for g = 0 .. G and zsize_g for g < G from a thinning = 1 history."""
    n, M0 = pop.nchains, pop.M0
    Z = pop.Z.cpu().numpy()
    lp = pop.log_post.cpu().numpy()
    zc = pop.zchain.cpu().numpy()
    for g in range(G):
        got = zc[M0 + g*n:M0 + (g + 1)*n]
        _first(got != np.arange(n), g, 'zchain', lambda c: f'(row holds chain {got[c]})')
    Xs = [Z[:n]] + [Z[M0 + g*n:M0 + (g + 1)*n] for g in range(G)]
    curs = [-2.0*lp[:n]] + [-2.0*lp[M0 + g*n:M0 + (g + 1)*n] for g in range(G)]
    return Xs, curs, [M0 + g*n for g in range(G)]


def walk(pop, spec, chisq, G, states=None, f32=False, last=True):
    """Check generations 0 .. G-1 of `pop` against the restatement; returns counts.
    states: (Xs, curs, zsizes) when the history does not hold the trajectory."""
    torch.cuda.synchronize()
    n, nfree = pop.nchains, pop.nfree
    Xs, curs, zs = states if states is not None else history_states(pop, G)
    Z = pop.Z.cpu().numpy()
    rtol, mrel = (1e-5, 1e-5) if f32 else (1e-10, 1e-9)
    st = ls.State(Xs[0], curs[0], nfree)
    lo, hi = spec.pmin[spec.ifree], spec.pmax[spec.ifree]
    cnt = dict(steps=0, inb=0, marginal_bound=0, marginal_decision=0, accepted=0)
    for g in range(G):
        X, cur, Xn, curn = Xs[g], curs[g], Xs[g + 1], curs[g + 1]
        dr = ls.chain_draws(spec.seed, spec.sampler, n, g, zs[g])
        nrm = ls.chain_normals(spec.seed, n, g, spec.pstep, spec.ifree)
        pr = ls.propose(spec, X, Z[:zs[g]], dr, nrm)
        v = pr['nextp'][:, spec.ifree]
        tol = 4*EPS*(np.abs(pr['x']) + np.abs(pr['jump']))
        mb = np.any((np.abs(v - lo) <= tol) | (np.abs(v - hi) <= tol), axis=1)
        inb = pr['inb']
        data = np.full(n, np.nan)
        if np.any(inb):
            data[inb] = chisq(pr['nextp'][inb])
        nxt = data + ls.prior_terms(spec, pr['nextp'])
        with np.errstate(invalid='ignore'):
            md = inb & ~mb & (np.abs(ls.log_margin(cur, nxt, pr['mrfactor'], dr['u']))
                              < mrel*np.maximum(np.maximum(cur, nxt), 1.0))
        ref = inb & ls.decide(cur, nxt, pr['mrfactor'], dr['u'])
        rej = np.all(_bits(Xn) == _bits(X), axis=1) & (_bits(curn) == _bits(cur))
        acc = ~rej
        # a proposal equal to the chain's row (a snooker jump between two equal history rows)
        # leaves the same history whether it is accepted or not: take the restatement's
        # decision there, which the per-chain acceptance counts check after the walk
        same = np.all(_bits(v) == _bits(X), axis=1)
        acc[same] = ref[same]
        _first(~mb & ~md & (acc != ref), g, 'accept/reject',
               lambda c: f'(device {"accepted" if acc[c] else "rejected"}, in bounds {inb[c]}, cur {cur[c]!r}, '
                         f'numpy nxt {nxt[c]!r}, mrfactor {pr["mrfactor"][c]!r}, u {dr["u"][c]!r})')
        rowok = np.all(np.where(pr['exact'][:, None], _bits(Xn) == _bits(v), np.abs(Xn - v) <= tol), axis=1)
        _first(acc & ~rowok, g, 'accepted row vs proposal',
               lambda c: f'(device {Xn[c].tolist()}, numpy {v[c].tolist()})')
        with np.errstate(invalid='ignore'):
            lpok = np.abs(curn - nxt) <= rtol*np.abs(nxt)
        _first(acc & inb & ~lpok, g, '-2 log_post vs chi-squared + prior',
               lambda c: f'(device {curn[c]!r}, numpy {nxt[c]!r})')
        st.naccept[acc] += 1
        st.outbounds += pr['out'].sum(axis=0)
        nb = acc & (curn < st.best_chisq)
        st.best_chisq[nb], st.best_gen[nb], st.best_x[nb] = curn[nb], g, Xn[nb]
        cnt['steps'] += n
        cnt['inb'] += int(inb.sum())
        cnt['accepted'] += int(acc.sum())
        cnt['marginal_bound'] += int(mb.sum())
        cnt['marginal_decision'] += int(md.sum())
    # counters after the walk
    g = G - 1
    _first(pop.naccept.cpu().numpy() != st.naccept, g, 'naccept (cumulative)')
    ob = pop.outbounds.cpu().numpy()
    assert np.all(np.abs(ob - st.outbounds) <= cnt['marginal_bound']), \
        f'outbounds per free parameter: device {ob.tolist()}, numpy {st.outbounds.tolist()}'
    if cnt['marginal_bound'] == 0:
        assert np.array_equal(ob, st.outbounds), (ob, st.outbounds)
    bc = pop.best_chisq.cpu().numpy()
    _first(_bits(bc) != _bits(st.best_chisq), g, 'best_chisq', lambda c: f'({bc[c]!r} vs {st.best_chisq[c]!r})')
    bg = pop.best_gen.cpu().numpy()
    _first(np.isfinite(st.best_chisq) & (bg != st.best_gen), g, 'best_gen', lambda c: f'({bg[c]} vs {st.best_gen[c]})')
    bx = pop.best_x.cpu().numpy()
    _first(np.isfinite(st.best_chisq) & np.any(_bits(bx) != _bits(st.best_x), axis=1), g, 'best_x')
    cc = pop.counters()
    assert cc['numaccept'] == int(st.naccept.sum())
    assert np.array_equal(cc['outbounds'], ob)
    best, bestp = -2.0*pop.best_log_post0, np.copy(pop.bestp0)
    o = np.lexsort((np.arange(n), st.best_gen, st.best_chisq))[0]
    if st.best_chisq[o] < best:
        best, bestp[spec.ifree] = st.best_chisq[o], st.best_x[o]
        for q in np.where(spec.pstep < 0)[0]:
            bestp[q] = bestp[-int(spec.pstep[q]) - 1]
    assert _bits(cc['best_log_post']) == _bits(-0.5*best), (cc['best_log_post'], -0.5*best)
    assert np.array_equal(_bits(cc['bestp']), _bits(bestp)), (cc['bestp'], bestp)
    if last:                                       # the last generation's internals
        u = pop.u.cpu().numpy()
        _first(_bits(u) != _bits(dr['u']), g, 'u', lambda c: f'({u[c]!r} vs {dr["u"][c]!r})')
        ib = pop.inb.cpu().numpy() != 0
        _first(~mb & (ib != inb), g, 'inb')
        npd = pop.nextp.cpu().numpy()
        tolf = np.zeros_like(npd)
        tolf[:, spec.ifree] = tol
        for q in np.where(spec.pstep < 0)[0]:
            tolf[:, q] = tolf[:, -int(spec.pstep[q]) - 1]
        exact = pr['exact'][:, None] | (tolf == 0)
        okp = np.where(exact, _bits(npd) == _bits(pr['nextp']), np.abs(npd - pr['nextp']) <= tolf)
        _first(~np.all(okp, axis=1), g, 'nextp', lambda c: f'({npd[c].tolist()} vs {pr["nextp"][c].tolist()})')
        mr = pop.mrfactor.cpu().numpy()
        with np.errstate(invalid='ignore'):
            okm = (mr == pr['mrfactor']) | (np.abs(mr - pr['mrfactor']) <= 8*EPS*np.abs(pr['mrfactor']))
        _first(ib & ~mb & ~okm, g, 'mrfactor', lambda c: f'({mr[c]!r} vs {pr["mrfactor"][c]!r})')
    cap = 0.05 if f32 else 1e-3
    assert cnt['marginal_decision'] <= cap*cnt['steps'], cnt
    print(f'lockstep: {spec.sampler} {G} generations x {n} chains: {cnt}')
    return cnt


def run_and_walk(pop, spec, chisq, G, f32=False, use_graph=None):
    pop.init_population('normal')
    pop.run(G, use_graph=use_graph)
    assert pop.gen == G
    return walk(pop, spec, chisq, G, f32=f32)


SINE = lambda p, x: om.sinusoid(p, x)           # noqa: E731


# ---------------------------------------------------------------------------
# the spectral form through block graphs, and the benchmark's own workload
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('sampler', ['demc', 'snooker', 'mrw'])
def test_spectral_generations(mc3, sampler):
    f = sine_fit(20000)
    G = 33                                        # one eager warm-up + a block graph of 32
    pop = population(mc3, f, sampler, 512, G, seed=41)
    assert pop.spectral is not None and pop.fused and not pop.small
    cnt = run_and_walk(pop, spec_of(pop, f, sampler), data_chisq_fn(f, SINE), G)
    assert pop._block == 32 and pop._block_graph is not None
    assert cnt['steps'] - cnt['inb'] > 0           # the bounds are hit


def test_benchmark_workload(mc3):
    from mc3_b200 import workloads
    w = workloads.config2()
    from mc3_b200.engine import Population
    pop = Population(w['data'], w['uncert'], mc3.models.sinusoid, w['params'], [w['x']], {}, w['pstep'],
                     w['pmin'], w['pmax'], w['prior'], w['priorlow'], w['priorup'], nchains=4096,
                     sampler='demc', fepsilon=w['fepsilon'], thinning=1, nzchain=3, seed=7)
    spec = ls.Spec(w['params'], w['pstep'], w['pmin'], w['pmax'], w['prior'], w['priorlow'], w['priorup'],
                   'demc', 1.0, w['fepsilon'], 7)
    run_and_walk(pop, spec, data_chisq_fn(w, SINE), 3)


# ---------------------------------------------------------------------------
# the other chi-squared forms and fused epilogues
# ---------------------------------------------------------------------------
def _gapped_x():
    """Constant cadence with three gaps: 9984 points in four runs of whole 128-point tiles."""
    idx = np.concatenate([np.arange(a, a + m) for a, m in ((0, 2560), (3000, 3840), (7500, 1280), (9100, 2304))])
    return idx*1e-3


FORMS = {
    'moment': (dict(MC3B_NO_SPECTRAL=1), 'demc', lambda: sine_fit(10000)),
    'pair': (dict(MC3B_NO_MOMENT=1), 'snooker', lambda: sine_fit(10000)),
    'unfused': (dict(MC3B_NO_FUSE=1), 'mrw', lambda: sine_fit(10000)),
    'per_point_sigma': ({}, 'demc',
                        lambda: sine_fit(10000, uncert=np.random.RandomState(5).uniform(0.4, 0.6, 10000))),
    'gapped': ({}, 'snooker', lambda: sine_fit(9984, x=_gapped_x())),
}


@pytest.mark.parametrize('form', sorted(FORMS))
def test_chisq_forms(mc3, form):
    envs, sampler, make = FORMS[form]
    f = make()
    with env(**envs):
        pop = population(mc3, f, sampler, 256, 12, seed=43)
    if form == 'moment':
        assert pop.use_moment and pop.spectral is None
    elif form == 'pair':
        assert pop.d_fold is not None and not pop.use_moment
    elif form == 'unfused':
        assert not pop.fused
    elif form == 'per_point_sigma':
        assert pop.grid and pop.d_fold is None
    else:
        assert pop.seg is not None and pop.use_moment
    run_and_walk(pop, spec_of(pop, f, sampler), data_chisq_fn(f, SINE), 12)


def test_guard_reevaluates_inside_fused_generations(mc3):
    """Signal-to-noise 3000: the initial population starts far enough off in the offset
    that the host's start-of-run estimate keeps the moment / spectral form, and as the
    chains close in, the expansion is no longer accurate enough for the best of them:
    the fused epilogue sends those to the exact evaluation inside the generation."""
    f = sine_fit(10000, sigma=1.0/3000.0)
    f['params'] = np.array([1.0, 2.5, 1.0, 5.06, -0.2])
    f['pstep'] = np.array([1e-4, 1e-6, -1.0, 5e-3, 0.0])
    f['pmin'], f['pmax'] = np.array([0.99, 2.3, -np.pi, 4.99, -1.0]), np.array([1.03, 2.7, np.pi, 5.08, 1.0])
    G = 40
    pop = population(mc3, f, 'mrw', 256, G, seed=44)
    assert pop.use_moment
    pop.init_population('normal')
    h0 = int(pop.guard_hits.item())
    pop.run(G)
    torch.cuda.synchronize()
    assert pop.use_moment and pop.gen == G
    assert int(pop.guard_hits.item()) > h0
    walk(pop, spec_of(pop, f, 'mrw'), data_chisq_fn(f, SINE), G)


def test_generic_model_kernel_multi_split(mc3):
    f = poly_fit(50000)
    pop = population(mc3, f, 'demc', 2048, 9, seed=45)
    assert not pop.grid and pop._plan(pop.nlocal) > 1
    run_and_walk(pop, spec_of(pop, f, 'demc'), data_chisq_fn(f, om.polynomial), 9)


# ---------------------------------------------------------------------------
# other models and paths
# ---------------------------------------------------------------------------
CUDA_SINE = '''
__device__ void prepare(real* p) { p[6] = p[5] / p[1]; }
__device__ real model(real x, const real* p) { return p[0] * sin(p[6] * x + p[2]) + p[3] + p[4] * x; }
'''


def test_cuda_model_with_constants(mc3):
    f = sine_fit(8192)
    m = mc3.CudaModel(CUDA_SINE, nparams=5, name='sine_k', nconst=1, nwork=1)
    pop = population(mc3, f, 'snooker', 256, 10, seed=46, func=m, indparams=[f['x'], 2.0*np.pi])
    assert pop.kind == 'cuda' and pop.fused

    def model(p, x):
        return p[0]*np.sin((2.0*np.pi/p[1])*x + p[2]) + p[3] + p[4]*x
    run_and_walk(pop, spec_of(pop, f, 'snooker'), data_chisq_fn(f, model), 10)


def test_fp32_chisq(mc3):
    f = sine_fit(4096)
    pop = population(mc3, f, 'demc', 256, 10, seed=47, dtype='f32')
    run_and_walk(pop, spec_of(pop, f, 'demc'), data_chisq_fn(f, SINE), 10, f32=True)


def test_wavelet_likelihood(mc3):
    rs = np.random.RandomState(8)
    n = 1024
    x = np.linspace(-0.5, 0.5, n)
    data = om.box([0.01, 0.0, 0.1, 1.0], x) + rs.normal(0, 1e-3, n)
    f = dict(data=data, uncert=np.full(n, 1e-3), x=x, func='box',
             params=np.array([0.0101, 0.001, 0.1003, 1.0, 1.0, 5e-4, 1e-3]),
             pstep=np.array([2e-4, 1e-3, 1e-3, 1e-4, 0.0, 1e-4, -6.0]),
             pmin=np.array([0.0095, -0.2, 0.01, 0.9, 0.0, 1e-5, 1e-5]),
             pmax=np.array([0.0105, 0.2, 0.3, 1.1, 2.0, 1e-2, 1e-2]),
             prior=np.array([0.01, 0.0, 0.1, 0.0, 0.0, 4e-4, 0.0]),
             priorlow=np.array([1e-3, 0.0, 0.02, 0.0, 0.0, 1e-4, 0.0]),
             priorup=np.array([2e-3, 0.0, 0.01, 0.0, 0.0, 3e-4, 0.0]))
    pop = population(mc3, f, 'demc', 128, 10, seed=48, wlike=True, fepsilon=0.0)

    def chi(P):
        return np.array([ok.dwt_chisq(om.box(p[:-3], x), data, p) for p in P])
    run_and_walk(pop, spec_of(pop, f, 'demc', 0.0), chi, 10)


def test_torch_model(mc3):
    f = poly_fit(3000)

    def tpoly(P, x):
        y = torch.zeros((P.shape[0], x.shape[0]), dtype=P.dtype, device=P.device)
        for k in range(P.shape[1] - 1, -1, -1):
            y = y*x[None, :] + P[:, k:k + 1]
        return y
    pop = population(mc3, f, 'mrw', 64, 8, seed=49, func=mc3.TorchModel(tpoly))
    assert pop.kind == 'torch'
    run_and_walk(pop, spec_of(pop, f, 'mrw'), data_chisq_fn(f, om.polynomial), 8)


@pytest.mark.parametrize('sampler', ['demc', 'snooker', 'mrw'])
def test_persistent_small_kernel(mc3, sampler):
    f = sine_fit(2000)
    pop = population(mc3, f, sampler, 48, 60, seed=50)
    assert pop.small
    run_and_walk(pop, spec_of(pop, f, sampler), data_chisq_fn(f, SINE), 60, use_graph=True)


# ---------------------------------------------------------------------------
# thinning and the initial population
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('sampler', ['demc', 'mrw'])
def test_thinning_keeps_every_third_generation(mc3, sampler):
    """Draws depend on (seed, chain, generation) only: with thinning 3 the history is
    every third generation of the thinning-1 run, byte for byte."""
    f = sine_fit(10000)
    a = population(mc3, f, sampler, 256, 12, seed=51)
    b = population(mc3, f, sampler, 256, 4, seed=51, thinning=3)
    for p in (a, b):
        p.init_population('normal')
        p.run(12)
    torch.cuda.synchronize()
    M0, n = a.M0, a.nchains
    for k in range(4):
        ra, rb = slice(M0 + (3*k + 2)*n, M0 + (3*k + 3)*n), slice(M0 + k*n, M0 + (k + 1)*n)
        assert torch.equal(a.Z[ra], b.Z[rb]), k
        assert torch.equal(a.log_post[ra], b.log_post[rb]), k
        assert torch.equal(a.zchain[ra], b.zchain[rb]), k
    assert torch.equal(a.naccept, b.naccept) and torch.equal(a.outbounds, b.outbounds)
    walk(a, spec_of(a, f, sampler), data_chisq_fn(f, SINE), 12)


def test_snooker_thinning_from_snapshots(mc3):
    """Snooker's zsize depends on the thinning: eager generations, each checked from
    the device's population and chi-squared before and after it."""
    f = sine_fit(10000)
    G = 9
    pop = population(mc3, f, 'snooker', 256, 3, seed=52, thinning=3)
    pop.init_population('normal')
    Xs, curs = [pop.X.cpu().numpy().copy()], [pop.chisq_cur.cpu().numpy().copy()]
    for _ in range(G):
        pop.run(1, use_graph=False)
        Xs.append(pop.X.cpu().numpy().copy())
        curs.append(pop.chisq_cur.cpu().numpy().copy())
    zs = [ls.zsize(pop.M0, pop.nchains, 3, g) for g in range(G)]
    walk(pop, spec_of(pop, f, 'snooker'), data_chisq_fn(f, SINE), G, states=(Xs, curs, zs))
    # the rows written at generations 2, 5, 8 are the chains' states after them
    Z = pop.Z.cpu().numpy()
    for k in range(3):
        r0 = ls.zrow0(pop.M0, pop.nchains, 3, 3*k + 2)
        assert np.array_equal(Z[r0:r0 + pop.nchains], Xs[3*k + 3]), k


@pytest.mark.parametrize('kickoff', ['normal', 'uniform'])
def test_initial_population(mc3, kickoff):
    f = sine_fit(4096)
    pop = population(mc3, f, 'demc', 256, 1, seed=53)
    spec = spec_of(pop, f, 'demc')
    pop.init_population(kickoff)
    torch.cuda.synchronize()
    chi = data_chisq_fn(f, SINE)
    rows, lps, picks = ls.init_population(spec, kickoff, pop.M0, lambda P: chi(P) + ls.prior_terms(spec, P))
    got = pop.Z[:pop.M0].cpu().numpy()
    base = (spec.params0 if kickoff == 'normal' else spec.pmin)[spec.ifree]
    tol = 4*EPS*(np.abs(base) + np.abs(rows - base))
    bad = np.any(np.abs(got - rows) > tol, axis=1)
    assert not bad.any(), f'initial row {int(np.flatnonzero(bad)[0])} (trial {picks[int(np.flatnonzero(bad)[0])]})'
    np.testing.assert_allclose(pop.log_post[:pop.M0].cpu().numpy(), lps, rtol=1e-10)
