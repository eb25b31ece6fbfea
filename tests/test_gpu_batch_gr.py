"""sample_batch's Gelman-Rubin test and early stop on the GPU, for mrw, demc and snooker at
thinning 1 and 3.

  parity        every evaluated row of the PSRF table equals mc3b_gelman_rubin on the problem's
                history cut at that report, bit for bit; reports at or before burn-in stay NaN.
  no effects    the test at every report, with a threshold never met, leaves histories,
                counters and bests bit-equal to a run without it.
  stop points   with a threshold taken from that table, each problem stops at the first report
                the rule selects; its rows up to there equal the unstopped run's, later rows
                are untouched, counters and bests equal a run of that many samples.
  sample()      one problem stops where sample() stops, with the same posterior rows.
  CudaModel     CudaModel(HORNER3) stops where the built-in polynomial stops.
  outputs       row counts, acceptance rate, zmask, statistics and the 'psrf' key of stopped
                and unstopped problems.
"""
import numpy as np
import pytest
import torch

from oracle import models as om

pytestmark = pytest.mark.gpu
SIZES = (100, 257, 1000, 2000, 4096)
N, NZ, ZB, GRNMIN = 12, 60, 20, 0.3          # chains, thinned steps, burned thinned steps, grnmin
HORNER3 = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
STATE = ('Z', 'log_post', 'zchain', 'naccept', 'outbounds', 'best_chisq', 'best_x', 'best_gen')


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def sine_batch():
    """Sinusoids of different truths, noise and lengths, a shared phase and a fixed slope, with
    priors (test_gpu_batch.py's problems)."""
    B = len(SIZES)
    rs = np.random.RandomState(7)
    data, unc, xs = [], [], []
    truth = np.array([[1.0 + 0.05*b, 2.5 + 0.01*b, 1.0 + 0.05*b, 5.0 - 0.02*b, -0.2] for b in range(B)])
    for b, n in enumerate(SIZES):
        x = np.linspace(0.0, 10.0, n) if b % 2 == 0 else np.sort(rs.uniform(0.0, 10.0, n))
        u = np.full(n, 0.3 + 0.1*b)
        data.append(om.sinusoid(truth[b], x) + rs.normal(0.0, 1.0, n)*u)
        unc.append(u)
        xs.append([x])
    params = truth*np.array([1.01, 1.002, 1.01, 1.002, 1.0])
    pmin = np.stack([truth[:, 0] - 0.5, truth[:, 1] - 0.2, -np.pi*np.ones(B), truth[:, 3] - 0.5, -np.ones(B)], 1)
    pmax = np.stack([truth[:, 0] + 0.5, truth[:, 1] + 0.2, np.pi*np.ones(B), truth[:, 3] + 0.5, np.ones(B)], 1)
    return dict(data=data, uncert=unc, indparams=xs, params=params, pmin=pmin, pmax=pmax,
                pstep=np.array([1e-2, 1e-3, -1.0, 1e-2, 0.0]), prior=truth*np.array([1, 1, 1, 1, 0]),
                priorlow=np.array([0.02, 0.1, 0.03, 0.05, 0.0]), priorup=np.array([0.05, 0.2, 0.01, 0.0, 0.0]))


def quadratic_batch():
    rs = np.random.RandomState(11)
    truth = np.array([[1.0 + 0.1*b, -0.5 + 0.05*b, 0.2 - 0.01*b] for b in range(len(SIZES))])
    data, unc, xs = [], [], []
    for b, n in enumerate(SIZES):
        x = np.sort(rs.uniform(-1.0, 2.0, n))
        u = rs.uniform(0.05, 0.15, n)
        data.append(truth[b, 0] + truth[b, 1]*x + truth[b, 2]*x*x + rs.normal(0.0, 1.0, n)*u)
        unc.append(u)
        xs.append([x])
    return dict(data=data, uncert=unc, indparams=xs, params=truth*1.01, pstep=np.array([0.01, 0.01, 0.005]),
                pmin=truth - 0.5, pmax=truth + 0.5, prior=truth, priorlow=np.array([0.05, 0.0, 0.0]),
                priorup=np.array([0.03, 0.0, 0.0]))


def batch(mc3, f, sampler, thinning, func=None, state=True, nz=NZ, seed=(11, 5, 97, 3, 40), **kw):
    return mc3.sample_batch(f['data'], f['uncert'], func or mc3.models.sinusoid, f['params'], f['indparams'],
                            pmin=f['pmin'], pmax=f['pmax'], pstep=f['pstep'], prior=f['prior'],
                            priorlow=f['priorlow'], priorup=f['priorup'], sampler=sampler, nchains=N,
                            nsamples=N*nz*thinning, burnin=ZB*thinning, thinning=thinning, seed=list(seed),
                            fepsilon=0.01, grnmin=GRNMIN, _state=state, **kw)


def _bits_equal(a, b):
    v = lambda t: t.contiguous().view(torch.int64) if t.dtype == torch.float64 else t   # noqa: E731
    return torch.equal(v(a), v(b))


def _reports():
    from mc3_b200.mcmc_driver import report_points
    return report_points(NZ)


def _stops(table, g, M0):
    """(K_b, whether problem b stops): the first report past burn-in where every PSRF < g and the
    history exceeds grnmin, else the last report."""
    from mc3_b200.mcmc_driver import gr_min_size

    class L:
        def error(self, m):
            raise ValueError(m)
    gmin = gr_min_size(GRNMIN, N, NZ, ZB, 1, M0, L())
    ks = _reports()
    K, stop = [], []
    for t in table:
        hit = [k for i, k in enumerate(ks) if k > ZB and np.all(t[i] < g) and M0 + k*N > gmin]
        K.append(hit[0] if hit else NZ)
        stop.append(bool(hit))
    return np.array(K), np.array(stop)


def _threshold(table, M0):
    """A grbreak at which the problems stop at as many different reports as possible."""
    best, bestg = -1, None
    for g in np.unique(np.nextafter(table.max(axis=2), np.inf)):
        if not np.isfinite(g):
            continue
        n = len(set(_stops(table, g, M0)[0].tolist()))
        if n > best:
            best, bestg = n, g
    return bestg


@pytest.fixture(scope='module', params=[(s, t) for s in ('mrw', 'demc', 'snooker') for t in (1, 3)],
                ids=lambda p: f'{p[0]}-thin{p[1]}')
def runs(mc3, request):
    sampler, thinning = request.param
    f = sine_batch()
    plain = batch(mc3, f, sampler, thinning)
    every = batch(mc3, f, sampler, thinning, grtest=True, grbreak=1e-9)
    torch.cuda.synchronize()
    table = every.psrf.cpu().numpy()
    g = _threshold(table, every.M0)
    K, stop = _stops(table, g, every.M0)
    return dict(f=f, sampler=sampler, thinning=thinning, plain=plain, every=every, table=table, g=float(g),
                K=K, stop=stop)


def test_psrf_parity(mc3, runs):
    from mc3_b200 import _lib
    run = runs['every']
    ks = _reports()
    table = run.psrf.cpu().numpy()
    nf, M0 = run.nfree, run.M0
    assert run.status.cpu().numpy().tolist() == [0]*5
    assert run.kstop.cpu().numpy().tolist() == [NZ]*5
    work = torch.empty((2, N, nf), dtype=torch.float64, device=run.dev)
    ref = torch.empty(nf, dtype=torch.float64, device=run.dev)
    assert any(k <= ZB for k in ks) and any(k > ZB for k in ks)
    for b in range(5):
        for i, k in enumerate(ks):
            if k <= ZB:
                assert np.all(np.isnan(table[b, i])), (b, k)
                continue
            _lib.call('mc3b_gelman_rubin', run.Z[b].data_ptr(), nf, N, M0, None, 0, ZB, k - ZB,
                      work.data_ptr(), ref.data_ptr(), _lib.stream_ptr())
            r = ref.cpu().numpy()
            assert np.array_equal(table[b, i].view(np.int64), r.view(np.int64)), (b, k, table[b, i], r)


def test_no_side_effects(runs):
    for name in STATE:
        assert _bits_equal(getattr(runs['every'], name), getattr(runs['plain'], name)), name


def test_stop_points(mc3, runs):
    every, thinning, table, want = runs['every'], runs['thinning'], runs['table'], runs['K']
    M0 = every.M0
    assert len(set(want.tolist())) >= 2, (want, table.max(axis=2))
    run = batch(mc3, runs['f'], runs['sampler'], thinning, grtest=True, grbreak=runs['g'])
    torch.cuda.synchronize()
    K = run.kstop.cpu().numpy()
    assert K.tolist() == want.tolist()
    assert run.status.cpu().numpy().tolist() == [3 if s else 0 for s in runs['stop']]
    got = run.psrf.cpu().numpy()
    ks = _reports()
    for b in range(5):
        end = M0 + K[b]*N
        for name in ('Z', 'log_post', 'zchain'):
            assert _bits_equal(getattr(run, name)[b, :end], getattr(every, name)[b, :end]), (b, name)
        assert bool((run.zchain[b, end:] == -1).all()) and bool((run.Z[b, end:] == 0).all())
        i = ks.index(K[b])
        assert np.array_equal(got[b, :i + 1], table[b, :i + 1], equal_nan=True)
        assert np.all(np.isnan(got[b, i + 1:]))
    for k in np.unique(K):                       # counters and bests of a run of K_b n thinning samples
        short = batch(mc3, runs['f'], runs['sampler'], thinning, nz=int(k))
        torch.cuda.synchronize()
        for b in np.flatnonzero(K == k):
            for name in ('naccept', 'outbounds', 'best_chisq', 'best_x', 'best_gen'):
                assert _bits_equal(getattr(run, name)[b], getattr(short, name)[b]), (b, name)


def test_outputs(mc3, runs, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    f, thinning, K, table = runs['f'], runs['thinning'], runs['K'], runs['table']
    outs = batch(mc3, f, runs['sampler'], thinning, state=False, grtest=True, grbreak=runs['g'])
    ks = _reports()
    plain = batch(mc3, f, runs['sampler'], thinning, state=False)
    assert 'psrf' not in plain[0] and set(outs[0]) == set(plain[0]) | {'psrf'}
    for b, out in enumerate(outs):
        rows = K[b]*N
        for k in ('posterior', 'zchain', 'log_post', 'chisq'):
            assert len(out[k]) == rows, (b, k)
            assert np.array_equal(out[k], plain[b][k][:rows]), (b, k)
        zmask = (np.arange(ZB, K[b])[None, :]*N + np.arange(N)[:, None]).ravel()
        assert np.array_equal(out['zmask'], zmask)
        post = out['posterior'][zmask]
        if len(post) > 20000:
            post = post[np.random.default_rng(314159).choice(len(post), 20000, replace=False)]
        ifree = np.where(f['pstep'] > 0)[0]
        mode, hlo, hhi = mc3.stats.hpd_statistics(post)
        for k, v in (('mode', mode), ('hpd_low_bounds', hlo), ('hpd_high_bounds', hhi)):
            assert np.array_equal(out[k][ifree], v), (b, k)
        want = mc3.stats.calc_sample_statistics(post, out['bestp'], f['pstep'], calc_hpd=True, device=True)
        for k, v in zip(('medianp', 'meanp', 'stdp', 'median_low_bounds', 'median_high_bounds'), want):
            np.testing.assert_allclose(out[k], v, rtol=1e-12, atol=0, err_msg=f'{b} {k}')
        assert np.array_equal(out['psrf'], table[b, ks.index(K[b])])
    # acceptance rates: the counters of a run of K_b n thinning samples
    for k in np.unique(K):
        short = batch(mc3, f, runs['sampler'], thinning, state=False, nz=int(k))
        for b in np.flatnonzero(K == k):
            assert outs[b]['acceptance_rate'] == short[b]['acceptance_rate'], b
            for key in ('bestp', 'best_log_post', 'best_model'):
                assert np.array_equal(outs[b][key], short[b][key]), (b, key)


def _one(f, b):
    vec = lambda k: np.array(f[k][b] if np.ndim(f[k]) == 2 else f[k], dtype=float)    # noqa: E731
    return dict(data=f['data'][b], uncert=f['uncert'][b], indparams=f['indparams'][b], params=f['params'][b],
                **{k: vec(k) for k in ('pstep', 'pmin', 'pmax', 'prior', 'priorlow', 'priorup')})


def test_same_stop_as_sample(mc3, runs, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    f, thinning, K, g = runs['f'], runs['thinning'], runs['K'], runs['g']
    seeds = (11, 5, 97, 3, 40)
    outs = batch(mc3, f, runs['sampler'], thinning, state=False, grtest=True, grbreak=g)
    for b in sorted({int(np.argmin(K)), int(np.argmax(K))}):
        q = _one(f, b)
        ref = mc3.sample(q['data'], q['uncert'], func=mc3.models.sinusoid, params=q['params'],
                         indparams=q['indparams'], pmin=q['pmin'], pmax=q['pmax'], pstep=q['pstep'],
                         prior=q['prior'], priorlow=q['priorlow'], priorup=q['priorup'], sampler=runs['sampler'],
                         nchains=N, nsamples=N*NZ*thinning, burnin=ZB*thinning, thinning=thinning,
                         fepsilon=0.01, grtest=True, grbreak=g, grnmin=GRNMIN, seed=seeds[b],
                         log=mc3.Log(verb=-1))
        assert ref['posterior'].shape == outs[b]['posterior'].shape, (b, K[b])
        assert np.array_equal(ref['posterior'], outs[b]['posterior']), b
        assert np.array_equal(ref['zchain'], outs[b]['zchain']), b


@pytest.mark.parametrize('thinning', [1, 3])
@pytest.mark.parametrize('sampler', ['mrw', 'demc', 'snooker'])
def test_cuda_model_stops_as_the_builtin(mc3, sampler, thinning):
    f = quadratic_batch()
    um = mc3.CudaModel(HORNER3, 3, name='horner')
    every = batch(mc3, f, sampler, thinning, func=mc3.models.polynomial, grtest=True, grbreak=1e-9)
    torch.cuda.synchronize()
    table = every.psrf.cpu().numpy()
    g = _threshold(table, every.M0)
    runs = [batch(mc3, f, sampler, thinning, func=func, grtest=True, grbreak=float(g))
            for func in (mc3.models.polynomial, um)]
    torch.cuda.synchronize()
    K = runs[0].kstop.cpu().numpy()
    assert K.tolist() == _stops(table, g, every.M0)[0].tolist()
    for name in STATE + ('status', 'kstop'):
        assert _bits_equal(getattr(runs[0], name), getattr(runs[1], name)), name
    assert np.array_equal(runs[0].psrf.cpu().numpy(), runs[1].psrf.cpu().numpy(), equal_nan=True)
