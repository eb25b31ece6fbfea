"""sample_batch with a CudaModel on the GPU.

  built-in      CudaModel(HORNER3) against mc3.models.polynomial on the same batch of 5
                problems of different lengths and seeds: the state after k_init_batch and
                k_run_batch and the output dictionaries' posterior, bestp and best_model are
                bit-equal, for every sampler and thinning 1 and 3.  test_gpu_batch.py ties
                the built-in batch to k_run_small and oracle/lockstep.py.
  oracle        a 3-input systematics transit on a per-problem period constant with a
                prepare work slot: the initial population against ls.init_population, every
                problem's generations chain by chain against oracle/lockstep.py (walk of
                test_gpu_lockstep.py) with a numpy chi-squared on the problem's own constants,
                and problem 2 alone in a batch of one gives the bytes it has in the batch.
  outputs       best_model equals the model at bestp; the key set is sample()'s.
  statistics    32 two-input linear problems against their analytic Gaussian posteriors.
  errors        a problem whose model is NaN everywhere is named.
"""
import numpy as np
import pytest
import torch

from oracle import lockstep as ls
from test_gpu_lockstep import walk

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
SIZES = (100, 257, 1000, 2000, 4096)
HORNER3 = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
# p[8]: the period (a constant), p[9]: 1/period (prepare)
SYSTRANSIT_P = '''__device__ void prepare(real* p) { p[9] = 1 / p[8]; }
__device__ real model(real t, real xc, real yc, const real* p) {
    real dt = t - p[1];
    dt -= p[8] * rint(dt * p[9]);
    real z = fabs(dt) / p[2];
    real transit = p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
    return transit * (1 + p[5]*xc + p[6]*yc + p[7]*xc*yc);
}'''
BATCH_KEYS = ('Z', 'log_post', 'zchain', 'naccept', 'outbounds', 'best_chisq', 'best_x', 'best_gen')


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int64) if a.dtype == torch.float64 else a,
                       b.contiguous().view(torch.int64) if b.dtype == torch.float64 else b)


def batch(mc3, f, func, sampler, nchains, nsamples, seed, state=True, **kw):
    return mc3.sample_batch(f['data'], f['uncert'], func, f['params'], f['indparams'], pmin=f['pmin'],
                            pmax=f['pmax'], pstep=f['pstep'], prior=f.get('prior'), priorlow=f.get('priorlow'),
                            priorup=f.get('priorup'), sampler=sampler, nchains=nchains, nsamples=nsamples,
                            seed=seed, _state=state, fepsilon=kw.pop('fepsilon', 0.01), **kw)


# ---------------------------------------------------------------------------
# bit identity with the built-in batch
# ---------------------------------------------------------------------------
def quadratic_batch():
    """Quadratics of different truths, noise and lengths; a two-sided prior on the offset."""
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


@pytest.mark.parametrize('thinning', [1, 3])
@pytest.mark.parametrize('sampler', ['demc', 'snooker', 'mrw'])
def test_equals_the_builtin_batch(mc3, sampler, thinning):
    f = quadratic_batch()
    um = mc3.CudaModel(HORNER3, 3, name='horner')
    n, nz, seeds = 24, 20, [11, 5, 97, 3, 40]
    runs = [batch(mc3, f, func, sampler, n, n*nz*thinning, seeds, thinning=thinning)
            for func in (mc3.models.polynomial, um)]
    torch.cuda.synchronize()
    for run in runs:
        assert run.status.cpu().numpy().tolist() == [0]*5
    for name in BATCH_KEYS + ('X', 'chisq_cur', 'nextp', 'u', 'mrfactor', 'inb'):
        assert _bits_equal(getattr(runs[0], name), getattr(runs[1], name)), name
    outs = [batch(mc3, f, func, sampler, n, n*nz*thinning, seeds, state=False, thinning=thinning, burnin=5)
            for func in (mc3.models.polynomial, um)]
    for b in range(5):
        for k in ('posterior', 'bestp', 'best_model', 'log_post', 'zchain', 'best_log_post'):
            assert np.array_equal(outs[0][b][k], outs[1][b][k]), (b, k)


# ---------------------------------------------------------------------------
# inputs, constants and prepare against the oracle
# ---------------------------------------------------------------------------
PERIODS = np.array([3.1, 2.7, 4.05, 3.55, 2.2])


def np_systransit(p, t, xc, yc, period):
    """SYSTRANSIT_P in numpy, p [npars, ...] broadcasting against the points."""
    dt = t - p[1]
    dt = dt - period*np.rint(dt*(1.0/period))
    z = np.abs(dt)/p[2]
    tr = p[3] - p[0]*np.where(z < 1, 1.0, np.where(z < p[4], (p[4] - z)/(p[4] - 1), 0.0))
    return tr*(1 + p[5]*xc + p[6]*yc + p[7]*xc*yc)


def systransit_batch(sizes=(300, 512, 777, 1000, 640)):
    rs = np.random.RandomState(5)
    B = len(sizes)
    truth = np.array([[0.01 + 0.001*b, 0.3 + 0.05*b, 0.08, 1.0, 1.4, 0.01, -0.02, 0.005] for b in range(B)])
    data, unc, ind = [], [], []
    for b, n in enumerate(sizes):
        t = np.sort(rs.uniform(0.0, 3*PERIODS[b], n))
        xc, yc = rs.normal(0, 0.3, n), rs.normal(0, 0.3, n)
        u = np.full(n, 5e-4)
        data.append(np_systransit(truth[b], t, xc, yc, PERIODS[b]) + rs.normal(0, 1, n)*u)
        unc.append(u)
        ind.append([t, xc, yc, PERIODS[b]])
    return dict(data=data, uncert=unc, indparams=ind, params=truth*np.array([1.02, 1.0, 1.01, 1.0, 1.0, 1, 1, 1]),
                pstep=np.array([5e-4, 2e-3, 1e-3, 1e-4, 0.0, 1e-3, 1e-3, 1e-3]),
                pmin=truth - np.array([0.005, 0.05, 0.03, 0.01, 0.0, 0.05, 0.05, 0.05]),
                pmax=truth + np.array([0.005, 0.05, 0.03, 0.01, 0.0, 0.05, 0.05, 0.05]))


def chisq_of(f, b):
    t, xc, yc, period = f['indparams'][b]
    d, w = f['data'][b], 1.0/f['uncert'][b]

    def chi(P):
        r = (np_systransit(P.T[:, :, None], t[None, :], xc[None, :], yc[None, :], period) - d[None, :])*w[None, :]
        return np.einsum('ij,ij->i', r, r)
    return chi


class _Problem:
    """Problem b of a batch run with the attributes walk() reads of a Population; the
    counters come from the batch's own output dictionary."""

    def __init__(self, run, b, out, ifree, params):
        for name in BATCH_KEYS + ('u', 'inb', 'nextp', 'mrfactor'):
            setattr(self, name, getattr(run, name)[b])
        self.nchains, self.nfree, self.M0 = run.nchains, run.nfree, run.M0
        lp0 = run.log_post[b, :run.M0].cpu().numpy()
        i0 = int(np.argmax(lp0))
        self.best_log_post0 = lp0[i0]
        self.bestp0 = np.array(params, dtype=float)
        self.bestp0[ifree] = run.Z[b, i0].cpu().numpy()
        self.out = out

    def counters(self):
        return dict(numaccept=int(self.naccept.sum()), outbounds=self.outbounds.cpu().numpy(),
                    best_log_post=self.out['best_log_post'], bestp=self.out['bestp'])


@pytest.mark.parametrize('sampler', ['demc', 'snooker', 'mrw'])
def test_inputs_constants_and_prepare_against_the_oracle(mc3, sampler):
    f = systransit_batch()
    m = mc3.CudaModel(SYSTRANSIT_P, 8, name='systransit_p', ninputs=3, nconst=1, nwork=1)
    n, G, seeds = 16, 12, [31, 32, 33, 34, 35]
    run = batch(mc3, f, m, sampler, n, n*G, seeds)
    outs = batch(mc3, f, m, sampler, n, n*G, seeds, state=False)
    torch.cuda.synchronize()
    assert run.status.cpu().numpy().tolist() == [0]*5
    M0 = run.M0
    for b in range(5):
        spec = ls.Spec(f['params'][b], f['pstep'], f['pmin'][b], f['pmax'][b], None, None, None, sampler, 1.0,
                       0.01, seeds[b])
        chi = chisq_of(f, b)
        rows, lps, _ = ls.init_population(spec, 'normal', M0, chi)
        got = run.Z[b, :M0].cpu().numpy()
        base = spec.params0[spec.ifree]
        tol = 4*EPS*(np.abs(base) + np.abs(rows - base))
        assert not np.any(np.abs(got - rows) > tol), f'problem {b}'
        np.testing.assert_allclose(run.log_post[b, :M0].cpu().numpy(), lps, rtol=1e-10)
        walk(_Problem(run, b, outs[b], spec.ifree, f['params'][b]), spec, chi, G)
    # problem 2 alone in a batch of one: the same bytes (no constants or inputs leak between CTAs)
    g = {k: ([v[2]] if isinstance(v, list) else v[2:3] if np.ndim(v) == 2 else v) for k, v in f.items()}
    one = batch(mc3, g, m, sampler, n, n*G, [seeds[2]])
    torch.cuda.synchronize()
    for name in BATCH_KEYS:
        assert _bits_equal(getattr(one, name)[0], getattr(run, name)[2]), name


# ---------------------------------------------------------------------------
# output dictionaries
# ---------------------------------------------------------------------------
def test_outputs(mc3, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)                          # sample() writes its statistics file
    f = systransit_batch()
    m = mc3.CudaModel(SYSTRANSIT_P, 8, name='systransit_p', ninputs=3, nconst=1, nwork=1)
    n, seed = 16, 7
    outs = batch(mc3, f, m, 'demc', n, n*300, seed, state=False, burnin=50)
    assert len(outs) == 5
    for b, out in enumerate(outs):
        want = m(out['bestp'], *f['indparams'][b])
        np.testing.assert_allclose(out['best_model'], want, rtol=1e-12, atol=1e-12, err_msg=f'problem {b}')
        assert out['best_log_post'] >= out['log_post'].max() - 1e-9
    ref = mc3.sample(f['data'][0], f['uncert'][0], func=m, params=f['params'][0], indparams=f['indparams'][0],
                     pmin=f['pmin'][0], pmax=f['pmax'][0], pstep=f['pstep'], sampler='demc', nchains=n,
                     nsamples=n*300, burnin=50, seed=seed, log=mc3.Log(verb=-1))
    assert set(outs[0]) == set(ref)


# ---------------------------------------------------------------------------
# statistics
# ---------------------------------------------------------------------------
def test_two_input_line_posteriors(mc3):
    """32 planes y = a + b x1 + c x2: the posterior is Gaussian with covariance (A^T W A)^-1
    and mean at the weighted least-squares solution."""
    B, n = 32, 200
    rs = np.random.RandomState(4)
    truth = np.stack([rs.uniform(-2, 2, B), rs.uniform(-1, 1, B), rs.uniform(-1, 1, B)], axis=1)
    sig = rs.uniform(0.05, 0.5, B)
    x1 = [rs.uniform(-1, 1, n) for _ in range(B)]
    x2 = [rs.uniform(-1, 1, n) for _ in range(B)]
    data = [truth[b, 0] + truth[b, 1]*x1[b] + truth[b, 2]*x2[b] + rs.normal(0, sig[b], n) for b in range(B)]
    plane = mc3.CudaModel('__device__ real model(real x1, real x2, const real* p) '
                          '{ return p[0] + p[1] * x1 + p[2] * x2; }', 3, name='plane', ninputs=2)
    outs = mc3.sample_batch(data, [np.full(n, s) for s in sig], plane, truth, [[x1[b], x2[b]] for b in range(B)],
                            pstep=np.array([0.02, 0.02, 0.02]), sampler='snooker', nchains=16,
                            nsamples=16*4000, burnin=500, seed=100)
    z = []
    for b, out in enumerate(outs):
        A = np.stack([np.ones(n), x1[b], x2[b]], axis=1)
        cov = np.linalg.inv(A.T @ A)*sig[b]**2
        mu = cov @ (A.T @ data[b])/sig[b]**2
        sd = np.sqrt(np.diag(cov))
        post = out['posterior'][out['zmask']]
        neff = post.shape[0]/50.0                         # a conservative autocorrelation allowance
        z.append((post.mean(0) - mu)/(sd/np.sqrt(neff)))
        np.testing.assert_allclose(post.std(0), sd, rtol=0.15)
    z = np.array(z)
    assert np.all(np.abs(z) < 5), np.abs(z).max()
    assert abs(z.mean()) < 5/np.sqrt(z.size) + 0.3 and np.sqrt(np.mean(z**2)) < 2.0


# ---------------------------------------------------------------------------
# errors
# ---------------------------------------------------------------------------
def test_unpopulated_problem_is_named(mc3):
    """The constant p[2] is a scale; problem 3's is negative, so its model is NaN everywhere."""
    m = mc3.CudaModel('__device__ real model(real x, const real* p) { return (p[0] + p[1] * x) * sqrt(p[2]); }',
                      2, name='scaled_line', nconst=1)
    B, n = 5, 100
    x = np.linspace(0, 1, n)
    data = [1.0 + x for _ in range(B)]
    with pytest.raises(ValueError, match=r'^problem 3: Cannot populate an initial sample set of parameters'):
        mc3.sample_batch(data, [np.full(n, 0.1)]*B, m, np.array([[1.0, 1.0]]*B),
                         [[x, -1.0 if b == 3 else 1.0] for b in range(B)], pstep=np.array([0.01, 0.01]),
                         sampler='demc', nchains=8, nsamples=80, seed=1)
