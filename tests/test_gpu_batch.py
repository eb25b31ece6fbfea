"""sample_batch on the GPU: every problem of a batch against the one-problem paths.

  trajectories  a batch of 5 problems of different lengths, parameters and seeds, run by
                k_init_batch + k_run_batch, against one Population per problem started from
                the batch's initial state (set_initial) and run by k_run_small: history,
                counters and per-chain bests equal bit for bit.  test_persistent_small_kernel
                (test_gpu_lockstep.py) ties k_run_small to oracle/lockstep.py.
  initial set   Z[0:M0] equals Population.init_population's byte for byte; log_post within
                rtol 1e-10 of oracle/lockstep.py's restatement.
  outputs       key set, history slices, chi-squared column, HPD statistics (bit-equal to
                hpd_statistics on the problem's subsample), medians and bounds, best model.
  statistics    64 straight lines of different truths and noise: posterior means and
                standard deviations against the analytic Gaussian posterior.
"""
import numpy as np
import pytest
import torch

from oracle import lockstep as ls
from oracle import models as om

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
SIZES = (100, 257, 1000, 2000, 4096)


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def sine_batch(sizes=SIZES, tight=None):
    """Sinusoid + line with a shared phase (p2 := p0), a fixed slope, two-sided priors of
    unequal widths, a one-sided prior on the offset and bounds that cut the posterior;
    truths and noise differ between problems.  tight: index of a problem whose amplitude
    bounds hold only a few per cent of the normal trials (several rounds)."""
    B = len(sizes)
    rs = np.random.RandomState(7)
    data, unc, xs = [], [], []
    truth = np.array([[1.0 + 0.05*b, 2.5 + 0.01*b, 1.0 + 0.05*b, 5.0 - 0.02*b, -0.2] for b in range(B)])
    for b, n in enumerate(sizes):
        x = np.linspace(0.0, 10.0, n) if b % 2 == 0 else np.sort(rs.uniform(0.0, 10.0, n))
        u = np.full(n, 0.3 + 0.1*b) if b != 3 else rs.uniform(0.3, 0.6, n)
        data.append(om.sinusoid(truth[b], x) + rs.normal(0.0, 1.0, n)*u)
        unc.append(u)
        xs.append([x])
    params = truth*np.array([1.01, 1.002, 1.01, 1.002, 1.0])
    pmin = np.stack([truth[:, 0] - 0.02, truth[:, 1] - 0.2, -np.pi*np.ones(B), truth[:, 3] - 0.006,
                     -np.ones(B)], axis=1)
    pmax = np.stack([truth[:, 0] + 0.035, truth[:, 1] + 0.2, np.pi*np.ones(B), truth[:, 3] + 0.03,
                     np.ones(B)], axis=1)
    if tight is not None:
        pmin[tight, 0], pmax[tight, 0] = params[tight, 0] - 1e-4, params[tight, 0] + 1e-4
    return dict(data=data, uncert=unc, indparams=xs, params=params,
                pstep=np.array([1e-2, 1e-3, -1.0, 1e-2, 0.0]), pmin=pmin, pmax=pmax,
                prior=truth*np.array([1, 1, 1, 1, 0]), priorlow=np.array([0.02, 0.1, 0.03, 0.05, 0.0]),
                priorup=np.array([0.05, 0.2, 0.01, 0.0, 0.0]))


def problem(f, b):
    """Problem b as sample() hands it to the sampler (no prior terms on fixed or shared parameters)."""
    vec = lambda k: np.array(f[k][b] if np.ndim(f[k]) == 2 else f[k], dtype=float)      # noqa: E731
    q = dict(data=f['data'][b], uncert=f['uncert'][b], x=f['indparams'][b][0], params=f['params'][b],
             **{k: vec(k) for k in ('pstep', 'pmin', 'pmax', 'prior', 'priorlow', 'priorup')})
    q['priorlow'][q['pstep'] <= 0] = q['priorup'][q['pstep'] <= 0] = 0.0
    return q


def population(mc3, q, sampler, nchains, nzchain, seed, thinning=1, fepsilon=0.01):
    from mc3_b200.engine import Population
    return Population(q['data'], q['uncert'], mc3.models.sinusoid, q['params'], [q['x']], {}, q['pstep'],
                      q['pmin'], q['pmax'], q['prior'], q['priorlow'], q['priorup'], nchains=nchains,
                      sampler=sampler, fepsilon=fepsilon, hsize=10, thinning=thinning, nzchain=nzchain,
                      seed=seed)


def batch_state(mc3, f, sampler, nchains, nsamples, seed, **kw):
    from mc3_b200 import batch_driver
    return batch_driver.sample_batch(f['data'], f['uncert'], mc3.models.sinusoid, f['params'], f['indparams'],
                                     pmin=f['pmin'], pmax=f['pmax'], pstep=f['pstep'], prior=f['prior'],
                                     priorlow=f['priorlow'], priorup=f['priorup'], sampler=sampler,
                                     nchains=nchains, nsamples=nsamples, seed=seed, _state=True,
                                     fepsilon=kw.pop('fepsilon', 0.01), **kw)


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int64) if a.dtype == torch.float64 else a,
                       b.contiguous().view(torch.int64) if b.dtype == torch.float64 else b)


# ---------------------------------------------------------------------------
# trajectories
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('thinning', [1, 3])
@pytest.mark.parametrize('sampler', ['demc', 'snooker', 'mrw'])
def test_trajectories_equal_the_small_kernel(mc3, sampler, thinning):
    f = sine_batch()
    n, nz = 24, 20
    run = batch_state(mc3, f, sampler, n, n*nz*thinning, seed=[11, 5, 97, 3, 40], thinning=thinning)
    torch.cuda.synchronize()
    assert run.status.cpu().numpy().tolist() == [0]*5
    seeds = [11, 5, 97, 3, 40]
    for b in range(5):
        pop = population(mc3, problem(f, b), sampler, n, nz, seeds[b], thinning=thinning)
        assert pop.small
        pop.set_initial(run.Z[b, :pop.M0], run.log_post[b, :pop.M0])
        pop.run(nz*thinning, use_graph=True)
        torch.cuda.synchronize()
        for name, mine, ref in (('Z', run.Z[b], pop.Z), ('log_post', run.log_post[b], pop.log_post),
                                ('zchain', run.zchain[b], pop.zchain), ('naccept', run.naccept[b], pop.naccept),
                                ('outbounds', run.outbounds[b], pop.outbounds),
                                ('best_chisq', run.best_chisq[b], pop.best_chisq),
                                ('best_x', run.best_x[b], pop.best_x), ('best_gen', run.best_gen[b], pop.best_gen)):
            assert _bits_equal(mine, ref), f'problem {b}: {name}'
    # problem 2 alone in a batch of one: the same bytes (nothing leaks between CTAs)
    g = {k: ([v[2]] if isinstance(v, list) else v[2:3] if np.ndim(v) == 2 else v) for k, v in f.items()}
    one = batch_state(mc3, g, sampler, n, n*nz*thinning, seed=[97], thinning=thinning)
    torch.cuda.synchronize()
    for name in ('Z', 'log_post', 'zchain', 'naccept', 'outbounds', 'best_chisq', 'best_x', 'best_gen'):
        assert _bits_equal(getattr(one, name)[0], getattr(run, name)[2]), name


# ---------------------------------------------------------------------------
# initial population
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('kickoff', ['normal', 'uniform'])
def test_initial_population(mc3, kickoff):
    f = sine_batch(tight=1 if kickoff == 'normal' else None)
    n, seeds = 32, [21, 22, 23, 24, 25]
    run = batch_state(mc3, f, 'demc', n, n, seed=seeds, kickoff=kickoff)
    torch.cuda.synchronize()
    M0 = 10*n
    for b in range(5):
        q = problem(f, b)
        pop = population(mc3, q, 'demc', n, 1, seeds[b])
        pop.init_population(kickoff)
        torch.cuda.synchronize()
        assert _bits_equal(run.Z[b, :M0], pop.Z[:M0]), f'problem {b}'
        # after the one generation (thinning 1), row M0 + c holds chain c's state and log-posterior
        assert _bits_equal(run.X[b], run.Z[b, M0:M0 + n])
        assert _bits_equal(run.chisq_cur[b], -2.0*run.log_post[b, M0:M0 + n])
        spec = ls.Spec(q['params'], q['pstep'], q['pmin'], q['pmax'], q['prior'], q['priorlow'], q['priorup'],
                       'demc', 1.0, 0.01, seeds[b])

        def chi(P, q=q, spec=spec):
            r = (om.sinusoid(P.T[:, :, None], q['x'][None, :]) - q['data'][None, :])/q['uncert'][None, :]
            return np.einsum('ij,ij->i', r, r) + ls.prior_terms(spec, P)
        rows, lps, picks = ls.init_population(spec, kickoff, M0, chi)
        if b == 1 and kickoff == 'normal':
            assert picks[-1][0] >= 2, 'the tight problem was meant to need several rounds'
        got = run.Z[b, :M0].cpu().numpy()
        base = (spec.params0 if kickoff == 'normal' else spec.pmin)[spec.ifree]
        tol = 4*EPS*(np.abs(base) + np.abs(rows - base))
        assert not np.any(np.abs(got - rows) > tol), f'problem {b}'
        np.testing.assert_allclose(run.log_post[b, :M0].cpu().numpy(), lps, rtol=1e-10)


def test_unpopulated_problem_is_named(mc3):
    f = sine_batch()
    f['pmin'][3, 1], f['pmax'][3, 1] = f['params'][3, 1] - 1e-13, f['params'][3, 1] + 1e-13
    with pytest.raises(ValueError, match=r'^problem 3: Cannot populate an initial sample set of parameters'):
        batch_state(mc3, f, 'demc', 8, 80, seed=1)


# ---------------------------------------------------------------------------
# output dictionaries
# ---------------------------------------------------------------------------
def test_outputs(mc3, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)                          # sample() writes its statistics file
    f = sine_batch()
    n, seed = 16, 30
    outs = mc3.sample_batch(f['data'], f['uncert'], mc3.models.sinusoid, f['params'], f['indparams'],
                            pmin=f['pmin'], pmax=f['pmax'], pstep=f['pstep'], prior=f['prior'],
                            priorlow=f['priorlow'], priorup=f['priorup'], sampler='snooker', nchains=n,
                            nsamples=n*1500, burnin=100, seed=seed)
    assert len(outs) == 5
    q0 = problem(f, 0)
    ref = mc3.sample(q0['data'], q0['uncert'], func=mc3.models.sinusoid, params=q0['params'],
                     indparams=[q0['x']], pmin=q0['pmin'], pmax=q0['pmax'], pstep=q0['pstep'], prior=q0['prior'],
                     priorlow=q0['priorlow'], priorup=q0['priorup'], sampler='snooker', nchains=n,
                     nsamples=n*1500, burnin=100, seed=seed, log=mc3.Log(verb=-1))
    assert set(outs[0]) == set(ref)
    run = batch_state(mc3, f, 'snooker', n, n*1500, seed=seed, burnin=100, fepsilon=0.0)
    M0 = 10*n
    for b, out in enumerate(outs):
        q = problem(f, b)
        assert np.array_equal(out['posterior'], run.Z[b, M0:].cpu().numpy())
        assert np.array_equal(out['log_post'], run.log_post[b, M0:].cpu().numpy())
        assert np.array_equal(out['zchain'], run.zchain[b, M0:].cpu().numpy())
        lpr = mc3.stats.log_prior(out['posterior'], q['prior'], q['priorlow'], q['priorup'], q['pstep'])
        np.testing.assert_allclose(out['chisq'], -2.0*(out['log_post'] - lpr), rtol=1e-12)
        posterior = out['posterior'][out['zmask']]
        pick = np.random.default_rng(314159).choice(len(posterior), 20000, replace=False)
        stat_post = posterior[pick]
        mode, hlo, hhi = mc3.stats.hpd_statistics(stat_post)
        ifree = np.where(q['pstep'] > 0)[0]
        for k, v in (('mode', mode), ('hpd_low_bounds', hlo), ('hpd_high_bounds', hhi)):
            assert np.array_equal(out[k][ifree], v), (b, k)
        want = mc3.stats.calc_sample_statistics(stat_post, out['bestp'], q['pstep'], calc_hpd=True, device=True)
        for k, v in zip(('medianp', 'meanp', 'stdp', 'median_low_bounds', 'median_high_bounds',
                         'mode', 'hpd_low_bounds', 'hpd_high_bounds'), want):
            np.testing.assert_allclose(out[k], v, rtol=1e-12, atol=0, err_msg=f'{b} {k}')
        np.testing.assert_allclose(out['best_model'], om.sinusoid(out['bestp'], q['x']), rtol=1e-12, atol=1e-12)
        assert out['bestp'][2] == out['bestp'][0] and out['bestp'][4] == q['params'][4]
        assert out['best_log_post'] >= out['log_post'].max() - 1e-9
        assert out['chisq_factor'] == 1.0 and 0 < out['acceptance_rate'] < 100


# ---------------------------------------------------------------------------
# statistics
# ---------------------------------------------------------------------------
def test_line_posteriors(mc3):
    """64 straight lines y = a + b x: the posterior is Gaussian with covariance (A^T W A)^-1 and
    mean at the weighted least-squares solution."""
    B, n = 64, 200
    rs = np.random.RandomState(3)
    x = np.linspace(-1.0, 1.0, n)
    truth = np.stack([rs.uniform(-2, 2, B), rs.uniform(-1, 1, B)], axis=1)
    sig = rs.uniform(0.05, 0.5, B)
    data = [truth[b, 0] + truth[b, 1]*x + rs.normal(0, sig[b], n) for b in range(B)]
    outs = mc3.sample_batch(data, [np.full(n, s) for s in sig], mc3.models.polynomial, truth,
                            [[x]]*B, pstep=np.array([0.02, 0.02]), sampler='snooker', nchains=16,
                            nsamples=16*4000, burnin=500, seed=100)
    A = np.stack([np.ones(n), x], axis=1)
    z = []
    for b, out in enumerate(outs):
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
