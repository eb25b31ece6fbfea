"""GPU tests of the spectral form of the uniform-sigma sinusoid + line chi-squared
(csrc/chisq_grid.cu k_spectral_chisq, include/mc3b200.h mc3b_spectral_t) against the per-point
evaluation of the oracle, the pair kernel (MC3B_NO_MOMENT=1) and the tile moment form
(MC3B_NO_SPECTRAL=1)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import models as om             # noqa: E402

pytestmark = pytest.mark.gpu
TRUTH = np.array([1.0, 2.5, 0.3, 5.0, -0.2])


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def _population(mc3, x, snr, offset=5.0, nchains=256, seed=5, **kw):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(seed)
    truth = TRUTH.copy()
    truth[3] = offset
    sigma = truth[0]/snr
    data = om.sinusoid(truth, x) + rs.normal(0, sigma, x.size)
    pop = Population(data, np.full(x.size, sigma), mc3.models.sinusoid, truth*(1 + 1e-3/snr), [x], {},
                     pstep=np.array([1e-2, 1e-3, 1e-2, 1e-2, 1e-3])/max(1.0, snr/2),
                     pmin=np.array([0.0, 1.0, -np.pi, -1e9, -10.0]), pmax=np.array([50.0, 5.0, np.pi, 1e9, 10.0]),
                     nchains=nchains, sampler='demc', fepsilon=0.01, nzchain=20, seed=seed, **kw)
    return pop, data, sigma


def _oracle(P, x, data, sigma):
    return np.array([np.sum(((om.sinusoid(p, x) - data)/sigma)**2) for p in P])


def _chains(pop, truth, rs, m=200, spread=0.01):
    """Periods across the band, next to nodes and half-way between them, the band's edges."""
    p = pop.spectral_plan
    P = truth*(1 + spread*rs.standard_normal((m, 5)))
    P[:, 1] = rs.uniform(1.0, 5.0, m)
    j = rs.randint(1, p['n1'] - 3, 40)
    w = p['w1'] + p['delta']*(j + np.where(np.arange(40) % 2, 0.5 - 1e-9, 1e-9))
    P[:40, 1] = np.clip(2*np.pi/w, 1.0, 5.0)
    P[40:44, 1] = (1.0, 5.0, 1.0 + 1e-12, 5.0 - 1e-12)
    P[:, 2] = rs.uniform(-np.pi, np.pi, m)
    return P


def _gapped(n, seed):
    rs = np.random.RandomState(seed)
    x = np.linspace(0.0, 10.0, n)
    keep = np.ones(n, dtype=bool)
    for lo, w in ((n//5, n//33), (n//2, 10), (3*n//4, 1), (n - 700, 300)):
        keep[lo:lo + w] = False
    x = x[keep]
    x[x > 6.0] += 0.37*(x[1] - x[0])
    return x


@pytest.mark.parametrize('n', [100000, 20000 + 77, 1000, 'gapped'])
def test_spectral_rows_match_oracle_and_pair_kernel(mc3, monkeypatch, n):
    """Unfused rows (Population.chisq: one row + mc3b_moment_finish) against the oracle and the
    pair kernel within 1e-11, over periods across the band, at nodes and between them."""
    x = _gapped(40000, 8) if n == 'gapped' else np.linspace(0.0, 10.0, n)
    pop, data, sigma = _population(mc3, x, 2.0)
    assert pop.use_moment and pop.spectral is not None and (pop.seg is not None) == (n == 'gapped')
    P = _chains(pop, TRUTH, np.random.RandomState(1))
    Pd = torch.as_tensor(P, device=pop.dev)
    part, ld, ns = pop.data_chisq(Pd, moment_ok=True)
    assert ns == 1
    got = pop.chisq(Pd).cpu().numpy()
    want = _oracle(P, x, data, sigma)
    np.testing.assert_allclose(got, want, rtol=1e-11)
    assert int(pop.guard_hits.item()) == 0
    monkeypatch.setenv('MC3B_NO_MOMENT', '1')
    pair, *_ = _population(mc3, x, 2.0)
    assert not pair.use_moment
    np.testing.assert_allclose(got, pair.chisq(Pd).cpu().numpy(), rtol=1e-11)


def test_spectral_guard_at_high_signal_to_noise(mc3):
    """Near the mode of S/N 3000 data the amplification exceeds amp_max: the guard re-evaluates
    those chains point by point (fused and unfused) and counts them."""
    x = np.linspace(0.0, 10.0, 20000 + 77)
    pop, data, sigma = _population(mc3, x, 3000.0, nchains=128)
    assert pop.spectral is not None
    rs = np.random.RandomState(4)
    P = TRUTH*(1 + 1e-5*rs.standard_normal((128, 5)))
    h0 = int(pop.guard_hits.item())
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    want = _oracle(P, x, data, sigma)
    np.testing.assert_allclose(got, want, rtol=1e-10)
    assert int(pop.guard_hits.item()) - h0 >= 100
    # fused: one host-driven generation forced into the moment form
    pop.init_population('normal')
    pop.use_moment = True
    pop.gen_dev.fill_(0)
    before = pop.chisq_cur.clone()
    h1 = int(pop.guard_hits.item())
    pop._generation(0)
    torch.cuda.synchronize()
    Pn, after, before = pop.nextp.cpu().numpy(), pop.chisq_cur.cpu().numpy(), before.cpu().numpy()
    moved = after != before
    assert moved.any() and int(pop.guard_hits.item()) > h1
    np.testing.assert_allclose(after[moved], _oracle(Pn, x, data, sigma)[moved], rtol=1e-10)


def test_chain_outside_the_band_takes_the_exact_path(mc3):
    """A fixed period gives a band of one frequency: other periods have no node and are
    evaluated point by point (and counted); the period itself takes the table."""
    from mc3_b200.engine import Population
    x = np.linspace(0.0, 10.0, 30000)
    rs = np.random.RandomState(2)
    data = om.sinusoid(TRUTH, x) + rs.normal(0, 0.5, x.size)
    pop = Population(data, np.full(x.size, 0.5), mc3.models.sinusoid, TRUTH, [x], {},
                     pstep=np.array([1e-2, 0.0, 1e-2, 1e-2, 1e-3]), pmin=np.array([0.0, 1.0, -np.pi, 0.0, -1.0]),
                     pmax=np.array([5.0, 5.0, np.pi, 10.0, 1.0]), nchains=128, sampler='demc', nzchain=10, seed=3)
    assert pop.spectral is not None and pop.spectral_plan['n1'] == 3
    P = TRUTH*(1 + 0.01*rs.standard_normal((64, 5)))
    P[:32, 1] = TRUTH[1]
    P[32:, 1] = np.where(np.arange(32) % 2, rs.uniform(1.5, 2.3, 32), rs.uniform(2.8, 4.5, 32))   # no node near
    h0 = int(pop.guard_hits.item())
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    np.testing.assert_allclose(got, _oracle(P, x, data, 0.5), rtol=1e-11)
    assert int(pop.guard_hits.item()) - h0 == 32


def test_population_spectral_walks_the_same_chain(mc3, monkeypatch):
    """A whole run in the spectral form against the tile moment form (MC3B_NO_SPECTRAL=1):
    the same accepts and posterior rows, log-posterior within 1e-11; graph = eager, bytewise."""
    from mc3_b200 import workloads
    from mc3_b200.engine import Population
    w = workloads.config2(n=30000)
    kw = dict(pstep=w['pstep'], pmin=w['pmin'], pmax=w['pmax'], prior=w['prior'], priorlow=w['priorlow'],
              priorup=w['priorup'], nchains=512, sampler='demc', fepsilon=w['fepsilon'], nzchain=30, seed=11)
    runs = []
    for env, graph in ((None, True), (None, False), ('MC3B_NO_SPECTRAL', True)):
        if env:
            monkeypatch.setenv(env, '1')
        pop = Population(w['data'], w['uncert'], mc3.models.sinusoid, w['params'], [w['x']], {}, **kw)
        assert pop.use_moment and (pop.spectral is None) == (env is not None)
        pop.init_population('normal')
        for _ in range(3):
            pop.run(10, use_graph=graph)
        torch.cuda.synchronize()
        assert pop.use_moment
        runs.append((pop.zchain.cpu().numpy(), pop.log_post.cpu().numpy(), pop.Z.cpu().numpy(),
                     pop.counters()['numaccept']))
    assert all(np.array_equal(a, b) for a, b in zip(runs[0][:3], runs[1][:3]))
    assert np.array_equal(runs[0][0], runs[2][0]) and runs[0][3] == runs[2][3]
    np.testing.assert_allclose(runs[0][1], runs[2][1], rtol=1e-11)
    assert np.array_equal(runs[0][2], runs[2][2])


def test_spectral_table_does_not_depend_on_the_device():
    """Fixed-order sums: two GPUs build the same table bytes (skips on one GPU)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    import ctypes
    from mc3_b200 import _lib, spectral
    x = np.linspace(0.0, 10.0, 50000)
    d = om.sinusoid(TRUTH, x) + np.random.RandomState(0).normal(0, 0.5, x.size)
    p = spectral.plan(0.0, 10.0, 2*np.pi/5, 2*np.pi, x.size)
    outs = []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            S = _lib.SpectralStruct()
            S.w1, S.w2, S.delta, S.xc, S.n1, S.n2, S.order = (p[k] for k in ('w1', 'w2', 'delta', 'xc', 'n1', 'n2',
                                                                                 'order'))
            size = ctypes.c_int64(0)
            _lib.call('mc3b_spectral_size', S.n1, S.n2, S.order, ctypes.byref(size))
            tab = torch.zeros(size.value, dtype=torch.float64, device=f'cuda:{dev}')
            dx, dd = (torch.from_numpy(a).to(f'cuda:{dev}') for a in (x, d))
            S.table = tab.data_ptr()
            _lib.call('mc3b_spectral_prepare', dx.data_ptr(), dd.data_ptr(), x.size, 5.0, -0.2, ctypes.byref(S),
                      _lib.stream_ptr())
            torch.cuda.synchronize()
            outs.append(tab.cpu().numpy())
    assert np.array_equal(outs[0].view(np.int64), outs[1].view(np.int64))
