"""GPU tests of the spectral-form generation (k_spectral_chisq with the fused Metropolis epilogue
of a one-split launch: no arrival spin, the chain's row added from a register): whole runs
through block graphs equal host-driven generations byte for byte, and the order-15 table (long
baselines) gives the point-by-point chi-squared."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import models as om             # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def _run(mc3, nchains, sampler, thinning, graph, ngen):
    from mc3_b200 import workloads
    from mc3_b200.engine import Population
    w = workloads.config2()
    pop = Population(w['data'], w['uncert'], mc3.models.sinusoid, w['params'], [w['x']], {},
                     pstep=w['pstep'], pmin=w['pmin'], pmax=w['pmax'], prior=w['prior'], priorlow=w['priorlow'],
                     priorup=w['priorup'], nchains=nchains, sampler=sampler, fepsilon=w['fepsilon'],
                     thinning=thinning, nzchain=ngen + 2, seed=21)
    assert pop.use_moment and pop.spectral is not None
    pop.init_population('normal')
    pop.run(ngen, use_graph=graph)
    torch.cuda.synchronize()
    assert pop.use_moment
    if graph:
        # 1e5 points: 32 generations per block graph at 128 chains, 8 at 512 (Population.run)
        assert pop._block == (32 if nchains == 128 else 8)
    c = pop.counters()
    return (pop.Z.cpu().numpy(), pop.log_post.cpu().numpy(), pop.zchain.cpu().numpy(), pop.chisq_cur.cpu().numpy(),
            c['numaccept'], np.asarray(c['bestp']), int(pop.fuse_done.abs().sum().item()))


@pytest.mark.parametrize('thinning', [1, 3])
@pytest.mark.parametrize('sampler', ['demc', 'snooker', 'mrw'])
@pytest.mark.parametrize('nchains', [128, 512])
def test_block_graphs_equal_host_driven_generations(mc3, nchains, sampler, thinning):
    ngen = 1 + 2*(32 if nchains == 128 else 8)          # warm-up generation, then two block replays
    g = _run(mc3, nchains, sampler, thinning, True, ngen)
    e = _run(mc3, nchains, sampler, thinning, False, ngen)
    for a, b in zip(g[:4], e[:4]):
        assert a.tobytes() == b.tobytes()
    assert g[4] == e[4] and g[5].tobytes() == e[5].tobytes()
    assert g[6] == 0 and e[6] == 0                      # the arrival counters reset themselves


def test_order_15_table_matches_point_by_point(mc3):
    """A long baseline (x over 1000 periods of the shortest one) plans K = 15."""
    from mc3_b200.engine import Population
    truth = np.array([1.0, 2.5, 0.3, 5.0, -2e-3])
    x = np.linspace(0.0, 1000.0, 1000)
    rs = np.random.RandomState(6)
    sigma = 0.5
    data = om.sinusoid(truth, x) + rs.normal(0, sigma, x.size)
    pop = Population(data, np.full(x.size, sigma), mc3.models.sinusoid, truth, [x], {},
                     pstep=np.array([1e-2, 1e-4, 1e-2, 1e-2, 1e-5]), pmin=np.array([0.0, 1.0, -np.pi, -10.0, -1.0]),
                     pmax=np.array([5.0, 5.0, np.pi, 20.0, 1.0]), nchains=256, sampler='demc', nzchain=10, seed=4)
    assert pop.spectral is not None and pop.spectral_plan['order'] == 15
    P = truth*(1 + 0.01*rs.standard_normal((256, 5)))
    P[:, 1] = rs.uniform(1.0, 5.0, 256)
    P[:, 2] = rs.uniform(-np.pi, np.pi, 256)
    h0 = int(pop.guard_hits.item())
    got = pop.chisq(torch.as_tensor(P, device=pop.dev)).cpu().numpy()
    want = np.array([np.sum(((om.sinusoid(p, x) - data)/sigma)**2) for p in P])
    np.testing.assert_allclose(got, want, rtol=1e-10)
    assert int(pop.guard_hits.item()) - h0 < 256 // 4      # most rows come from the table
