"""GPU test of the guard count of a fused spectral-form launch (csrc/chisq_args.cuh
fused_metropolis_end): when the guard fires in several CTAs, guard_hits and the guard record
end with the count of flagged chains, whether the launch counts its arrivals (record or
advance on) or not (each CTA adds its hits to the counter), and the arrival word returns to
zero."""
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


def test_fused_spectral_counts_hits_with_and_without_arrival():
    import mc3_b200 as mc3
    from mc3_b200.engine import Population
    x = np.linspace(0.0, 10.0, 30000)
    rs = np.random.RandomState(2)
    data = om.sinusoid(TRUTH, x) + rs.normal(0, 0.5, x.size)
    nchains = 512                                   # four CTAs of k_spectral_chisq
    # a fixed period: a band of one frequency, so that any other period has no node and
    # takes the guard's point-by-point path
    pop = Population(data, np.full(x.size, 0.5), mc3.models.sinusoid, TRUTH, [x], {},
                     pstep=np.array([1e-2, 0.0, 1e-2, 1e-2, 1e-3]), pmin=np.array([0.0, 1.0, -np.pi, 0.0, -1.0]),
                     pmax=np.array([5.0, 5.0, np.pi, 10.0, 1.0]), nchains=nchains, sampler='demc', nzchain=10,
                     seed=3)
    assert pop.spectral is not None and pop.spectral_plan['n1'] == 3
    pop.init_population('normal')
    pop.use_moment = True
    c0, c1 = pop.chain0, pop.chain0 + pop.nlocal
    P = TRUTH*(1 + 0.01*rs.standard_normal((nchains, 5)))
    P[:, 1] = TRUTH[1]
    flagged = np.array([0, 5, 127, 128, 300, 301, 302, 511])      # in CTAs 0, 1, 2 and 3
    P[flagged, 1] = rs.uniform(1.5, 2.3, flagged.size)
    pop.nextp[c0:c1] = torch.as_tensor(P, device=pop.dev)
    pop.inb[c0:c1] = 1
    ring = pop.moment.record
    assert ring
    for record, advance in ((True, True), (True, False), (False, True), (False, False)):
        pop.moment.record = ring if record else None
        h0 = int(pop.guard_hits.item())
        g0 = int(pop.gen_dev.item())
        gen = pop.gen
        pop.data_chisq(pop.nextp[c0:c1], fuse=(c0, gen, -1, advance))
        torch.cuda.synchronize()
        hits = int(pop.guard_hits.item())
        assert hits - h0 == flagged.size, (record, advance)
        assert int(pop.gen_dev.item()) == g0 + (1 if advance else 0)
        assert int(pop.fuse_done.abs().sum().item()) == 0
        if record:
            v = int(pop._guard_ring.numpy()[(gen + 1) % 64])
            assert (v >> 32) & 0xffffffff == gen + 1 and v & 0xffffffff == hits
        pop.gen += 1
    pop.moment.record = ring
