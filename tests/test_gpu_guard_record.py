"""GPU tests of the guard records of the moment form (include/mc3b200.h mc3b_moment_t.record):
the fused epilogue stores the guard count of every generation into page-locked host memory, and
Population's policy reads it from there instead of copying the counter on every run() call."""
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
# amp_max of the population whose guard fires inside generations (see _firing)
AMP_FIRING = 36.0


@pytest.fixture(scope='module')
def mc3():
    import mc3_b200
    return mc3_b200


def _population(mc3, x, snr, nchains=256, seed=5):
    from mc3_b200.engine import Population
    rs = np.random.RandomState(seed)
    sigma = TRUTH[0]/snr
    data = om.sinusoid(TRUTH, x) + rs.normal(0, sigma, x.size)
    pop = Population(data, np.full(x.size, sigma), mc3.models.sinusoid, TRUTH*(1 + 1e-3/snr), [x], {},
                     pstep=np.array([1e-2, 1e-3, 1e-2, 1e-2, 1e-3]), pmin=np.array([0.0, 1.0, -np.pi, -1e9, -10.0]),
                     pmax=np.array([50.0, 5.0, np.pi, 1e9, 10.0]), nchains=nchains, sampler='demc', fepsilon=0.01,
                     nzchain=1000, seed=seed)
    pop.init_population('normal')
    return pop


def _firing(mc3, monkeypatch, amp=AMP_FIRING):
    """S/N 2 data over 0.64 of a period: the least-squares reference line is far from the chains'
    lines, so the guard's bound (which has the line term) exceeds the a-priori estimate before
    generation 0 (which has not, 10.4 here against a limit of amp_max / 2) about three times near
    the mode.  With amp_max = 36 the a-priori check keeps the moment form, no chain of the initial
    population trips the guard, and the chains start to trip it after about 20 generations, a
    growing fraction of them as they converge (a B200 run: 2, 4, 10, ... 90 of 256 per generation)."""
    monkeypatch.setenv('MC3B_MOMENT_AMP', str(amp))
    return _population(mc3, np.linspace(0.0, 1.6, 20000), 2.0)


def _ring(pop):
    """{generation mod 2^32: hits} of the records in the ring."""
    v = pop._guard_ring.numpy().astype(np.int64)
    return {int(s): int(h) for s, h in zip((v >> 32) & 0xffffffff, v & 0xffffffff)}


def _drive(pop, calls, ngen, graph):
    """`calls` run(ngen) calls.  Returns (index of the call that ran in the pair form first or
    None, {generation: hits} of every record written, generation count at each call's start)."""
    hist, starts, switched = {}, [], None
    for k in range(calls):
        starts.append(pop.gen)
        pop.run(ngen, use_graph=graph)
        torch.cuda.synchronize()
        if not pop.use_moment:
            switched = k
            break
        rec = _ring(pop)
        for g in range(pop.gen - ngen + 1, pop.gen + 1):
            hist[g] = rec[g]
    return switched, hist, starts


def _predict(starts, ngen, hist, nlocal, R=64):
    """The documented rule: at the start of call k the record of G* = the generation count at the
    start of call k - 2 (clamped to >= gen - R + 1) is compared with the last record read; the
    form is left when the hits between them exceed 1e-3 per chain-step."""
    seen = (0, 0)
    for k in range(3, len(starts)):   # at call 2, G* = 0: generation 0 has no record
        g = max(starts[k - 2], starts[k] - R + 1)
        if g <= seen[0]:
            continue
        if hist[g] - seen[1] > 1e-3*nlocal*(g - seen[0]):
            return k
        seen = (g, hist[g])
    return None


@pytest.mark.parametrize('ngen,graph', [(1, True), (64, True), (1, False)])
def test_switch_at_the_generation_the_records_predict(mc3, monkeypatch, ngen, graph):
    calls = 40 if ngen == 1 else 8
    pop = _firing(mc3, monkeypatch)
    switched, hist, starts = _drive(pop, calls, ngen, graph)
    assert switched is not None and switched >= 3           # the a-priori check kept the moment form
    assert hist[max(hist)] > 0                                 # ... and the guard fired inside generations
    assert switched == _predict(starts, ngen, hist, pop.nlocal)
    # a fixed call sequence gives the same history, byte for byte
    pop2 = _firing(mc3, monkeypatch)
    switched2, hist2, _ = _drive(pop2, calls, ngen, graph)
    assert switched2 == switched and hist2 == hist
    for _ in range(3):
        pop.run(ngen, use_graph=graph)
        pop2.run(ngen, use_graph=graph)
    torch.cuda.synchronize()
    for a, b in ((pop.Z, pop2.Z), (pop.log_post, pop2.log_post), (pop.zchain, pop2.zchain)):
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()


def test_ring_holds_the_last_records(mc3, monkeypatch):
    """After G generations slot g % 64 holds record g for g = max(1, G - 63) .. G, and record G
    holds the counter's value; a short eager run writes records too."""
    pop = _firing(mc3, monkeypatch)
    pop.run(5, use_graph=False)                       # eager generations, host-driven
    torch.cuda.synchronize()
    rec = _ring(pop)
    assert all(g in rec for g in range(1, 6)) and rec[5] == int(pop.guard_hits.item())
    pop.run(100, use_graph=True)                      # one call: no decision inside it
    torch.cuda.synchronize()
    G = pop.gen
    v = pop._guard_ring.numpy().astype(np.int64)
    for g in range(G - 63, G + 1):
        assert (v[g % 64] >> 32) & 0xffffffff == g
    assert int(v[G % 64] & 0xffffffff) == int(pop.guard_hits.item()) > 0


def test_no_copy_between_replays(mc3):
    """Steady state of run(1) in the moment form: the stream holds graph replays only, no
    device-to-host copy."""
    from torch.profiler import ProfilerActivity, profile
    pop = _population(mc3, np.linspace(0.0, 10.0, 20000), 2.0)
    pop.run(4, use_graph=True)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            pop.run(1, use_graph=True)
        torch.cuda.synchronize()
    assert pop.use_moment
    names = [e.name for e in prof.events()]
    assert any('k_propose' in n for n in names)
    assert not [n for n in names if 'DtoH' in n or 'Device -> Pinned' in n or 'Memcpy' in n]
