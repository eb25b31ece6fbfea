"""CPU-only: the host rule of the moment form's guard records (mc3_b200.engine.GuardRecords) on a
ring written by hand the way the fused epilogue writes it."""
import numpy as np
import pytest

from mc3_b200 import _lib
from mc3_b200.engine import GuardRecords

R = GuardRecords.R


def _store(ring, g, hits):
    """What the last CTA of generation g stores: (g mod 2^32) << 32 | hits."""
    ring[g % R] = np.int64(np.uint64(((g & 0xffffffff) << 32) | hits).view(np.int64))


def _busy():
    raise AssertionError('the record should have been there')


def test_fill_matches_no_generation():
    ring = np.zeros(R, dtype=np.int64)
    gr = GuardRecords(ring)
    for g in list(range(0, 4 * R)) + [(1 << 32) + s for s in range(R)] + [(1 << 32) - 1]:
        assert gr.read(g) is None


def test_stamp_is_compared_on_32_bits():
    ring = np.zeros(R, dtype=np.int64)
    gr = GuardRecords(ring)
    g = (1 << 32) + 5                      # generation 2^32 + 5 stores stamp 5
    _store(ring, g, 7)
    assert gr.read(g) == 7
    assert gr.read(g - R) is None          # an older record of the slot is not it
    _store(ring, g - R, 3)
    assert gr.read(g) is None and gr.read(g - R) == 3
    _store(ring, 9, 0xffffffff)            # hits are 32 unsigned bits
    assert gr.read(9) == 0xffffffff


def test_record_of_the_call_before_the_previous_one():
    """run(1) calls: the call at generation k reads record k - 2 (k >= 3); the first decision
    compares record 1 with no hits before generation 1."""
    ring = np.zeros(R, dtype=np.int64)
    gr = GuardRecords(ring)
    nlocal = 4096                          # threshold: 4.096 hits per generation
    read = []
    for gen in range(12):
        for g in range(1, gen + 1):
            _store(ring, g, 4 * g)         # 4 hits per generation: under the threshold
        before = gr.seen
        assert not gr.step(gen, 1, nlocal, True, _busy)
        if gr.seen != before:
            read.append((gen, gr.seen[0]))
    assert read == [(gen, gen - 2) for gen in range(3, 12)]


def test_threshold_and_clamp():
    ring = np.zeros(R, dtype=np.int64)
    gr = GuardRecords(ring)
    calls = [(0, 1), (1, 200), (201, 1), (202, 1)]
    for g in range(1, 203):
        _store(ring, g, 0)
    for gen, ngen in calls[:3]:
        assert not gr.step(gen, ngen, 1000, True, _busy)
    # the call at 202 would read record 1, long overwritten: it reads 202 - 63 = 139 instead
    _store(ring, 139, 139)                 # 1 hit per generation: 1e-3 per chain-step of 1000 chains
    assert not gr.step(202, 1, 1000, True, _busy)
    assert gr.seen == (139, 139)
    gr2 = GuardRecords(np.zeros(R, dtype=np.int64))
    for g in range(1, 203):
        _store(gr2.ring, g, 0)
    _store(gr2.ring, 139, 140)             # one hit more: above the threshold
    for gen, ngen in calls[:3]:
        gr2.step(gen, ngen, 1000, True, _busy)
    assert gr2.step(202, 1, 1000, True, _busy)


def test_missing_record_with_idle_stream_raises():
    ring = np.zeros(R, dtype=np.int64)
    gr = GuardRecords(ring)
    for gen in (0, 1, 2):
        gr.step(gen, 1, 256, True, _busy)
    with pytest.raises(_lib.Mc3bError, match='generation 1'):
        gr.step(3, 1, 256, True, lambda: True)


def test_calls_without_records_are_not_read():
    """A call whose generations write no records (the small-population kernel) drops the
    pending records, and the call after it does not wait for the record it would start at."""
    ring = np.zeros(R, dtype=np.int64)
    gr = GuardRecords(ring)
    gr.step(0, 1, 256, True, _busy)
    gr.step(1, 1, 256, True, _busy)
    assert not gr.step(2, 5, 256, False, _busy) and gr.starts == []
    for gen in (7, 8, 9):                  # record 7 does not exist: only 8 and 9 are pending
        gr.step(gen, 1, 256, True, _busy)
    assert gr.starts == [8, 9]
