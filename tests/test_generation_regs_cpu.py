"""Resource usage of the two kernels of a spectral-form generation, read from ptxas (no GPU
needed): the proposal kernel keeps a chain's proposal in registers (no local-memory frame, no
spills), and the spectral chi-squared kernel does not spill at either Taylor order (its stack
frame is the slow-path argument reduction of sincos only)."""
import os
import re
import subprocess

import pytest

from mc3_b200 import build as b


def _ptxas(src, tmp_path):
    """{kernel name: (stack bytes, spill store bytes, spill load bytes)} of the entry functions of src."""
    cmd = [b._nvcc()] + b.NVCC_FLAGS + ['-c', os.path.join(b.CSRC, src), '-o', str(tmp_path / (src + '.o'))]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            out[cur] = tuple(int(v) for v in m.groups())
            cur = None
    return out


def _one(props, pattern):
    hits = [v for k, v in props.items() if re.search(pattern, k)]
    assert len(hits) == 1, (pattern, sorted(props))
    return hits[0]


@pytest.fixture(scope='module')
def props(tmp_path_factory):
    tmp = tmp_path_factory.mktemp('ptxas')
    return {src: _ptxas(src, tmp) for src in ('sampler.cu', 'chisq_grid.cu')}


@pytest.mark.parametrize('replay', [0, 1])
def test_propose_has_no_local_memory(props, replay):
    assert _one(props['sampler.cu'], rf'k_proposeILb{replay}E') == (0, 0, 0)


@pytest.mark.parametrize('order', [9, 15])
def test_spectral_chisq_does_not_spill(props, order):
    stack, st, ld = _one(props['chisq_grid.cu'], rf'k_spectral_chisqILi{order}E')
    assert st == 0 and ld == 0
    assert stack <= 96
