"""The end of a fused spectral-form launch, read from the SASS (no GPU needed): on one device the
launch-wide arrival carries the guard hits in its atomic and needs no fence, so neither
k_spectral_chisq instantiation holds a device-scope sequentially-consistent fence; the
system-scope fence of peer mode stays."""
import os
import re
import subprocess

import pytest

from mc3_b200 import build as b


@pytest.fixture(scope='module')
def sass(tmp_path_factory):
    obj = tmp_path_factory.mktemp('sass') / 'chisq_grid.o'
    cmd = [b._nvcc()] + b.NVCC_FLAGS + ['-c', os.path.join(b.CSRC, 'chisq_grid.cu'), '-o', str(obj)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    dump = os.path.join(os.path.dirname(b._nvcc()), 'cuobjdump')
    r = subprocess.run([dump if os.path.exists(dump) else 'cuobjdump', '-sass', str(obj)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out, cur = {}, None
    for line in r.stdout.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur:
            out[cur].append(line)
    return out


@pytest.mark.parametrize('order', [9, 15])
def test_spectral_tail_has_no_device_fence(sass, order):
    hits = [v for k, v in sass.items() if re.search(rf'k_spectral_chisqILi{order}E', k)]
    assert len(hits) == 1
    text = '\n'.join(hits[0])
    assert 'MEMBAR.SC.GPU' not in text
    assert 'MEMBAR.SC.SYS' in text                  # peer mode
    assert 'ATOMG.E.ADD.64' in text                 # the arrival word
