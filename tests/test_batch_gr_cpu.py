"""CPU-only checks of sample_batch's Gelman-Rubin test: the argument errors raised before the
device, the report schedule and grnmin rule shared with mcmc() against a restatement of the
reference's loop, the ctypes signature of mc3b_batch_gelman_rubin, and the resources of its
kernel (no local memory, no stack)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import mc3_b200 as mc3
from mc3_b200 import _lib
from mc3_b200.mcmc_driver import gr_min_size, report_points

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = '/usr/local/cuda/bin/cuobjdump'


def line_fits(B=3, n=40):
    x = np.linspace(0.0, 1.0, n)
    return dict(data=[1.0 + 0.5*b + 2.0*x for b in range(B)], uncert=[np.full(n, 0.1)]*B,
                func=mc3.models.polynomial, params=np.array([[1.0 + 0.5*b, 2.0] for b in range(B)]),
                indparams=[[x]]*B, pstep=np.array([0.01, 0.01]), sampler='mrw', nchains=8, nsamples=800,
                grtest=True)


@pytest.mark.parametrize('kw,match', [
    (dict(grnmin=-1), r"^Invalid 'grnmin' argument \(minimum number of samples to stop the MCMC under GR "
                      r"convergence\), must either be grnmin > 1to set the minimum number of samples, "
                      r"or 0 < grnmin < 1to set the fraction of samples required to evaluate\.$"),
    (dict(grnmin=-0.5, grtest=False), r"^Invalid 'grnmin' argument"),
    (dict(nchains=1), r'^the Gelman-Rubin test needs at least 2 chains, got 1$'),
    (dict(nchains=1, grbreak=1.01), r'^the Gelman-Rubin test needs at least 2 chains, got 1$'),
])
def test_errors_before_the_device(kw, match):
    args = line_fits()
    args.update(kw)
    with pytest.raises(ValueError, match=match):
        mc3.sample_batch(**args)


class _Raise:
    def error(self, message, exception=ValueError):
        raise exception(message)


def _reference_loop(nzchain, nchains, thinning, zburn, M0, grnmin):
    """mcmc()'s report loop and grnmin rule as they stood before they were factored out."""
    if grnmin >= 1:
        grnmin = int(grnmin/thinning)
    elif grnmin > 0:
        grnmin = int(grnmin*nchains*(nzchain - zburn))
    grnmin += int(M0 + zburn*nchains)
    step_k = max(1, int(np.ceil(nzchain/10)))
    k_done, ks = 0, []
    while k_done < nzchain:
        k_next = min(nzchain, k_done + step_k)
        ks.append(k_next)
        k_done = k_next
    return ks, grnmin


@pytest.mark.parametrize('nzchain', [0, 1, 2, 9, 10, 11, 19, 99, 100, 101, 14286, 33334])
@pytest.mark.parametrize('grnmin', [0.0, 0.2, 0.5, 0.999, 1, 1.5, 250, 7000])
@pytest.mark.parametrize('nchains,thinning', [(7, 1), (24, 3), (256, 2)])
def test_schedule_and_grnmin_match_the_loop(nzchain, grnmin, nchains, thinning):
    zburn = nzchain//4
    M0 = 10*nchains
    ks, gmin = _reference_loop(nzchain, nchains, thinning, zburn, M0, grnmin)
    assert report_points(nzchain) == ks
    assert gr_min_size(grnmin, nchains, nzchain, zburn, thinning, M0, _Raise()) == gmin


def test_grnmin_error_goes_through_the_log():
    with pytest.raises(ValueError, match=r"^Invalid 'grnmin' argument"):
        gr_min_size(-1e-3, 7, 100, 10, 1, 70, _Raise())


def test_ctypes_signature():
    text = open(os.path.join(ROOT, 'include', 'mc3b200.h')).read()
    decl = re.search(r'int mc3b_batch_gelman_rubin\(([^)]*)\);', text).group(1)
    params = [p.strip() for p in decl.split(',')]
    assert params == ['const mc3b_batch_t* b', 'int64_t k', 'int64_t zburn', 'double grbreak', 'int64_t grnmin',
                      'double* psrf', 'int64_t ldpsrf', 'int64_t* kstop', 'void* stream']
    res, args = _lib._SIGS['mc3b_batch_gelman_rubin']
    assert res is ctypes.c_int
    assert args == [ctypes.POINTER(_lib.BatchStruct), ctypes.c_int64, ctypes.c_int64, ctypes.c_double,
                    ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
    assert hasattr(_lib.load(), 'mc3b_batch_gelman_rubin')


def test_kernel_has_no_local_memory():
    if not os.path.exists(CUOBJDUMP):
        pytest.skip('no cuobjdump')
    lib = _lib.load()._name
    out = subprocess.run([CUOBJDUMP, '-res-usage', lib], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.splitlines()
    hits = [lines[i + 1] for i, line in enumerate(lines) if re.search(r'Function \S*k_batch_gr\S*:', line)]
    assert len(hits) == 1, hits
    assert re.search(r'\bSTACK:0\b', hits[0]) and re.search(r'\bLOCAL:0\b', hits[0]), hits[0]
