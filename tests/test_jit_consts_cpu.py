"""CPU-only: user models of run-time constants and a prepare step (CudaModel(...,
nconst=m, nwork=w)) compile to sm_100a CUBINs whose kernels carry the names the loader
derives; work slots without a prepare, a prepare of the wrong signature, the 32-slot cap
and negative counts are refused; a comment that mentions prepare( does not count; the
model pickles with its counts; the cache key tracks the counts, not the constant values,
and a model of neither keeps its key and its UserModel wrapper."""
import ctypes
import hashlib
import os
import pickle
import subprocess

import numpy as np
import pytest

from mc3_b200 import _lib
from mc3_b200 import jit
from mc3_b200.models import CudaModel

try:
    NVRTC = jit.find_nvrtc()[0]
except _lib.Mc3bError:
    NVRTC = None
pytestmark = pytest.mark.skipif(NVRTC is None, reason='no NVRTC 12.8+ found')

HORNER = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
GAUSS = '''__device__ void prepare(real* p) { p[4] = 1 / p[2]; }
__device__ real model(real x, const real* p) {
    real d = (x - p[1]) * p[4];
    return fma(p[0], exp((real)(-0.5) * d * d), p[3]);
}'''


def consts_source(k, nconst):
    """p[0] + p[1] x_0 + ... over k inputs, scaled by the sum of nconst constants; prepare
    keeps that sum in the work slot."""
    args = ', '.join(f'real x{j}' for j in range(k))
    body = ' + '.join(['p[0]'] + [f'p[{j + 1}] * x{j}' for j in range(k)])
    csum = ' + '.join(f'p[{k + 1 + j}]' for j in range(nconst))
    return (f'__device__ void prepare(real* p) {{ p[{k + 1 + nconst}] = {csum}; }}\n'
            f'__device__ real model({args}, const real* p) {{ return ({body}) * p[{k + 1 + nconst}]; }}')


def _compile(source, nmodel, ninputs=1, nconst=0, nwork=0, dtype=_lib.F64, cap=1 << 22):
    lib = _lib.load()
    buf = ctypes.create_string_buffer(max(cap, 1))
    size = ctypes.c_int64(-1)
    log = ctypes.create_string_buffer(1 << 16)
    desc = _lib.UserModelDesc(nmodel, ninputs, nconst, nwork, dtype)
    rc = lib.mc3b_user_model_compile_desc(NVRTC.encode(), source.encode(), ctypes.byref(desc), buf, cap,
                                          ctypes.byref(size), log, len(log))
    return rc, buf.raw[:max(size.value, 0)], log.value.decode(), lib.mc3b_last_error().decode()


def _elf(cubin, tmp_path):
    cuobjdump = '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('no cuobjdump')
    path = tmp_path / 'm.cubin'
    path.write_bytes(cubin)
    return subprocess.run([cuobjdump, '-elf', str(path)], capture_output=True, text=True).stdout


@pytest.mark.parametrize('k', [1, 3])
@pytest.mark.parametrize('dtype', [_lib.F64, _lib.F32])
def test_constants_and_prepare_compile_to_sm100a_cubin(k, dtype, tmp_path):
    # compile_desc checks NVRTC's lowered names against the symbols the loader looks up
    # and fails (MC3B_ERR_CUDA) on any mismatch, so rc == OK covers that check
    rc, cubin, log, err = _compile(consts_source(k, 2), k + 1, k, 2, 1, dtype)
    assert rc == _lib.OK, (err, log)
    out = _elf(cubin, tmp_path)
    assert 'sm_100a' in out
    t = 'd' if dtype == _lib.F64 else 'f'
    model = f'10UserModelKI{t}Li{k + 1}ELi{k}ELi2ELi1EE'
    for lc in (32, 8, 1):
        for usig in (1, 0):
            assert f'k_model_chisqINS_{model}E{t}Li{lc}ELi1ELb{usig}E' in out, (lc, usig)
    assert f'k_model_eval_kINS_{model}' in out and 'mc3b_jit_abi' in out


def test_prepare_alone_takes_the_constants_wrapper():
    rc, cubin, log, err = _compile(GAUSS.replace('p[4]', 'p[2]'), 4)   # 1/sigma in place
    assert rc == _lib.OK, (err, log)
    assert b'10UserModelKIdLi4ELi1ELi0ELi0EE' in cubin and b'9UserModelI' not in cubin


def test_work_slots_without_prepare_are_refused():
    rc, _, log, err = _compile(HORNER, 3, nwork=1)
    assert rc == _lib.ERR_ARG and 'prepare' in err and 'prepare' in log
    with pytest.raises(ValueError, match='prepare'):
        jit.compile_cubin(HORNER, 3, _lib.F64, 'nowork', nwork=2)


@pytest.mark.parametrize('line', [1, 3])
def test_prepare_of_the_wrong_signature_fails_at_its_line(line):
    src = ''.join(f'__device__ real helper{i}(real a) {{ return a; }}\n' for i in range(line - 1))
    src += '__device__ void prepare(real* p, int n) { p[3] = n; }\n' + HORNER
    rc, _, log, _ = _compile(src, 3, nwork=1)
    assert rc == _lib.ERR_ARG
    assert f'model.cu({line})' in log
    with pytest.raises(ValueError, match=r'model\.cu\(%d\)' % line):
        jit.compile_cubin(src, 3, _lib.F64, 'badprep', nwork=1)


def test_a_comment_that_mentions_prepare_does_not_count():
    src = ('// prepare(real* p) would hoist 1/sigma here\n'
           '/* so would a\n   prepare(p) */\n' + HORNER)
    rc, cubin, log, err = _compile(src, 3)
    assert rc == _lib.OK, (err, log)
    assert b'9UserModelIdLi3EE' in cubin and b'UserModelK' not in cubin
    rc, _, _, err = _compile(src, 3, nwork=1)
    assert rc == _lib.ERR_ARG and 'prepare' in err


def test_slot_cap_and_negative_counts():
    with pytest.raises(ValueError, match='32 slots'):
        CudaModel(GAUSS, 4, nconst=20, nwork=9)
    CudaModel(GAUSS, 4, nconst=20, nwork=8)
    for nc, nw in ((-1, 0), (0, -1)):
        with pytest.raises(ValueError, match='negative'):
            CudaModel(GAUSS, 4, nconst=nc, nwork=nw)
        rc, _, _, err = _compile(GAUSS, 4, 1, nc, nw)
        assert rc == _lib.ERR_ARG and 'negative' in err
    rc, _, _, err = _compile(GAUSS, 4, 1, 20, 9)
    assert rc == _lib.ERR_ARG and '32 slots' in err


def test_pickle_keeps_the_counts():
    m = CudaModel(consts_source(3, 2), 4, name='k3', ninputs=3, nconst=2, nwork=1)
    m2 = pickle.loads(pickle.dumps(m))
    assert (m2.source, m2.nparams, m2.name, m2.ninputs, m2.nconst, m2.nwork) == (m.source, 4, 'k3', 3, 2, 1)
    g = pickle.loads(pickle.dumps(CudaModel(GAUSS, 4, name='gauss', nwork=1)))
    assert vars(g) == {'source': GAUSS, 'nparams': 4, 'name': 'gauss', 'nwork': 1} and g.nconst == 0
    one = pickle.loads(pickle.dumps(CudaModel(HORNER, 3, name='horner')))
    assert vars(one) == {'source': HORNER, 'nparams': 3, 'name': 'horner'}
    assert (one.ninputs, one.nconst, one.nwork) == (1, 0, 0)


def test_cache_key_tracks_the_counts_not_the_values():
    h = hashlib.sha256()
    ver = jit.find_nvrtc()[1]
    for part in (HORNER, '3', str(_lib.F64), str(_lib.load().mc3b_version()), f'{ver[0]}.{ver[1]}',
                 jit._headers_digest()):
        h.update(part.encode() + b'\0')
    plain = CudaModel(HORNER, 3)
    assert plain.cache_key() == h.hexdigest() == jit.cache_key(HORNER, 3, _lib.F64, 1, 0, 0)
    keys = {CudaModel(HORNER, 3, nconst=c, nwork=w).cache_key() for c in (0, 1, 2) for w in (0, 1)}
    assert len(keys) == 6
    # the values come with the arguments, not the model: one model, one key, any values
    m = CudaModel(HORNER, 2, nconst=1)
    assert m.split_args([np.zeros(4), 0.5])[1].tolist() == [0.5]
    assert m.split_args([np.zeros(4), 7.0])[1].tolist() == [7.0]


def test_constants_are_flattened_in_order():
    m = CudaModel(HORNER, 2, ninputs=2, nconst=5)
    x, y = np.arange(3.0), np.ones(3)
    xs, k = m.split_args([x, y, 1, np.float64(2.0), np.array(3.0), np.array([4.0, 5.0])])
    assert len(xs) == 2 and xs[0] is x and xs[1] is y
    assert k.tolist() == [1, 2, 3, 4, 5]
    with pytest.raises(ValueError, match='takes 5 constant.*got 4'):
        m.split_args([x, y, 1, 2, [3, 4]])
    with pytest.raises(ValueError, match='1-D'):
        m.split_args([x, y, np.ones((2, 3))])
    # a model of neither constants nor work slots takes its arrays as before
    assert CudaModel(HORNER, 3).split_args([x, 3.5]) == ([x, 3.5], None)
