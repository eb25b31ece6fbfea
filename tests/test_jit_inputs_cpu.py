"""CPU-only: user models of several per-point inputs (CudaModel(..., ninputs=k)) compile
to sm_100a CUBINs whose kernels carry the names the loader derives; a `model` of
another arity fails to compile at its own line; ninputs outside 1..4 is refused; the
model pickles with its ninputs; the cache key of a one-input model is unchanged."""
import ctypes
import os
import pickle
import subprocess

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


def linear_source(k):
    """p[0] + sum_j p[j+1] x_j over k inputs."""
    args = ', '.join(f'real x{j}' for j in range(k))
    body = ' + '.join(['p[0]'] + [f'p[{j + 1}] * x{j}' for j in range(k)])
    return f'__device__ real model({args}, const real* p) {{ return {body}; }}'


def _compile(source, nmodel, ninputs, dtype=_lib.F64, cap=1 << 22):
    lib = _lib.load()
    buf = ctypes.create_string_buffer(max(cap, 1))
    size = ctypes.c_int64(-1)
    log = ctypes.create_string_buffer(1 << 16)
    rc = lib.mc3b_user_model_compile_ex(NVRTC.encode(), source.encode(), nmodel, ninputs, dtype, buf, cap,
                                        ctypes.byref(size), log, len(log))
    return rc, buf.raw[:max(size.value, 0)], log.value.decode(), lib.mc3b_last_error().decode()


@pytest.mark.parametrize('k', [2, 4])
@pytest.mark.parametrize('dtype', [_lib.F64, _lib.F32])
def test_several_inputs_compile_to_sm100a_cubin(k, dtype, tmp_path):
    # compile_ex checks NVRTC's lowered names against the symbols the loader looks up
    # and fails (MC3B_ERR_CUDA) on any mismatch, so rc == OK covers that check
    rc, cubin, log, err = _compile(linear_source(k), k + 1, k, dtype)
    assert rc == _lib.OK, (err, log)
    assert cubin[:4] == b'\x7fELF'
    cuobjdump = '/usr/local/cuda/bin/cuobjdump'
    if os.path.exists(cuobjdump):
        path = tmp_path / 'm.cubin'
        path.write_bytes(cubin)
        out = subprocess.run([cuobjdump, '-elf', str(path)], capture_output=True, text=True).stdout
        assert 'sm_100a' in out
        t = 'd' if dtype == _lib.F64 else 'f'
        model = f'10UserModelXI{t}Li{k + 1}ELi{k}EE'
        for lc in (32, 8, 1):
            for usig in (1, 0):
                assert f'k_model_chisqINS_{model}E{t}Li{lc}ELi1ELb{usig}E' in out, (lc, usig)
        assert f'k_model_eval_xINS_{model}' in out and 'mc3b_jit_abi' in out


def test_one_input_through_ex_is_the_plain_module():
    rc, cubin, _, _ = _compile(HORNER, 3, 1)
    assert rc == _lib.OK
    assert b'Li32ELi1ELb1E' in cubin and b'UserModelX' not in cubin


@pytest.mark.parametrize('k, line', [(2, 2), (3, 3)])
def test_arity_mismatch_fails_at_the_model_line(k, line):
    src = ''.join(f'__device__ real helper{i}(real a) {{ return a; }}\n' for i in range(line - 1))
    src += linear_source(k - 1 if k > 2 else 3)
    rc, _, log, _ = _compile(src, 4, k)
    assert rc == _lib.ERR_ARG
    assert f'model.cu({line})' in log
    with pytest.raises(ValueError, match=r'model\.cu\(%d\)' % line):
        jit.compile_cubin(src, 4, _lib.F64, 'arity', ninputs=k)


def test_ninputs_out_of_range():
    for k in (0, 5):
        with pytest.raises(ValueError, match='1 to 4 inputs'):
            CudaModel(HORNER, 3, ninputs=k)
        rc, _, _, err = _compile(HORNER, 3, k)
        assert rc == _lib.ERR_ARG and 'inputs' in err
    assert _lib.MAX_INPUTS == 4


def test_pickle_keeps_ninputs():
    m = CudaModel(linear_source(3), 4, name='lin3', ninputs=3)
    m2 = pickle.loads(pickle.dumps(m))
    assert (m2.source, m2.nparams, m2.name, m2.ninputs) == (m.source, 4, 'lin3', 3)
    one = pickle.loads(pickle.dumps(CudaModel(HORNER, 3, name='horner')))
    assert vars(one) == {'source': HORNER, 'nparams': 3, 'name': 'horner'} and one.ninputs == 1


def test_cache_key_of_one_input_is_unchanged():
    import hashlib
    src = linear_source(2)
    k = jit.cache_key(src, 3, _lib.F64)
    # the key as it was before models took several inputs
    h = hashlib.sha256()
    ver = jit.find_nvrtc()[1]
    for part in (src, '3', str(_lib.F64), str(_lib.load().mc3b_version()), f'{ver[0]}.{ver[1]}',
                 jit._headers_digest()):
        h.update(part.encode() + b'\0')
    assert k == h.hexdigest()
    assert k == jit.cache_key(src, 3, _lib.F64, ninputs=1)
    assert k != jit.cache_key(src, 3, _lib.F64, ninputs=2)
    assert jit.cache_key(src, 3, _lib.F64, ninputs=2) != jit.cache_key(src, 3, _lib.F64, ninputs=3)
    assert CudaModel(src, 3, ninputs=2).cache_key() == jit.cache_key(src, 3, _lib.F64, ninputs=2)
