"""CPU-only: user models (mc3_b200.CudaModel) compile to sm_100a CUBINs through the
library's NVRTC entry point without a device; compile errors, a missing `model`,
a small buffer and the NVRTC discovery order behave as documented; the model object
pickles as its source; the cache key tracks source, parameter count and dtype."""
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


def _compile(source, nmodel=3, dtype=_lib.F64, cap=1 << 22):
    lib = _lib.load()
    buf = ctypes.create_string_buffer(max(cap, 1))
    size = ctypes.c_int64(-1)
    log = ctypes.create_string_buffer(1 << 16)
    rc = lib.mc3b_user_model_compile(NVRTC.encode(), source.encode(), nmodel, dtype, buf, cap,
                                     ctypes.byref(size), log, len(log))
    return rc, buf.raw[:max(size.value, 0)], size.value, log.value.decode()


@pytest.mark.parametrize('dtype', [_lib.F64, _lib.F32])
def test_valid_source_compiles_to_sm100a_cubin(dtype, tmp_path):
    rc, cubin, size, _ = _compile(HORNER, dtype=dtype)
    assert rc == _lib.OK and size > 0 and cubin[:4] == b'\x7fELF'
    path = tmp_path / 'm.cubin'
    path.write_bytes(cubin)
    cuobjdump = '/usr/local/cuda/bin/cuobjdump'
    if os.path.exists(cuobjdump):
        out = subprocess.run([cuobjdump, '-elf', str(path)], capture_output=True, text=True).stdout
        assert 'sm_100a' in out
        for lc in (32, 8, 1):
            assert f'Li{lc}ELi1ELb1E' in out and f'Li{lc}ELi1ELb0E' in out
        assert 'k_model_eval' in out and 'mc3b_jit_abi' in out


def test_syntax_error_names_the_line():
    src = ('__device__ real helper(real x) { return x; }\n'
           '__device__ real model(real x, const real* p) {\n'
           '    return p[0] * x +;\n'
           '}\n')
    rc, _, _, log = _compile(src)
    assert rc == _lib.ERR_ARG
    assert 'model.cu(3)' in log


def test_source_without_model_is_refused():
    rc, _, _, log = _compile('__device__ real f(real x, const real* p) { return p[0]; }')
    assert rc == _lib.ERR_ARG and 'model' in log
    with pytest.raises(ValueError, match='model'):
        jit.compile_cubin('__device__ double g(double x) { return x; }', 1, _lib.F64)


def test_size_reported_when_buffer_too_small():
    rc, _, size, _ = _compile(HORNER, cap=16)
    assert rc == _lib.ERR_ARG and size > 16
    rc2, cubin, size2, _ = _compile(HORNER, cap=size)
    assert rc2 == _lib.OK and size2 == size and len(cubin) == size


def test_compile_error_raises_value_error_with_log():
    with pytest.raises(ValueError, match='undefined'):
        jit.compile_cubin('__device__ real model(real x, const real* p) { return undefined_thing(x); }',
                          1, _lib.F64, 'broken')


def test_discovery_honours_mc3b_nvrtc(monkeypatch):
    cands = [c for c in jit.nvrtc_candidates() if os.path.exists(c)]
    assert cands
    pick = cands[-1]
    monkeypatch.setenv('MC3B_NVRTC', pick)
    assert jit.nvrtc_candidates() == [pick]
    assert jit.find_nvrtc()[0] == pick
    monkeypatch.setenv('MC3B_NVRTC', '/nonexistent/libnvrtc.so.12')
    with pytest.raises(_lib.Mc3bError, match='/nonexistent/libnvrtc.so.12'):
        jit.find_nvrtc()
    monkeypatch.delenv('MC3B_NVRTC')
    order = jit.nvrtc_candidates()
    wheel = [i for i, c in enumerate(order) if 'cuda_nvrtc' in c]
    system = order.index('/usr/local/cuda/lib64/libnvrtc.so.12')
    assert not wheel or max(wheel) < system
    assert order[-1] == 'libnvrtc.so.12'


def test_library_refuses_old_or_missing_nvrtc():
    lib = _lib.load()
    size = ctypes.c_int64(0)
    rc = lib.mc3b_user_model_compile(b'/nonexistent/libnvrtc.so.12', HORNER.encode(), 3, _lib.F64, None, 0,
                                     ctypes.byref(size), None, 0)
    assert rc == _lib.ERR_CUDA
    assert 'nonexistent' in lib.mc3b_last_error().decode()


def test_cuda_model_pickles_without_handle():
    m = CudaModel(HORNER, 3, name='horner')
    m2 = pickle.loads(pickle.dumps(m))
    assert vars(m2) == {'source': HORNER, 'nparams': 3, 'name': 'horner'}
    with pytest.raises(ValueError):
        CudaModel(HORNER, 0)
    with pytest.raises(ValueError, match='takes 3'):
        m.nmodel(4)


def test_cache_key_tracks_source_nparams_dtype():
    k = jit.cache_key(HORNER, 3, _lib.F64)
    assert k == jit.cache_key(HORNER, 3, _lib.F64)
    assert k != jit.cache_key(HORNER + ' ', 3, _lib.F64)
    assert k != jit.cache_key(HORNER, 4, _lib.F64)
    assert k != jit.cache_key(HORNER, 3, _lib.F32)
