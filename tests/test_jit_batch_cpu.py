"""CPU-only: the batch module of a user model (CudaModel.batch_handle, mc3b_user_batch_*)
compiles to an sm_100a CUBIN whose kernels carry the names the loader derives, for one and
three inputs, with and without constants and prepare; the user k_run_batch of the README's
transit models uses no local memory and no stack; the batch module has its own ABI record
and its own cache key, and the key of the sample() module keeps its formula; work slots
without a prepare, and fp32, are refused."""
import ctypes
import hashlib
import os
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
CUOBJDUMP = '/usr/local/cuda/bin/cuobjdump'

HORNER = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
# the README's trapezoid transit, its 3-input systematics transit, and its transit on a known
# period and exposure time (p[5], p[6]; prepare keeps 1/period and the widened half duration)
TRAPEZOID = '''__device__ real model(real x, const real* p) {
    real z = fabs(x - p[1]) / p[2];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}'''
SYSTRANSIT = '''__device__ real model(real t, real xc, real yc, const real* p) {
    real z = fabs(t - p[1]) / p[2];
    real transit = p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
    return transit * (1 + p[5]*xc + p[6]*yc + p[7]*xc*yc);
}'''
PTRANSIT = '''__device__ void prepare(real* p) { p[7] = 1 / p[5]; p[8] = p[2] + (real)0.5 * p[6]; }
__device__ real model(real x, const real* p) {
    real dt = x - p[1];
    dt -= p[5] * rint(dt * p[7]);
    real z = fabs(dt) / p[8];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}'''
README_MODELS = {'trapezoid': (TRAPEZOID, 5, 1, 0, 0), 'systransit': (SYSTRANSIT, 8, 3, 0, 0),
                 'period transit': (PTRANSIT, 5, 1, 2, 2)}


def consts_source(k, nconst):
    """p[0] + p[1] x_0 + ... over k inputs, scaled by the sum of nconst constants; prepare
    keeps that sum in the work slot."""
    args = ', '.join(f'real x{j}' for j in range(k))
    body = ' + '.join(['p[0]'] + [f'p[{j + 1}] * x{j}' for j in range(k)])
    csum = ' + '.join(f'p[{k + 1 + j}]' for j in range(nconst))
    return (f'__device__ void prepare(real* p) {{ p[{k + 1 + nconst}] = {csum}; }}\n'
            f'__device__ real model({args}, const real* p) {{ return ({body}) * p[{k + 1 + nconst}]; }}')


def linear_source(k):
    args = ', '.join(f'real x{j}' for j in range(k))
    body = ' + '.join(['p[0]'] + [f'p[{j + 1}] * x{j}' for j in range(k)])
    return f'__device__ real model({args}, const real* p) {{ return {body}; }}'


def _compile(source, nmodel, ninputs=1, nconst=0, nwork=0, dtype=_lib.F64, cap=1 << 22):
    lib = _lib.load()
    buf = ctypes.create_string_buffer(max(cap, 1))
    size = ctypes.c_int64(-1)
    log = ctypes.create_string_buffer(1 << 16)
    desc = _lib.UserModelDesc(nmodel, ninputs, nconst, nwork, dtype)
    rc = lib.mc3b_user_batch_compile(NVRTC.encode(), source.encode(), ctypes.byref(desc), buf, cap,
                                     ctypes.byref(size), log, len(log))
    return rc, buf.raw[:max(size.value, 0)], log.value.decode(), lib.mc3b_last_error().decode()


def _cuobjdump(cubin, tmp_path, flag):
    if not os.path.exists(CUOBJDUMP):
        pytest.skip('no cuobjdump')
    path = tmp_path / 'm.cubin'
    path.write_bytes(cubin)
    return subprocess.run([CUOBJDUMP, flag, str(path)], capture_output=True, text=True).stdout


@pytest.mark.parametrize('k', [1, 3])
@pytest.mark.parametrize('consts', [False, True])
def test_batch_module_compiles_to_sm100a_cubin(k, consts, tmp_path):
    # the compile checks NVRTC's lowered names against the symbols the loader looks up and
    # fails (MC3B_ERR_CUDA) on any mismatch, so rc == OK covers that check
    if consts:
        src, desc, model = consts_source(k, 2), (k + 1, k, 2, 1), f'10UserModelKIdLi{k + 1}ELi{k}ELi2ELi1EE'
    else:
        src, desc = linear_source(k), (k + 1, k, 0, 0)
        model = f'9UserModelIdLi{k + 1}EE' if k == 1 else f'10UserModelXIdLi{k + 1}ELi{k}EE'
    rc, cubin, log, err = _compile(src, *desc)
    assert rc == _lib.OK, (err, log)
    out = _cuobjdump(cubin, tmp_path, '-elf')
    assert 'sm_100a' in out and 'mc3b_jit_batch_abi' in out and 'mc3b_jit_abi' not in out
    for kernel in ('12k_init_batch', '11k_run_batch', '12k_batch_eval'):
        assert f'_ZN8mc3b_jit{kernel}INS_{model}' in out, kernel
    assert 'k_model_chisq' not in out                 # the sample() kernels stay in their own module


@pytest.mark.parametrize('name', sorted(README_MODELS))
def test_readme_models_run_without_local_memory(name, tmp_path):
    rc, cubin, log, err = _compile(*README_MODELS[name])
    assert rc == _lib.OK, (err, log)
    lines = _cuobjdump(cubin, tmp_path, '-res-usage').splitlines()
    usage = [lines[i + 1] for i, line in enumerate(lines) if '11k_run_batch' in line]
    assert len(usage) == 1
    assert 'LOCAL:0' in usage[0] and 'STACK:0' in usage[0], usage[0]


def test_work_slots_without_prepare_and_f32_are_refused():
    rc, _, log, err = _compile(HORNER, 3, nwork=1)
    assert rc == _lib.ERR_ARG and 'prepare' in err and 'prepare' in log
    with pytest.raises(ValueError, match='prepare'):
        jit.compile_cubin(HORNER, 3, _lib.F64, 'nowork', nwork=2, kind='batch')
    rc, _, _, err = _compile(HORNER, 3, dtype=_lib.F32)
    assert rc == _lib.ERR_ARG and 'fp64 only' in err


def test_a_module_of_one_kind_does_not_load_as_the_other():
    lib = _lib.load()
    desc = _lib.UserModelDesc(3, 1, 0, 0, _lib.F64)
    chisq = jit.compile_cubin(HORNER, 3, _lib.F64, 'horner')
    batch = jit.compile_cubin(HORNER, 3, _lib.F64, 'horner', kind='batch')
    assert chisq != batch
    h = ctypes.c_void_p()
    # without a device the load fails before the ABI check; with one, at the ABI record
    assert lib.mc3b_user_batch_load(chisq, len(chisq), ctypes.byref(desc), ctypes.byref(h)) != _lib.OK
    assert lib.mc3b_user_model_load_desc(batch, len(batch), ctypes.byref(desc), ctypes.byref(h)) != _lib.OK


def test_batch_cache_key_is_its_own():
    h = hashlib.sha256()
    ver = jit.find_nvrtc()[1]
    for part in (HORNER, '3', str(_lib.F64), str(_lib.load().mc3b_version()), f'{ver[0]}.{ver[1]}',
                 jit._headers_digest()):
        h.update(part.encode() + b'\0')
    m = CudaModel(HORNER, 3)
    assert m.cache_key() == h.hexdigest() == jit.cache_key(HORNER, 3, _lib.F64)
    h.update(b'kind=batch\0')
    assert jit.cache_key(HORNER, 3, _lib.F64, kind='batch') == h.hexdigest() != m.cache_key()
    keys = {jit.cache_key(HORNER, 3, _lib.F64, 1, c, w, kind) for c in (0, 1) for w in (0, 1)
            for kind in ('chisq', 'batch')}
    assert len(keys) == 8
