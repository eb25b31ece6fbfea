"""CPU-only: the fp64 module of a user model carries the wavelet likelihood's D4 kernels
that read the model (k_dwt_reg_model, k_dwt_pass and k_dwt_last of dwt_kernel.cuh) under
the names the loader derives; an fp32 module carries none; the register stage of a model
of one and of four inputs keeps everything in registers."""
import ctypes
import os
import subprocess

import pytest

from mc3_b200 import _lib
from mc3_b200 import jit

try:
    NVRTC = jit.find_nvrtc()[0]
except _lib.Mc3bError:
    NVRTC = None
pytestmark = pytest.mark.skipif(NVRTC is None, reason='no NVRTC 12.8+ found')
CUOBJDUMP = '/usr/local/cuda/bin/cuobjdump'

HORNER = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'


def inputs_source(k, nconst=0):
    """p[0] + p[1] x_0 + ... over k inputs; with constants, scaled by their sum, which
    prepare keeps in the work slot."""
    args = ', '.join(f'real x{j}' for j in range(k))
    body = ' + '.join(['p[0]'] + [f'p[{j + 1}] * x{j}' for j in range(k)])
    if not nconst:
        return f'__device__ real model({args}, const real* p) {{ return {body}; }}'
    csum = ' + '.join(f'p[{k + 1 + j}]' for j in range(nconst))
    return (f'__device__ void prepare(real* p) {{ p[{k + 1 + nconst}] = {csum}; }}\n'
            f'__device__ real model({args}, const real* p) {{ return ({body}) * p[{k + 1 + nconst}]; }}')


def _compile(source, nmodel, ninputs=1, nconst=0, nwork=0, dtype=_lib.F64, cap=1 << 23):
    lib = _lib.load()
    buf = ctypes.create_string_buffer(cap)
    size = ctypes.c_int64(-1)
    log = ctypes.create_string_buffer(1 << 16)
    desc = _lib.UserModelDesc(nmodel, ninputs, nconst, nwork, dtype)
    rc = lib.mc3b_user_model_compile_desc(NVRTC.encode(), source.encode(), ctypes.byref(desc), buf, cap,
                                          ctypes.byref(size), log, len(log))
    assert rc == _lib.OK, (lib.mc3b_last_error().decode(), log.value.decode())
    return buf.raw[:size.value]


def _dump(cubin, tmp_path, what):
    if not os.path.exists(CUOBJDUMP):
        pytest.skip('no cuobjdump')
    path = tmp_path / 'm.cubin'
    path.write_bytes(cubin)
    return subprocess.run([CUOBJDUMP, what, str(path)], capture_output=True, text=True, check=True).stdout


def dwt_symbols(wrapper):
    """The loader's names (jit.cu dwt_symbol) for the Itanium-mangled wrapper type."""
    return ['_ZN8mc3b_jit15k_dwt_reg_modelINS_' + wrapper + 'ENS_8RegArgsXEEEvT0_',
            '_ZN8mc3b_jit10k_dwt_passILi0ENS_' + wrapper + 'ENS_9PassArgsXEEEvT1_',
            '_ZN8mc3b_jit10k_dwt_lastILi0ENS_' + wrapper + 'ENS_9LastArgsXEEEvT1_']


@pytest.mark.parametrize('case', ['one_input', 'three_inputs_consts_prepare'])
def test_fp64_module_carries_the_d4_kernels(case, tmp_path):
    # compile_desc also checks NVRTC's lowered names against the loader's and fails on a
    # mismatch, so the compile itself covers that
    if case == 'one_input':
        cubin, wrapper = _compile(HORNER, 3), '9UserModelIdLi3EE'
    else:
        cubin, wrapper = _compile(inputs_source(3, 2), 4, 3, 2, 1), '10UserModelKIdLi4ELi3ELi2ELi1EE'
    out = _dump(cubin, tmp_path, '-elf')
    for sym in dwt_symbols(wrapper):
        assert sym in out, sym


def test_fp32_module_has_no_d4_kernels(tmp_path):
    out = _dump(_compile(HORNER, 3, dtype=_lib.F32), tmp_path, '-elf')
    assert 'k_model_chisq' in out and 'k_dwt' not in out


@pytest.mark.parametrize('k', [1, 4])
def test_register_stage_has_no_local_memory(k, tmp_path):
    src = HORNER if k == 1 else inputs_source(k)
    cubin = _compile(src, 3 if k == 1 else k + 1, k)
    out = _dump(cubin, tmp_path, '--dump-resource-usage')
    lines = out.splitlines()
    i = next(i for i, line in enumerate(lines) if 'k_dwt_reg_model' in line)
    usage = lines[i + 1]
    assert 'STACK:0 ' in usage and 'LOCAL:0 ' in usage, usage
