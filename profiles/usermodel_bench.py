"""User models (mc3_b200.CudaModel) against the built-in kernels and TorchModel at the
config 2 shape: DEMC, 4096 chains, N = 1e5, fp64, one uncertainty for all points, on a
jittered abscissa (so that the sinusoid grid kernels stay out and every model runs
the general k_model_chisq).  Warm time per generation from CUDA events around
run(200), median of 3 runs; NVRTC compile time cold and from a CUBIN on disk.

    python profiles/usermodel_bench.py [--out profiles/r3_usermodel.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import mc3_b200 as mc3
from mc3_b200 import _lib, jit
from mc3_b200.engine import Population

NCH, N, GENS, REPS = 4096, 100_000, 200, 3

SRC = {
    'horner3': '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }',
    'gaussian': '''__device__ real model(real x, const real* p) {
    real d = (x - p[1]) / p[2];
    return p[0] * exp((real)-0.5 * d * d) + p[3];
}''',
    'sine_fast': '''__device__ real model(real x, const real* p) {
    return p[0] * fast_sin(6.283185307179586 / p[1] * x + p[2]) + p[3] + p[4] * x;
}''',
    'sine_lib': '''__device__ real model(real x, const real* p) {
    return p[0] * sin(6.283185307179586 / p[1] * x + p[2]) + p[3] + p[4] * x;
}''',
    'trapezoid': '''__device__ real model(real x, const real* p) {
    real z = fabs(x - p[1]) / p[2];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}''',
}


def t_poly(P, x):
    return P[:, 0:1] + x[None, :]*(P[:, 1:2] + x[None, :]*P[:, 2:3])


def t_gauss(P, x):
    return P[:, 0:1]*torch.exp(-0.5*((x[None, :] - P[:, 1:2])/P[:, 2:3])**2) + P[:, 3:4]


def t_sine(P, x):
    return P[:, 0:1]*torch.sin(2*np.pi*x[None, :]/P[:, 1:2] + P[:, 2:3]) + P[:, 3:4] + P[:, 4:5]*x[None, :]


def t_trap(P, x):
    z = (x[None, :] - P[:, 1:2]).abs()/P[:, 2:3]
    inner = torch.where(z < P[:, 4:5], (P[:, 4:5] - z)/(P[:, 4:5] - 1), torch.zeros_like(z))
    return P[:, 3:4] - P[:, 0:1]*torch.where(z < 1, torch.ones_like(z), inner)


def np_model(name, p, x):
    if name == 'poly':
        return p[0] + x*(p[1] + x*p[2])
    if name == 'gauss':
        return p[0]*np.exp(-0.5*((x - p[1])/p[2])**2) + p[3]
    if name == 'sine':
        return p[0]*np.sin(2*np.pi*x/p[1] + p[2]) + p[3] + p[4]*x
    z = np.abs(x - p[1])/p[2]
    return p[3] - p[0]*np.where(z < 1, 1.0, np.where(z < p[4], (p[4] - z)/(p[4] - 1), 0.0))


PROBLEMS = {   # truth, pstep
    'poly': (np.array([1.0, -0.3, 0.05]), np.array([1e-3, 1e-4, 1e-5])),
    'gauss': (np.array([2.0, 5.0, 1.2, 1.0]), np.array([1e-3, 1e-3, 1e-3, 1e-3])),
    'sine': (np.array([1.0, 2.5, 0.3, 5.0, -0.2]), np.array([1e-2, 1e-3, 1e-2, 1e-2, 1e-3])),
    'trap': (np.array([0.3, 5.0, 1.0, 1.0, 1.5]), np.array([1e-3, 1e-3, 1e-3, 1e-3, 1e-3])),
}


def timed(pop):
    pop.init_population('normal')
    pop.run(10)                                     # warm-up: modules, graphs, workspaces
    torch.cuda.synchronize()
    ms = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pop.run(GENS)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b)/GENS)
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.abspath(__file__)), 'r3_usermodel.json'))
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    path, ver = jit.find_nvrtc()
    res = {'shape': f'DEMC, {NCH} chains, N={N}, fp64, uniform sigma, jittered abscissa',
           'timing': f'CUDA events around run({GENS}) after run(10), median of {REPS}; ms per generation',
           'gpu': gpu[0] if gpu else None, 'cases': {},
           'nvrtc': f'{ver[0]}.{ver[1]} ' + ('(the nvidia-cuda-nvrtc wheel)' if 'cuda_nvrtc' in path else f'({path})')}
    rs = np.random.RandomState(7)
    dx = 10.0/(N - 1)
    x = np.sort(np.linspace(0, 10, N) + rs.uniform(-0.25, 0.25, N)*dx)
    cuda = {'poly': mc3.CudaModel(SRC['horner3'], 3, 'horner3'), 'gauss': mc3.CudaModel(SRC['gaussian'], 4, 'gauss'),
            'sine_fast': mc3.CudaModel(SRC['sine_fast'], 5, 'sine_fast'),
            'sine_lib': mc3.CudaModel(SRC['sine_lib'], 5, 'sine_lib'),
            'trap': mc3.CudaModel(SRC['trapezoid'], 5, 'trapezoid')}
    cases = [('poly', 'builtin polynomial(3)', mc3.models.polynomial),
             ('poly', 'CudaModel Horner', cuda['poly']),
             ('poly', 'TorchModel polynomial', mc3.TorchModel(t_poly)),
             ('gauss', 'builtin gaussian', mc3.models.gaussian),
             ('gauss', 'CudaModel gaussian', cuda['gauss']),
             ('gauss', 'TorchModel gaussian', mc3.TorchModel(t_gauss)),
             ('sine', 'builtin sinusoid (fast_sin, no grid)', mc3.models.sinusoid),
             ('sine', 'CudaModel sinusoid fast_sin', cuda['sine_fast']),
             ('sine', 'CudaModel sinusoid library sin', cuda['sine_lib']),
             ('sine', 'TorchModel sinusoid', mc3.TorchModel(t_sine)),
             ('trap', 'CudaModel trapezoid', cuda['trap']),
             ('trap', 'TorchModel trapezoid', mc3.TorchModel(t_trap))]
    data = {k: np_model(k, p, x) + rs.normal(0, 0.5, N) for k, (p, _) in PROBLEMS.items()}
    chk = {}
    for prob, label, func in cases:
        p0, step = PROBLEMS[prob]
        pop = Population(data[prob], np.full(N, 0.5), func, p0*1.001, [x], {}, step, None, None, None, None,
                         None, nchains=NCH, sampler='demc', fepsilon=0.01, hsize=2, thinning=1,
                         nzchain=10 + REPS*GENS, seed=3)
        assert not getattr(pop, 'grid', False) and not getattr(pop, 'use_moment', False)
        # the same 64 parameter vectors through every variant of a problem
        P = torch.as_tensor(p0*(1 + 1e-3*np.random.RandomState(1).normal(size=(64, p0.size))), device=pop.dev)
        c2 = pop.chisq(P).cpu().numpy()
        ms = timed(pop)
        ref = chk.setdefault(prob, c2)
        res['cases'][label] = {'ms_per_generation': float(np.median(ms)), 'runs_ms': ms,
                               'kind': pop.kind, 'graph': pop._graph is not None, 'fused': pop.fused,
                               'chisq_max_rel_diff_vs_first_variant': float(np.max(np.abs(c2 - ref)/ref))}
        print(label, res['cases'][label], flush=True)
        del pop
        torch.cuda.empty_cache()
    # compile times: cold (a source NVRTC has not seen) and from a CUBIN on disk
    comp = {}
    for name in ('horner3', 'trapezoid'):
        src = SRC[name] + f'\n// {time.time_ns()}'
        t0 = time.perf_counter()
        cubin = jit.compile_cubin(src, 3 if name == 'horner3' else 5, _lib.F64, name)
        cold = time.perf_counter() - t0
        with tempfile.TemporaryDirectory() as d:
            f = os.path.join(d, 'm.cubin')
            with open(f, 'wb') as fh:
                fh.write(cubin)
            t0 = time.perf_counter()
            with open(f, 'rb') as fh:
                h = jit._load(fh.read(), 3 if name == 'horner3' else 5, _lib.F64)
            disk = time.perf_counter() - t0
        assert h is not None and not isinstance(h, int)
        _lib.call('mc3b_user_model_free', h)
        comp[name] = {'cold_nvrtc_s': cold, 'from_disk_cache_s': disk, 'cubin_bytes': len(cubin)}
    res['compile'] = comp
    print(json.dumps(comp), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
