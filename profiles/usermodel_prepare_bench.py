"""CudaModels with a prepare step and run-time constants against the built-in models at
the r3_usermodel shape: DEMC, 4096 chains, N = 1e5, one uncertainty for all points,
jittered abscissa (so that the sinusoid grid kernels stay out), fp64 and fp32.

Variants: the built-in Gaussian, and the Gaussian CudaModel without and with a prepare
that hoists 1/sigma; the built-in sinusoid, and the sinusoid CudaModel (mathx<real>::sin_:
fast_sin in fp64, sinf in fp32, as the built-in) without and with a prepare that hoists
2 pi/P; the trapezoid transit folded on a period given as a constant; the built-in
polynomial and the Horner CudaModel.  Time per generation from CUDA events around run(G)
after run(10); the variants of a dtype take turns, REPS rounds, so that a drift of the
machine spreads over all of them.  Also the cold NVRTC compile of a model with and without
a prepare step, and the GPU's name and power limit, read in the same run.

    python profiles/usermodel_prepare_bench.py [--out profiles/r3_usermodel_prepare.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import mc3_b200 as mc3
from mc3_b200 import _lib, jit
from mc3_b200.engine import Population

NCH, N, GENS, REPS = 4096, 100_000, 200, 5
PERIOD = 3.7

SRC = {
    'horner3': '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }',
    'gauss': '''__device__ real model(real x, const real* p) {
    real d = (x - p[1]) / p[2];
    return p[0] * exp((real)-0.5 * d * d) + p[3];
}''',
    'gauss_prepare': '''__device__ void prepare(real* p) { p[4] = 1 / p[2]; }
__device__ real model(real x, const real* p) {
    real d = (x - p[1]) * p[4];
    return fma(p[0], exp((real)(-0.5) * d * d), p[3]);
}''',
    'sine': '''__device__ real model(real x, const real* p) {
    return fma(p[0], mathx<real>::sin_(fma(x, (real)6.283185307179586 / p[1], p[2])), fma(p[4], x, p[3]));
}''',
    'sine_prepare': '''__device__ void prepare(real* p) { p[5] = (real)6.283185307179586 / p[1]; }
__device__ real model(real x, const real* p) {
    return fma(p[0], mathx<real>::sin_(fma(x, p[5], p[2])), fma(p[4], x, p[3]));
}''',
    # p[5]: the period (a constant), p[6]: 1/period
    'ptrapezoid': '''__device__ void prepare(real* p) { p[6] = 1 / p[5]; }
__device__ real model(real x, const real* p) {
    real dt = x - p[1];
    dt -= p[5] * rint(dt * p[6]);
    real z = fabs(dt) / p[2];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}''',
}


def np_model(name, p, x):
    if name == 'poly':
        return p[0] + x*(p[1] + x*p[2])
    if name == 'gauss':
        return p[0]*np.exp(-0.5*((x - p[1])/p[2])**2) + p[3]
    if name == 'sine':
        return p[0]*np.sin(2*np.pi*x/p[1] + p[2]) + p[3] + p[4]*x
    dt = x - p[1]
    dt = dt - PERIOD*np.rint(dt/PERIOD)
    z = np.abs(dt)/p[2]
    return p[3] - p[0]*np.where(z < 1, 1.0, np.where(z < p[4], (p[4] - z)/(p[4] - 1), 0.0))


PROBLEMS = {   # truth, pstep
    'poly': (np.array([1.0, -0.3, 0.05]), np.array([1e-3, 1e-4, 1e-5])),
    'gauss': (np.array([2.0, 5.0, 1.2, 1.0]), np.array([1e-3, 1e-3, 1e-3, 1e-3])),
    'sine': (np.array([1.0, 2.5, 0.3, 5.0, -0.2]), np.array([1e-2, 1e-3, 1e-2, 1e-2, 1e-3])),
    'ptrap': (np.array([0.3, 1.0, 0.3, 1.0, 1.5]), np.array([1e-3, 1e-3, 1e-3, 1e-3, 1e-3])),
}


def gen_ms(pop):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    pop.run(GENS)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)/GENS


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                  'r3_usermodel_prepare.json'))
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    path, ver = jit.find_nvrtc()
    res = {'shape': f'DEMC, {NCH} chains, N={N}, uniform sigma, jittered abscissa',
           'timing': f'CUDA events around run({GENS}) after run(10); the variants of a dtype alternate, '
                     f'{REPS} rounds; ms per generation, median and every round',
           'gpu': gpu[0] if gpu else None, 'cases': {},
           'nvrtc': f'{ver[0]}.{ver[1]} ' + ('(the nvidia-cuda-nvrtc wheel)' if 'cuda_nvrtc' in path else f'({path})')}
    rs = np.random.RandomState(7)
    dx = 10.0/(N - 1)
    x = np.sort(np.linspace(0, 10, N) + rs.uniform(-0.25, 0.25, N)*dx)
    data = {k: np_model(k, p, x) + rs.normal(0, 0.5, N) for k, (p, _) in PROBLEMS.items()}
    cuda = {'poly': mc3.CudaModel(SRC['horner3'], 3, 'horner3'),
            'gauss': mc3.CudaModel(SRC['gauss'], 4, 'gauss'),
            'gauss_prepare': mc3.CudaModel(SRC['gauss_prepare'], 4, 'gauss_prepare', nwork=1),
            'sine': mc3.CudaModel(SRC['sine'], 5, 'sine'),
            'sine_prepare': mc3.CudaModel(SRC['sine_prepare'], 5, 'sine_prepare', nwork=1),
            'ptrap': mc3.CudaModel(SRC['ptrapezoid'], 5, 'ptrapezoid', nconst=1, nwork=1)}
    cases = [('poly', 'builtin polynomial(3)', mc3.models.polynomial, []),
             ('poly', 'CudaModel Horner', cuda['poly'], []),
             ('gauss', 'builtin gaussian', mc3.models.gaussian, []),
             ('gauss', 'CudaModel gaussian', cuda['gauss'], []),
             ('gauss', 'CudaModel gaussian + prepare', cuda['gauss_prepare'], []),
             ('sine', 'builtin sinusoid (no grid)', mc3.models.sinusoid, []),
             ('sine', 'CudaModel sinusoid', cuda['sine'], []),
             ('sine', 'CudaModel sinusoid + prepare', cuda['sine_prepare'], []),
             ('ptrap', 'CudaModel trapezoid, period a constant', cuda['ptrap'], [PERIOD])]
    for dtype in ('f64', 'f32'):
        pops, chk = {}, {}
        for prob, label, func, consts in cases:
            p0, step = PROBLEMS[prob]
            pop = Population(data[prob], np.full(N, 0.5), func, p0*1.001, [x] + consts, {}, step, None, None, None,
                             None, None, nchains=NCH, sampler='demc', fepsilon=0.01, hsize=2, thinning=1,
                             nzchain=10 + REPS*GENS, seed=3, dtype=dtype)
            assert not getattr(pop, 'grid', False) and not getattr(pop, 'use_moment', False)
            # the same 64 parameter vectors through every variant of a problem
            P = torch.as_tensor(p0*(1 + 1e-3*np.random.RandomState(1).normal(size=(64, p0.size))), device=pop.dev)
            c2 = pop.chisq(P).cpu().numpy()
            want = np.array([np.sum(((np_model(prob, p, x) - data[prob])/0.5)**2) for p in P.cpu().numpy()])
            ref = chk.setdefault(prob, c2)
            pop.init_population('normal')
            pop.run(10)                             # warm-up: modules, graphs, workspaces
            torch.cuda.synchronize()
            pops[label] = pop
            res['cases'][f'{dtype} {label}'] = {
                'kind': pop.kind, 'fused': pop.fused, 'runs_ms': [],
                'chisq_max_rel_diff_vs_first_variant': float(np.max(np.abs(c2 - ref)/ref)),
                'chisq_max_rel_diff_vs_numpy': float(np.max(np.abs(c2 - want)/want))}
        for _ in range(REPS):
            for _, label, _, _ in cases:
                res['cases'][f'{dtype} {label}']['runs_ms'].append(gen_ms(pops[label]))
        for _, label, _, _ in cases:
            r = res['cases'][f'{dtype} {label}']
            r['ms_per_generation'] = float(np.median(r['runs_ms']))
            print(dtype, label, r, flush=True)
        del pops
        torch.cuda.empty_cache()
    # cold compiles: a source NVRTC has not seen (a unique comment), with and without prepare
    comp = {}
    for name, nmodel, nwork in (('gauss', 4, 0), ('gauss_prepare', 4, 1)):
        times = []
        for _ in range(3):
            src = SRC[name] + f'\n// {time.time_ns()}'
            t0 = time.perf_counter()
            jit.compile_cubin(src, nmodel, _lib.F64, name, nwork=nwork)
            times.append(time.perf_counter() - t0)
        comp[name] = {'cold_nvrtc_s': times}
    res['compile'] = comp
    print(json.dumps(comp), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
