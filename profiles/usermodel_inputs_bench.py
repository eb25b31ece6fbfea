"""CudaModel of several per-point inputs against TorchModel at the config 2 shape: DEMC,
4096 chains, N = 1e5, one uncertainty for all points, jittered abscissa, fp64 and fp32.

Cases: the linear model p0 + sum_k p_k x_k for k = 1..4 inputs, and the 3-input
systematics transit trapezoid(t) * (1 + c1 xc + c2 yc + c3 xc yc), each as a CudaModel
and as a TorchModel (the torch formula computed in the run's dtype).  Warm time per
generation from CUDA events around run(GENS) after run(10), median of 3.  Also the
registers and static shared memory of the k = 4 kernels (cuobjdump -res-usage of the
CUBIN, the figures ptxas -v prints) and the GPU's name and power limit.

    python profiles/usermodel_inputs_bench.py [--out profiles/r3_usermodel_inputs.json]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import mc3_b200 as mc3
from mc3_b200 import _lib, jit
from mc3_b200.engine import Population

NCH, N, REPS = 4096, 100_000, 3
GENS = {'cuda': 200, 'torch': 40}


def linear_source(k):
    args = ', '.join(f'real x{j}' for j in range(k))
    body = ' + '.join(['p[0]'] + [f'p[{j + 1}] * x{j}' for j in range(k)])
    return f'__device__ real model({args}, const real* p) {{ return {body}; }}'


SYSTRANSIT = '''__device__ real trapezoid(real t, const real* p) {
    real z = fabs(t - p[1]) / p[2];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}
__device__ real model(real t, real xc, real yc, const real* p) {
    return trapezoid(t, p) * (1 + p[5]*xc + p[6]*yc + p[7]*xc*yc);
}'''


def t_linear(dt):
    def fn(P, *xs):
        P = P.to(dt)
        y = P[:, 0:1].expand(-1, xs[0].numel())
        for j, x in enumerate(xs):
            y = y + P[:, j + 1:j + 2]*x.to(dt)[None, :]
        return y
    return fn


def t_systransit(dt):
    def fn(P, t, xc, yc):
        P, t, xc, yc = P.to(dt), t.to(dt)[None, :], xc.to(dt)[None, :], yc.to(dt)[None, :]
        z = (t - P[:, 1:2]).abs()/P[:, 2:3]
        inner = torch.where(z < P[:, 4:5], (P[:, 4:5] - z)/(P[:, 4:5] - 1), torch.zeros_like(z))
        tr = P[:, 3:4] - P[:, 0:1]*torch.where(z < 1, torch.ones_like(z), inner)
        return tr*(1 + P[:, 5:6]*xc + P[:, 6:7]*yc + P[:, 7:8]*xc*yc)
    return fn


def timed(pop, gens):
    pop.init_population('normal')
    pop.run(10)                                     # warm-up: modules, graphs, workspaces
    torch.cuda.synchronize()
    ms = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pop.run(gens)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b)/gens)
    return ms


def resources(source, nmodel, ninputs, dtype):
    """Registers and static shared memory of every kernel of a compiled model."""
    cubin = jit.compile_cubin(source, nmodel, dtype, 'res', ninputs)
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, 'm.cubin')
        with open(f, 'wb') as fh:
            fh.write(cubin)
        out = subprocess.run(['cuobjdump', '-res-usage', f], capture_output=True, text=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.search(r'Function (\S+):', line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r'REG:(\d+).*SHARED:(\d+)', line)
        if m and name:
            lc = re.search(r'Li(\d+)ELi1ELb(\d)E', name)
            key = f'k_model_chisq LC={lc.group(1)} usig={lc.group(2)}' if lc else 'k_model_eval_x'
            regs, smem = int(m.group(1)), int(m.group(2))
            # CTAs of 128 threads per SM that registers (64 K) and shared memory (228 KB, 1 KB
            # reserved per CTA) allow; plan_shape plans for 6
            res[key] = {'registers': regs, 'static_smem_bytes': smem,
                        'ctas_per_sm_by_registers': 65536//(128*((regs + 7)//8*8)),
                        'ctas_per_sm_by_smem': 233472//(smem + 1024)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                  'r3_usermodel_inputs.json'))
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {'shape': f'DEMC, {NCH} chains, N={N}, uniform sigma, jittered abscissa',
           'timing': f'CUDA events around run(G) after run(10), median of {REPS}; ms per generation; '
                     f'G = {GENS["cuda"]} (CudaModel), {GENS["torch"]} (TorchModel)',
           'gpu': gpu[0] if gpu else None, 'cases': {}}
    rs = np.random.RandomState(7)
    dx = 0.4/(N - 1)
    t = np.sort(np.linspace(-0.2, 0.2, N) + rs.uniform(-0.25, 0.25, N)*dx)
    regs = [t] + [rs.normal(0, 0.3, N) for _ in range(3)]
    ptr = np.array([0.01, 0.002, 0.05, 1.0, 1.6, 1e-3, -2e-3, 5e-4])
    problems = {}
    for k in range(1, 5):
        p = np.array([1.0] + [0.1*(j + 1) for j in range(k)])
        problems[f'linear k={k}'] = (linear_source(k), p, regs[:k], t_linear)
    problems['systransit k=3'] = (SYSTRANSIT, ptr, regs[:3], t_systransit)
    for dtype, dt in (('f64', torch.float64), ('f32', torch.float32)):
        for label, (src, p0, xs, tfn) in problems.items():
            if label.startswith('linear'):
                data = p0[0] + sum(p0[j + 1]*x for j, x in enumerate(xs))
            else:
                z = np.abs(xs[0] - p0[1])/p0[2]
                tr = p0[3] - p0[0]*np.where(z < 1, 1.0, np.where(z < p0[4], (p0[4] - z)/(p0[4] - 1), 0.0))
                data = tr*(1 + p0[5]*xs[1] + p0[6]*xs[2] + p0[7]*xs[1]*xs[2])
            unc = np.full(N, 1e-3)
            data = data + rs.normal(0, 1, N)*unc
            step = 1e-4*np.maximum(np.abs(p0), 1e-2)
            chk = None
            for kind, func in (('cuda', mc3.CudaModel(src, p0.size, label, ninputs=len(xs))),
                               ('torch', mc3.TorchModel(tfn(dt)))):
                pop = Population(data, unc, func, p0*1.0001, xs, {}, step, None, None, None, None, None,
                                 nchains=NCH, sampler='demc', fepsilon=0.01, hsize=2, thinning=1,
                                 nzchain=10 + REPS*GENS[kind], seed=3, dtype=dtype)
                P = torch.as_tensor(p0*(1 + 1e-4*np.random.RandomState(1).normal(size=(64, p0.size))),
                                    device=pop.dev)
                c2 = pop.chisq(P).cpu().numpy()
                chk = c2 if chk is None else chk
                ms = timed(pop, GENS[kind])
                name = f'{dtype} {label} {"CudaModel" if kind == "cuda" else "TorchModel"}'
                res['cases'][name] = {'ms_per_generation': float(np.median(ms)), 'runs_ms': ms, 'kind': pop.kind,
                                      'fused': pop.fused,
                                      'chisq_max_rel_diff_vs_cudamodel': float(np.max(np.abs(c2 - chk)/chk))}
                print(name, res['cases'][name], flush=True)
                del pop
                torch.cuda.empty_cache()
    res['k4_kernels'] = {d: resources(linear_source(4), 5, 4, dt) for d, dt in (('f64', _lib.F64), ('f32', _lib.F32))}
    res['k1_kernels'] = {d: resources(linear_source(1), 2, 1, dt) for d, dt in (('f64', _lib.F64), ('f32', _lib.F32))}
    print(json.dumps(res['k4_kernels']), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
