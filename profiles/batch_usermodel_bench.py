"""sample_batch with a CudaModel (README "Many small fits at once").

    python profiles/batch_usermodel_bench.py [--out profiles/r10_batch_usermodel.json]

Three measurements, in one process, with the GPU's name, power limit and max SM clock:
  builtin_vs_cuda   generations time (device events around the k_run_batch launches) of
                    CudaModel(HORNER3) against the built-in polynomial at config 1's shape
                    (quadratic, snooker, 7 chains, N = 100, 1e5 samples), B = 148 and 4736;
                    the two alternate, twice each.  The state is the same bit for bit
                    (tests/test_gpu_batch_usermodel.py); the user kernel runs under its own
                    register bound (batch_dev.cuh BATCH_BLOCKS).
  period_transit    the trapezoid transit on a known period and exposure time (run-time
                    constants, a prepare step; N = 2000, 32 chains, DEMC, 6.4e4 samples),
                    B = 148 and 1184: wall time of sample_batch against 8 sequential sample()
                    calls of the same CudaModel timed after a warm-up call and extrapolated
                    to B (labelled as such).
  compile           seconds to the batch module of a model not compiled before: cold (NVRTC)
                    and from the MC3B_JIT_CACHE directory; the sample() module for reference.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mc3_b200 as mc3                      # noqa: E402
from mc3_b200 import batch_driver, jit      # noqa: E402
from oracle import problems as pb           # noqa: E402

HORNER3 = '__device__ real model(real x, const real* p) { return fma(fma(p[2], x, p[1]), x, p[0]); }'
# p[5] = period, p[6] = exposure time (constants); p[7] = 1/period, p[8] = half duration
# widened by half the exposure (prepare)
PTRANSIT = '''__device__ void prepare(real* p) { p[7] = 1 / p[5]; p[8] = p[2] + (real)0.5 * p[6]; }
__device__ real model(real x, const real* p) {
    real dt = x - p[1];
    dt -= p[5] * rint(dt * p[7]);
    real z = fabs(dt) / p[8];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}'''


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def generations_time(func, B):
    """Seconds of the k_run_batch launches of one sample_batch at config 1's shape."""
    rs = np.random.RandomState(B)
    p = pb.mcmc_case('quad')
    data = [p['data'] + rs.normal(0, 1e-3, p['data'].size)*p['uncert'] for _ in range(B)]
    R = batch_driver._BatchRun
    orig = R.run
    t = {}

    def run(self_, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(self_, *a)
        e1.record()
        e1.synchronize()
        t['s'] = e0.elapsed_time(e1)/1e3
    R.run = run
    try:
        mc3.sample_batch(data, [p['uncert']]*B, func, np.tile(p['params'], (B, 1)), [[p['x']]]*B, pstep=p['pstep'],
                         sampler='snooker', nchains=7, nsamples=1e5, burnin=1000, seed=1, _state=True)
    finally:
        R.run = orig
    return t['s']


def transit_workload(B):
    rs = np.random.RandomState(B)
    x = np.linspace(0.0, 10.0, 2000)
    period, exptime = 3.0, 0.01
    truth = np.array([0.01, 0.4, 0.1, 1.0, 1.3])
    m = mc3.CudaModel(PTRANSIT, 5, name='period_transit', nconst=2, nwork=2)
    clean = m(truth, x, period, exptime)
    data = [clean + rs.normal(0, 1e-3, x.size) for _ in range(B)]
    return dict(data=data, uncert=[np.full(x.size, 1e-3)]*B, func=m, params=np.tile(truth*1.01, (B, 1)),
                indparams=[[x, period, exptime]]*B, pstep=np.array([1e-4, 1e-3, 1e-3, 1e-4, 0.0]),
                pmin=np.array([0.0, 0.2, 0.01, 0.9, 1.0]), pmax=np.array([0.05, 0.6, 0.3, 1.1, 2.0]),
                sampler='demc', nchains=32, nsamples=6.4e4, burnin=0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    lines = []

    def emit(line):
        line = dict(gpu=info, **line)
        print(json.dumps(line), flush=True)
        lines.append(line)

    # compile times first: nothing of these models is in memory yet
    cache = tempfile.mkdtemp(prefix='mc3b_jit_')
    os.environ['MC3B_JIT_CACHE'] = cache
    src = PTRANSIT + '\n// compile-time probe\n'
    for kind in ('batch', 'chisq'):
        st = {}
        jit.handle(src, 5, mc3._lib.F64, 'probe', st, 1, 2, 2, kind=kind)
        cold = dict(st)
        jit._HANDLES.pop(jit.cache_key(src, 5, mc3._lib.F64, 1, 2, 2, kind))
        jit.forget()
        st = {}
        jit.handle(src, 5, mc3._lib.F64, 'probe', st, 1, 2, 2, kind=kind)
        emit(dict(case='compile', module=kind, cold_origin=cold['origin'], cold_s=cold['seconds'],
                  cache_origin=st['origin'], cache_s=st['seconds']))

    um = mc3.CudaModel(HORNER3, 3, name='horner')
    generations_time(mc3.models.polynomial, 148)           # warm-up: library and module loads
    generations_time(um, 148)
    for B in (148, 4736):
        t = {'builtin': [], 'cuda': []}
        for _ in range(2):
            t['builtin'].append(generations_time(mc3.models.polynomial, B))
            t['cuda'].append(generations_time(um, B))
        emit(dict(case='builtin_vs_cuda', B=B, builtin_generations_s=t['builtin'], cuda_generations_s=t['cuda'],
                  ratio_cuda_over_builtin=min(t['cuda'])/min(t['builtin'])))

    w = transit_workload(8)
    quiet = mc3.Log(verb=-1)
    opts = {k: w[k] for k in ('pstep', 'pmin', 'pmax', 'sampler', 'nchains', 'nsamples', 'burnin')}

    def call(b):
        return mc3.sample(w['data'][b], w['uncert'][b], func=w['func'], params=w['params'][b],
                          indparams=w['indparams'][b], seed=1 + b, log=quiet, **opts)
    call(0)                                                # warm-up (module load, first allocations)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in range(8):
        call(b)
    torch.cuda.synchronize()
    seq = (time.perf_counter() - t0)/8
    for B in (148, 1184):
        w = transit_workload(B)
        mc3.sample_batch(**{k: v[:1] if k in ('data', 'uncert', 'params', 'indparams') else v
                            for k, v in w.items()}, seed=1)              # warm-up of the module
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        outs = mc3.sample_batch(seed=1, **w)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        emit(dict(case='period_transit', B=B, wall_s=wall, per_problem_s=wall/B, sequential_per_call_s=seq,
                  sequential_extrapolated_s=seq*B, speedup_vs_sequential_extrapolated=seq*B/wall,
                  mean_acceptance=float(np.mean([o['acceptance_rate'] for o in outs]))))
        del outs
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(lines, f, indent=1)


if __name__ == '__main__':
    main()
