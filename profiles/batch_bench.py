"""sample_batch against sequential sample() calls (README "Many small fits at once").

    python profiles/batch_bench.py [--out profiles/r9_batch.json] [--quick]

Workloads: config 1's shape (quadratic, snooker, 7 chains, N = 100, 1e5 samples, burn-in
1000) for B = 1, 148, 1184, 4736, and a sinusoid (N = 2000, DEMC, 32 chains, 6.4e4
samples) for B = 1, 148, 1184.  Per run: wall time of sample_batch split into set-up +
initial population (host clock to a synchronise), generations (device events around
mc3b_batch_run) and outputs (statistics, copies, dictionaries); summed chain-steps/s and
the time per problem.  8 sequential sample() calls, timed after a warm-up call, are
extrapolated to B (labelled as such).  The GPU's name, power limit and max SM clock are
read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mc3_b200 as mc3                      # noqa: E402
from mc3_b200 import batch_driver           # noqa: E402
from oracle import problems as pb           # noqa: E402


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def workload(name, B):
    rs = np.random.RandomState(B)
    if name == 'config1':
        p = pb.mcmc_case('quad')
        data = [p['data'] + rs.normal(0, 1e-3, p['data'].size)*p['uncert'] for _ in range(B)]
        return dict(data=data, uncert=[p['uncert']]*B, func=mc3.models.polynomial,
                    params=np.tile(p['params'], (B, 1)), indparams=[[p['x']]]*B, pstep=p['pstep'],
                    sampler='snooker', nchains=7, nsamples=1e5, burnin=1000)
    x = np.linspace(0.0, 10.0, 2000)
    truth = np.array([1.0, 2.5, 0.3, 5.0, -0.2])
    data = [mc3.models.sinusoid(truth, x) + rs.normal(0, 0.5, x.size) for _ in range(B)]
    return dict(data=data, uncert=[np.full(x.size, 0.5)]*B, func=mc3.models.sinusoid,
                params=np.tile(truth*1.01, (B, 1)), indparams=[[x]]*B, pstep=np.array([1e-2, 1e-3, 1e-2, 1e-2, 1e-3]),
                pmin=np.array([0.5, 2.0, -np.pi, 4.0, -1.0]), pmax=np.array([1.5, 3.0, np.pi, 6.0, 1.0]),
                sampler='demc', nchains=32, nsamples=6.4e4, burnin=0)


class Stages:
    """Times the stages of sample_batch (wraps _BatchRun.init / run / outputs)."""

    def __init__(self):
        self.t = {}
        R = batch_driver._BatchRun
        self.orig = (R.init, R.run, R.outputs)
        st = self

        def init(self_, *a):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = st.orig[0](self_, *a)
            torch.cuda.synchronize()
            st.t['init_s'] = time.perf_counter() - t0
            return r

        def run(self_, *a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = st.orig[1](self_, *a)
            e1.record()
            e1.synchronize()
            st.t['generations_s'] = e0.elapsed_time(e1)/1e3
            return r

        def outputs(self_, *a):
            t0 = time.perf_counter()
            r = st.orig[2](self_, *a)
            torch.cuda.synchronize()
            st.t['outputs_s'] = time.perf_counter() - t0
            return r
        R.init, R.run, R.outputs = init, run, outputs


def run_batch(name, B, seed=1):
    w = workload(name, B)
    stages = Stages()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = mc3.sample_batch(w.pop('data'), w.pop('uncert'), w.pop('func'), w.pop('params'), w.pop('indparams'),
                            seed=seed, **w)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    R = batch_driver._BatchRun
    R.init, R.run, R.outputs = stages.orig
    return wall, stages.t, outs


def run_sequential(name, k=8):
    w = workload(name, k)
    quiet = mc3.Log(verb=-1)
    args = {a: w[a] for a in ('pstep', 'sampler', 'nchains', 'nsamples', 'burnin', 'pmin', 'pmax') if a in w}
    call = lambda b: mc3.sample(w['data'][b], w['uncert'][b], func=w['func'], params=w['params'][b],  # noqa: E731
                                indparams=w['indparams'][b], seed=1 + b, log=quiet, **args)
    call(0)                                   # warm-up (module load, first allocations)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in range(k):
        call(b)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0)/k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--quick', action='store_true', help='B = 1 and 148 only')
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    lines = []
    cases = [('config1', (1, 148, 1184, 4736)), ('sine2000', (1, 148, 1184))]
    run_batch('config1', 1)                   # warm-up: library load, first launches
    for name, Bs in cases:
        seq = run_sequential(name)
        for B in Bs:
            if args.quick and B > 148:
                continue
            wall, t, outs = run_batch(name, B)
            w = workload(name, 1)
            nchains = w['nchains']
            steps = B*int(np.ceil(w['nsamples']/nchains))*nchains
            line = dict(workload=name, B=B, gpu=info, wall_s=wall, **t,
                        chain_steps_per_s=steps/wall, generation_chain_steps_per_s=steps/t['generations_s'],
                        per_problem_s=wall/B, sequential_per_call_s=seq,
                        sequential_extrapolated_s=seq*B, speedup_vs_sequential_extrapolated=seq*B/wall,
                        mean_acceptance=float(np.mean([o['acceptance_rate'] for o in outs])))
            print(json.dumps(line), flush=True)
            lines.append(line)
            del outs
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(lines, f, indent=1)


if __name__ == '__main__':
    main()
