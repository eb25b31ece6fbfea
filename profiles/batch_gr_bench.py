"""sample_batch with the Gelman-Rubin test and early stop (README "Many small fits at once").

    python profiles/batch_gr_bench.py [--out profiles/r11_batch_gr.json] [--quick]

Four arms, alternated in one process, twice each, per workload and B:
  a  grtest=False                     the batch as it was
  b  grtest=True, grbreak=0           one test at the last report
  c  grtest=True, grbreak=1e-9        the test at every report past burn-in, never met: the
                                      cost of the test alone (the histories equal arm a's)
  d  grtest=True, grbreak=1.01        problems stop at the first report that passes
                                      (grnmin 0.5, sample()'s default)
Workloads: config 1's shape (quadratic, snooker, 7 chains, N = 100, 1e5 samples, burn-in
1000) at B = 148, 1184, 4736; the README's trapezoid transit CudaModel on a known period and
exposure time (N = 2000, 32 chains, DEMC, 6.4e4 samples, burn-in 200) at B = 148, 1184; and a
mixed catalogue at B = 1184: config 1's quadratic, half of the problems over x in [0, 10], half
over [0, 1/3], where the three coefficients are strongly correlated and the chains mix slowly,
with grnmin 0.1 so that the test, not grnmin, sets where each half stops (the other workloads
keep sample()'s grnmin 0.5).
Per run: wall time of sample_batch (host clock to a synchronise), the generations + test
window (device events from the end of the initial population to the start of the outputs),
and for arm d the fraction of generations that ran, sum K_b / (B nzchain).  Arms a and c are
checked to give the same posterior, log_post and zchain bytes (a digest per run).  The GPU's
name, power limit and max SM clock are read in the same process.
"""
import argparse
import hashlib
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

PTRANSIT = '''__device__ void prepare(real* p) { p[7] = 1 / p[5]; p[8] = p[2] + (real)0.5 * p[6]; }
__device__ real model(real x, const real* p) {
    real dt = x - p[1];
    dt -= p[5] * rint(dt * p[7]);
    real z = fabs(dt) / p[8];
    return p[3] - p[0] * (z < 1 ? (real)1 : (z < p[4] ? (p[4] - z)/(p[4] - 1) : (real)0));
}'''
ARMS = {'a': dict(grtest=False), 'b': dict(grtest=True, grbreak=0.0),
        'c': dict(grtest=True, grbreak=1e-9), 'd': dict(grtest=True, grbreak=1.01)}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


_TRANSIT = None


def workload(name, B):
    global _TRANSIT
    rs = np.random.RandomState(B)
    if name in ('config1', 'mixed'):
        p = pb.mcmc_case('quad')
        xs, data = [], []
        for b in range(B):
            x = p['x'] if name == 'config1' or b % 2 == 0 else p['x']/30.0
            y = 3.0 - 2.4*x + 0.5*x*x
            xs.append([x])
            data.append(y + rs.normal(0, 1.0, x.size)*p['uncert'])
        return dict(data=data, uncert=[p['uncert']]*B, func=mc3.models.polynomial,
                    params=np.tile(p['params'], (B, 1)), indparams=xs, pstep=p['pstep'],
                    sampler='snooker', nchains=7, nsamples=1e5, burnin=1000,
                    **({'grnmin': 0.1} if name == 'mixed' else {}))
    if _TRANSIT is None:
        _TRANSIT = mc3.CudaModel(PTRANSIT, 5, name='period_transit', nconst=2, nwork=2)
    x = np.linspace(0.0, 10.0, 2000)
    period, exptime = 3.0, 0.01
    truth = np.array([0.01, 0.4, 0.1, 1.0, 1.3])
    clean = _TRANSIT(truth, x, period, exptime)
    return dict(data=[clean + rs.normal(0, 1e-3, x.size) for _ in range(B)], uncert=[np.full(x.size, 1e-3)]*B,
                func=_TRANSIT, params=np.tile(truth*1.01, (B, 1)), indparams=[[x, period, exptime]]*B,
                pstep=np.array([1e-4, 1e-3, 1e-3, 1e-4, 0.0]), pmin=np.array([0.0, 0.2, 0.01, 0.9, 1.0]),
                pmax=np.array([0.05, 0.6, 0.3, 1.1, 2.0]), sampler='demc', nchains=32, nsamples=6.4e4, burnin=200)


class Window:
    """Device events from the end of _BatchRun.init to the start of _BatchRun.outputs."""

    def __init__(self):
        R = batch_driver._BatchRun
        self.orig = (R.init, R.outputs)
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w = self

        def init(self_, *a):
            r = w.orig[0](self_, *a)
            w.e0.record()
            return r

        def outputs(self_, *a):
            w.e1.record()
            return w.orig[1](self_, *a)
        R.init, R.outputs = init, outputs

    def close(self):
        R = batch_driver._BatchRun
        R.init, R.outputs = self.orig
        self.e1.synchronize()
        return self.e0.elapsed_time(self.e1)/1e3


def digest(outs):
    h = hashlib.blake2b(digest_size=16)
    for o in outs:
        for k in ('posterior', 'log_post', 'zchain'):
            h.update(np.ascontiguousarray(o[k]).data)
    return h.hexdigest()


def run_arm(name, B, arm, check):
    w = workload(name, B)
    nzchain = int(np.ceil(w['nsamples']/w['nchains']))
    win = Window()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = mc3.sample_batch(w.pop('data'), w.pop('uncert'), w.pop('func'), w.pop('params'), w.pop('indparams'),
                            seed=1, **ARMS[arm], **w)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    gen = win.close()
    K = np.array([len(o['posterior'])//w['nchains'] for o in outs])
    r = dict(wall_s=wall, generations_and_test_s=gen, ran_fraction=float(K.sum()/(B*nzchain)),
             stopped=int((K < nzchain).sum()),
             stop_fractions={f'{k/nzchain:.2f}': int(c) for k, c in zip(*np.unique(K, return_counts=True))})
    if check:
        r['digest'] = digest(outs)
    if arm != 'a':
        psrf = np.array([o['psrf'] for o in outs])
        r['max_psrf_median'] = float(np.median(psrf.max(axis=1)))
    del outs
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--quick', action='store_true', help='B = 148 only')
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    lines = []
    cases = [('config1', (148, 1184, 4736)), ('transit', (148, 1184)), ('mixed', (1184,))]
    for name, _ in cases:                               # warm-up: library and module loads
        for arm in ARMS:
            run_arm(name, 2, arm, False)
    for name, Bs in cases:
        for B in Bs:
            if args.quick and B > 148:
                continue
            res = {arm: [] for arm in ARMS}
            for rep in range(2):
                for arm in ARMS:
                    res[arm].append(run_arm(name, B, arm, check=rep == 0 and arm in 'ac'))
            best = {arm: min(r['generations_and_test_s'] for r in res[arm]) for arm in ARMS}
            wall = {arm: min(r['wall_s'] for r in res[arm]) for arm in ARMS}
            line = dict(workload=name, B=B, gpu=info, runs=res,
                        a_c_histories_identical=res['a'][0]['digest'] == res['c'][0]['digest'],
                        c_over_a_generations=best['c']/best['a'], b_over_a_generations=best['b']/best['a'],
                        d_over_a_generations=best['d']/best['a'], c_over_a_wall=wall['c']/wall['a'],
                        d_over_a_wall=wall['d']/wall['a'], d_ran_fraction=res['d'][0]['ran_fraction'],
                        d_stopped=res['d'][0]['stopped'], d_stop_fractions=res['d'][0]['stop_fractions'])
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(lines, f, indent=1)


if __name__ == '__main__':
    main()
