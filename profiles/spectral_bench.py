"""Spectral form against the tile moment form at config 2 (4096 chains, N = 1e5, fp64), CUDA-event
timing: table build, the chi-squared kernel alone with the fused Metropolis epilogue (k_spectral_chisq
against k_fold_consts + k_sinefold<MOM>), one generation as a graph replay, the initial population, and
the guard count.  Writes JSON to argv[1] (default profiles/r3_spectral.json).  Needs a GPU."""
import ctypes
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import mc3_b200 as mc3  # noqa: E402
from mc3_b200 import _lib, workloads  # noqa: E402
from mc3_b200.engine import Population  # noqa: E402


def timeit(fn, reps=300):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return 1e3*a.elapsed_time(b)/reps      # us per call


def timegraph(fn, calls=50, reps=20):
    """us per call of `calls` back-to-back calls captured in one CUDA graph (no host overhead)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    return timeit(g.replay, reps=reps)/calls


def population(no_spectral):
    if no_spectral:
        os.environ['MC3B_NO_SPECTRAL'] = '1'
    else:
        os.environ.pop('MC3B_NO_SPECTRAL', None)
    w = workloads.config2()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pop = Population(w['data'], w['uncert'], mc3.models.sinusoid, w['params'], [w['x']], {},
                     w['pstep'], w['pmin'], w['pmax'], w['prior'], w['priorlow'], w['priorup'],
                     nchains=4096, sampler='demc', fepsilon=0.01, thinning=1, nzchain=2000, seed=3)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    pop.init_population('normal')
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return pop, 1e3*(t1 - t0), 1e3*(t2 - t1)


def measure(no_spectral):
    pop, t_init, t_initpop = population(no_spectral)
    out = {'spectral': pop.spectral is not None, 'population_ctor_ms': t_init, 'initial_population_ms': t_initpop}
    if pop.spectral is not None:
        S = pop.spectral
        x, d = pop.k_x, pop.k_d
        M = pop.moment
        out['table_build_us'] = timeit(lambda: _lib.call('mc3b_spectral_prepare', x.data_ptr(), d.data_ptr(),
                                                         pop.ndata, M.c0ref, M.slref, ctypes.byref(S),
                                                         _lib.stream_ptr()), reps=20)
        out['plan'] = {k: (float(v) if k not in ('order', 'n1', 'n2') else int(v))
                       for k, v in pop.spectral_plan.items()}
    pop.run(5, use_graph=True)
    torch.cuda.synchronize()
    P = pop.nextp[:4096]
    g = pop.gen
    # the chi-squared launch(es) of one generation alone, with the fused Metropolis epilogue
    # (spectral: k_spectral_chisq; tile form: k_fold_consts + k_sinefold<MOM>), and without it
    out['chisq_kernel_fused_us'] = timegraph(lambda: pop.data_chisq(P, fuse=(0, g, -1, False)))
    out['chisq_kernel_unfused_us'] = timegraph(lambda: pop.data_chisq(P, moment_ok=True))
    pop.gen_dev.fill_(pop.gen)
    out['graph_replay_per_generation_us'] = timeit(lambda: pop._graph.replay(), reps=500)
    out['graph_launches_per_generation'] = pop._graph_launches
    torch.cuda.synchronize()
    out['guard_hits'] = int(pop.guard_hits.item())
    out['use_moment_after'] = bool(pop.use_moment)
    return out


if __name__ == '__main__':
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(__file__), 'r3_spectral.json')
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    measure(False)                     # warm-up: module loads and first allocations of the process
    res = {'workload': 'config 2: DEMC, 4096 chains, sinusoid + line, N = 1e5, fp64, one sigma',
           'gpu': gpu[0] if gpu else 'unknown',
           'timing': 'CUDA events over back-to-back calls, after warm-up; the data (0.8 MB) stay in L2',
           'note': 'population_ctor_ms includes the table build; both arms after one warm-up population',
           'spectral': measure(False), 'tile_moment_form': measure(True)}
    json.dump(res, open(path, 'w'), indent=1)
    print(json.dumps(res, indent=1))
