"""A CudaModel in the wavelet likelihood: the model evaluated inside the D4 kernels of its
fp64 module (mc3b_user_model_dwt_chisq) against the built-in model and against the path it
replaces (model rows written by mc3b_user_model_eval_consts, read back by
mc3b_dwt_chisq(-1)).

1. Config 3's shape (snooker, 16384 chains x 2^20 points, hsize = 10): initial-population
   time and ms per generation (CUDA events around run(K) after run(3)) of the built-in box
   and a CudaModel box, alternated.  Each case runs in a process of its own, so that every
   one starts from an empty device.  With --parent, the same CudaModel case also runs on
   the parent tree, where it cannot start (its model rows do not fit).
2. 4096 chains x 2^16: the wavelet chi-squared alone, new entry point against the rows
   path, alternated, for the box and for a model of three inputs and two constants.
3. The cold NVRTC compile of a user model (a source NVRTC has not seen), this tree against
   the parent tree, alternated, one process per compile.

The GPU's name, power limit and maximum SM clock are read in the same run.

    python profiles/usermodel_wavelet_bench.py [--parent DIR] [--out profiles/r7_usermodel_wavelet.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.environ.get('MC3B_BENCH_ROOT', os.path.dirname(HERE))     # the tree whose package runs
sys.path.insert(0, ROOT)

BOX = '''__device__ real model(real x, const real* p) {
    return fabs(x - p[1]) < (real)(0.5 * p[2]) ? (real)(p[3] - p[0]) : p[3];
}'''
K3 = '''__device__ void prepare(real* p) { p[6] = p[4] * p[5]; }
__device__ real model(real x, real y, real z, const real* p) {
    return fma(p[0], x, fma(p[1], y * z, p[2] * sin(p[3] * x))) * p[6];
}'''
C3_CHAINS, C3_STEPS, C3_HSIZE = 16384, 20, 10
DC_CHAINS, DC_N, DC_REPS, DC_ROUNDS = 4096, 1 << 16, 20, 5


def case_config3(model):
    import torch
    import mc3_b200 as mc3
    from mc3_b200 import _lib, workloads
    from mc3_b200.engine import Population
    w = workloads.config3()
    func = mc3.models.box if model == 'builtin' else mc3.CudaModel(BOX, 4, name='box')
    if model == 'cuda':
        func.handle(_lib.F64)                      # compiled outside the timed window
    pop = Population(w['data'], w['uncert'], func, w['params'], [w['x']], {}, w['pstep'], w['pmin'], w['pmax'],
                     w['prior'], w['priorlow'], w['priorup'], nchains=C3_CHAINS, sampler='snooker', wlike=True,
                     thinning=1, nzchain=C3_STEPS + 4, seed=5, hsize=C3_HSIZE)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    try:
        pop.init_population('normal')
        torch.cuda.synchronize()
    except (torch.OutOfMemoryError, RuntimeError) as e:
        return {'error': f'{type(e).__name__}: {str(e).splitlines()[0]}'}
    t_init = time.perf_counter() - t0
    pop.run(3)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    pop.run(C3_STEPS)
    b.record()
    torch.cuda.synchronize()
    c = pop.counters()
    return {'init_s': t_init, 'ms_per_generation': a.elapsed_time(b)/C3_STEPS,
            'best_chisq': -2*c['best_log_post'], 'numaccept': int(c['numaccept']),
            'peak_gb': torch.cuda.max_memory_allocated()/1e9}


def case_data_chisq():
    import numpy as np
    import torch
    import mc3_b200 as mc3
    from mc3_b200 import _lib
    dev = torch.device('cuda')
    rs = np.random.RandomState(1)
    n, nb = DC_N, DC_CHAINS
    xs = [torch.as_tensor(rs.uniform(-0.5, 0.5, n), device=dev) for _ in range(3)]
    data = torch.as_tensor(rs.normal(1.0, 1e-3, n), device=dev)
    kc = torch.as_tensor([0.5, 2.5], device=dev)
    ws = torch.empty(_lib.load().mc3b_dwt_workspace(nb, n)//8 + 1, dtype=torch.float64, device=dev)
    rows = torch.empty((nb, n), dtype=torch.float64, device=dev)
    out = torch.empty(nb, dtype=torch.float64, device=dev)
    st = _lib.stream_ptr()
    models = {
        'box': (mc3.CudaModel(BOX, 4, name='box'), [0.0101, 0.001, 0.1003, 1.0], xs[:1], None, 0),
        'k3_consts': (mc3.CudaModel(K3, 4, name='k3', ninputs=3, nconst=2, nwork=1), [0.3, -0.2, 0.1, 3.0],
                      xs, kc, 2),
    }
    res = {}
    for name, (um, p0, xin, k, nk) in models.items():
        h = um.handle(_lib.F64)
        full = np.concatenate([p0, [1.0, 5e-4, 1e-3]])
        P = torch.as_tensor(full*(1 + 0.01*rs.normal(size=(nb, full.size))), device=dev)
        xp = _lib.ptrs(xin)

        def fused():
            _lib.call('mc3b_user_model_dwt_chisq', h, P.data_ptr(), P.shape[1], nb, P.shape[1], xp, len(xin),
                      _lib.ptr(k), nk, data.data_ptr(), n, ws.data_ptr(), out.data_ptr(), st)

        def rows_path():
            _lib.call('mc3b_user_model_eval_consts', h, P.data_ptr(), P.shape[1], nb, xp, len(xin), _lib.ptr(k),
                      nk, n, rows.data_ptr(), st)
            _lib.call('mc3b_dwt_chisq', -1, P.data_ptr(), P.shape[1], nb, P.shape[1], 0, None, rows.data_ptr(), n,
                      data.data_ptr(), n, ws.data_ptr(), out.data_ptr(), st)
        fused()
        a = out.clone()
        rows_path()
        rel = float(((out - a).abs()/a.abs()).max())
        times = {'fused_ms': [], 'rows_ms': []}
        for _ in range(DC_ROUNDS):
            for key, fn in (('fused_ms', fused), ('rows_ms', rows_path)):
                fn()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(DC_REPS):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                times[key].append(e0.elapsed_time(e1)/DC_REPS)
        res[name] = dict(times, max_rel_diff=rel)
    return res


def case_compile(tag):
    from mc3_b200 import _lib, jit
    out = []
    for i in range(2):
        src = f'// {tag} {os.getpid()} {time.time_ns()} {i}\n' + BOX      # a source NVRTC has not seen
        t0 = time.perf_counter()
        jit.compile_cubin(src, 4, _lib.F64, 'box')
        out.append(time.perf_counter() - t0)
    return out


def sub(root, *args):
    """Run one case of this script in a process of its own, on the package of `root`."""
    env = dict(os.environ, MC3B_BENCH_ROOT=root)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), '--case', *args], env=env,
                       capture_output=True, text=True)
    lines = [line for line in r.stdout.splitlines() if line.startswith(('{', '['))]
    if r.returncode != 0 or not lines:
        return {'error': (r.stderr or r.stdout).strip().splitlines()[-1:]}
    return json.loads(lines[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--case', nargs='+')
    ap.add_argument('--parent', help='a built copy of the parent tree')
    ap.add_argument('--out', default=os.path.join(HERE, 'r7_usermodel_wavelet.json'))
    ap.add_argument('--rounds', type=int, default=2)
    args = ap.parse_args()
    if args.case:
        kind = args.case[0]
        res = (case_config3(args.case[1]) if kind == 'config3' else case_data_chisq() if kind == 'data_chisq'
               else case_compile(args.case[1]))
        print(json.dumps(res))
        return
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {'gpu': gpu[:1], 'config3': {'chains': C3_CHAINS, 'n': 1 << 20, 'hsize': C3_HSIZE, 'steps': C3_STEPS,
                                       'builtin': [], 'cuda': []}}
    me = os.path.dirname(HERE)
    if args.parent:
        res['config3']['cuda_parent'] = sub(args.parent, 'config3', 'cuda')
    for _ in range(args.rounds):
        for model in ('builtin', 'cuda'):
            res['config3'][model].append(sub(me, 'config3', model))
    res['data_chisq'] = dict(sub(me, 'data_chisq'), chains=DC_CHAINS, n=DC_N)
    comp = {'this': [], 'parent': []}
    for _ in range(args.rounds):
        comp['this'].append(sub(me, 'compile', 'this'))
        if args.parent:
            comp['parent'].append(sub(args.parent, 'compile', 'parent'))
    res['compile_s'] = comp
    print(json.dumps(res, indent=1))
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
