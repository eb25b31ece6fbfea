#!/usr/bin/env python
"""Benchmark of the mc3 sampling hot path (BASELINE.json metric: chain-steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--dump-outputs DIR]

Workload (N=1 and per GPU at N>1, weak scaling): BASELINE config 2 -- DEMC,
4096 chains per GPU, 5-parameter sinusoid+line model, 1e5 data points, fp64
chi-squared with Gaussian priors.  A "step" is one generation: every chain of
the population proposes, is evaluated against all data points and takes its
Metropolis decision.

One JSON line on stdout (rank 0):
  value      chain-steps/s with inputs resident in HBM, CUDA-event time of
             exactly K generations (one graph replay each), max over ranks
  e2e        the same metric through the public hub call mcmc_driver.mcmc()
             on HOST numpy inputs: H2D of the data, initial population, K
             generations, report-point reads, D2H of the posterior and the
             host post-statistics are all inside the timed region
  roofline   the fused model+chi-squared kernel timed alone with CUDA events,
             against the FP64 FMA peak measured live by mc3b_fma_peak
  cpu_baseline  the oracle port of the reference loop (numpy model + the
             reference's own C chi-squared from oracle/_ref when present) on
             the host cores: a bounded sample of the same workload

--impl reference prints the same line for the CPU reference arm.

--dump-outputs DIR writes, after the timed steps, what the last timed generation
computed (posterior rows, log-posterior, chi-squared, best parameters) as
DIR/<name>.npy in float64; the inputs are seeded, so two builds can be compared.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NCHAINS_PER_GPU = 4096
METRIC = 'chain-steps/s'


# --------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        # NVML in-process (a sample every 10 ms: the timed region lasts tens of ms);
        # the nvidia-smi loop of the profiling recipe when pynvml is missing.
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.stop_flag = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                 '-lms', '100', '-i', str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.h
        bits = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown',
                0x4: 'sw_power_cap'}
        try:
            smax = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            smax = None
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = ['', str(sm), str(smax), '', '']
                row += ['Active' if r & b else 'Not Active' for b in (0x8, 0x40, 0x20, 0x4)]
                self.rows.append(row)
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if getattr(self, 'nvml', None) is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
        elif self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': max(smax) if smax else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------
# CPU reference arm / baseline: the reference's own mcmc() on the host cores
# --------------------------------------------------------------------------
def _cpu_worker(args):
    """One process = one reference run: mc3.mcmc_driver.mcmc() itself (unmodified,
    byte-compiled by `make -C oracle refpy` into oracle/_ref, with the reference's C
    chi-squared from oracle/_ref) on 7 chains of config 2, ncpu=1 -- the reference's
    DEMC dead-locks with ncpu > 1 (SURVEY finding 5), so the host cores are filled
    with independent runs.  Falls back to the oracle port of the loop when the
    reference is not staged (kind 'port')."""
    seed, nchains, gens, warm = args
    os.dup2(2, 1)                                # the reference prints its greeting on stdout
    import random
    import numpy as np
    from oracle import models as om
    from oracle import ref
    from mc3_b200 import workloads
    w = workloads.config2()
    if ref.have_ref_py() and ref.have_ref_ext():
        R = ref.ref_py()
        log = R.utils.Log(verb=0)

        def run(ngen):
            random.randint = lambda a, b: seed + 1           # child seed, chain.py:180
            np.random.seed(seed)
            return R.mcmc_driver.mcmc(
                w['data'], np.copy(w['uncert']), om.sinusoid, np.copy(w['params']), [w['x']], {},
                w['pmin'], w['pmax'], w['pstep'], w['prior'], w['priorlow'], w['priorup'],
                nchains, 1, nchains*ngen, 'demc', False, None, False, 0.0, 0.5, 0, 1, 1.0,
                w['fepsilon'], 2, 'normal', None, False, log, None, None)
        kind = 'reference'
    else:
        from oracle import mcmc as omc
        from oracle import kernels as ok
        kw = dict(nchains=nchains, sampler='demc', thinning=1, fepsilon=w['fepsilon'],
                  hsize=2, record=False, chisq_fn=ok.chisq, parent_seed=seed, child_seed=seed + 1)
        a = (w['data'], w['uncert'], om.sinusoid, w['params'], [w['x']], {},
             w['pmin'], w['pmax'], w['pstep'], w['prior'], w['priorlow'], w['priorup'])

        def run(ngen):
            return omc.mcmc(*a, nsamples=nchains*ngen, **kw)
        kind = 'port'
    t_setup0 = time.perf_counter()
    run(max(warm, 1))                            # warm-up + setup cost (initial population, forks)
    t_setup = time.perf_counter() - t_setup0
    t0 = time.perf_counter()
    run(gens + max(warm, 1))
    t_all = time.perf_counter() - t0
    return max(t_all - t_setup, 1e-9), kind


def _cpu_proc(args, q):
    q.put(_cpu_worker(args))


def cpu_reference_run(steps, warmup, cores=None):
    """Time `steps` generations of `cores` independent 7-chain DEMC populations
    (one process each, the reference's own default chain count) at N=1e5.  Plain
    (non-daemonic) processes that exit normally: the reference forks its own chain
    process, and exit hooks get to run."""
    import multiprocessing as mp
    cores = cores or max(1, (os.cpu_count() or 2) - 1)      # sampler_driver.py:336-341
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    t0 = time.perf_counter()
    procs = [ctx.Process(target=_cpu_proc, args=((1000 + 7*i, 7, steps, warmup), q), daemon=False)
             for i in range(cores)]
    for p in procs:
        p.start()
    res = [q.get(timeout=3000) for _ in procs]
    for p in procs:
        p.join(60)
    wall = time.perf_counter() - t0
    tmax = max(r[0] for r in res)
    return dict(value=cores*7*steps/tmax, seconds=tmax, wall=wall, cores=cores,
                kind=res[0][1], chain_steps=cores*7*steps)


def _cpu_sample_text(r, steps):
    how = ('the UNMODIFIED reference mc3.mcmc_driver.mcmc() (byte-compiled into oracle/_ref, ncpu=1 '
           'per run: its DEMC dead-locks with ncpu > 1) with the reference C chi-squared'
           if r['kind'] == 'reference' else 'the oracle port of mc3/chain.py with the oracle C chi-squared')
    return (f'{r["cores"]} independent processes x 7 chains x {steps} generations of config 2 '
            f'(N=1e5, numpy sinusoid model) through {how}; {r["seconds"]:.1f} s')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    r = cpu_reference_run(K, W)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': METRIC,
        'n_gpus': args.gpus, 'steps': K, 'warmup': W,
        'ms_per_step': 1e3*r['seconds']/K, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'config2: DEMC, 5-param sinusoid+line, N=1e5, fp64 chisq + Gaussian priors',
                   'nchains': r['cores']*7, 'ndata': 100000, 'sampler': 'demc'},
        'cpu_baseline': {'value': r['value'], 'unit': METRIC, 'cores': r['cores'],
                         'kind': r['kind'], 'sample': _cpu_sample_text(r, K)},
        'e2e': {'value': r['value'], 'unit': METRIC, 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
        'chisq_evals_per_s': r['value']*100000,
        'gpu_launches': 0,
    }
    _emit(line)


# --------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import mc3_b200 as mc3
    from mc3_b200 import _lib, workloads
    from mc3_b200.engine import Population
    from mc3_b200.mcmc_driver import mcmc

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    K, W = args.steps, max(args.warmup, 3)
    w = workloads.config2()
    n = w['x'].size
    nchains = NCHAINS_PER_GPU*world
    model = mc3.models.BUILTIN[w['model']]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    pop = Population(w['data'], w['uncert'], model, w['params'], [w['x']], {},
                     w['pstep'], w['pmin'], w['pmax'], w['prior'], w['priorlow'],
                     w['priorup'], nchains=nchains, sampler=w['sampler'],
                     fepsilon=w['fepsilon'], thinning=1, nzchain=W + K + 1, seed=1234,
                     dtype=args.dtype, rank=rank, world=world)
    # clock sampler: started before the warm-up and stopped after the kernel-alone
    # timing, so that even a 4 ms timed region is bracketed by samples taken under
    # load of the same kernels (at least 3 samples are required below)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    parity = multi_gpu_parity(args, w, model, rank, world, dev) if world > 1 else None
    pop.init_population('normal')
    pop.run(W, use_graph=True)                   # warm-up (captures the generation graph)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(K)]
    launches0 = pop.launches
    barrier()
    align = torch.zeros(1, device=dev)
    for k in range(K):
        flush.fill_(k & 0xFF)                    # evict L2 between timed steps (untimed)
        if world > 1:
            # the generations of the devices are coupled (a proposal waits for every
            # device's previous generation): line the devices up after the untimed flush,
            # or its skew would be charged to the timed generation of the faster device
            dist.all_reduce(align)
        ev[k][0].record()
        pop.run(1, use_graph=True)
        ev[k][1].record()
    barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    launches = pop.launches - launches0
    value = nchains*K/(ms_total*1e-3)
    cnt = pop.counters()
    acc = cnt['numaccept']
    if args.dump_outputs:
        dump_outputs(pop, cnt, rank, args.dump_outputs)

    # ---- roofline of the dominant kernel, timed alone -------------------
    roof = None
    if rank == 0:
        import ctypes
        P = pop.nextp[pop.chain0:pop.chain0 + pop.nlocal]
        moment = bool(getattr(pop, 'use_moment', False))
        # the sufficient-statistics kernel exists only fused with the Metropolis epilogue
        # (its guard lives there): timed as the generation launches it, history write off
        fuse = (pop.chain0, pop.gen, -1, False) if moment else None
        pop.data_chisq(P, fuse=fuse)
        torch.cuda.synchronize(dev)
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
               for _ in range(K)]
        for k in range(K):
            flush.fill_(k & 0xFF)
            kev[k][0].record()
            pop.data_chisq(P, fuse=fuse)
            kev[k][1].record()
        torch.cuda.synchronize(dev)
        kms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
        flops = float(w['flops_per_point'])*pop.nlocal*n
        # FP64 (or FP32) FMA peak, measured now on this GPU
        sink = torch.zeros(8, dtype=torch.float64, device=dev)
        fl = ctypes.c_double(0.0)
        code = _lib.F64 if args.dtype == 'f64' else _lib.F32
        best = 0.0
        for it in range(4):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _lib.call('mc3b_fma_peak', code, 20000, sink.data_ptr(), ctypes.byref(fl),
                      _lib.stream_ptr())
            b.record()
            torch.cuda.synchronize(dev)
            if it:
                best = max(best, fl.value/(a.elapsed_time(b)*1e-3))
        achieved = flops/(kms*1e-3)
        prof = _profile_summary()
        # FP64-pipe instructions per (chain, point), read off the SASS: the plain
        # sinusoid takes 14 sine + 2 argument/line + 1 model + 3 residual/square = 20,
        # the uniform-grid recurrence 2 + 1 + 1 + 2 = 6 (profiles/r1_model_chisq.md);
        # each occupies the pipe like one FMA (2 flops) -- or 1.5x that when it reads
        # three fresh registers (profiles/r1_fp64_peak_probe.txt), which the peak
        # probe's FMAs never do, so fp64_pipe_frac understates the pipe's busy time.
        # The mirrored-pair kernel (k_sinefold) needs 425 per 128-point tile = 3.32: two points
        # share one sine/cosine product pair, so `frac` (SURVEY's 10 algorithmic flops per
        # chain-point over the FMA peak) can exceed what a per-point evaluation could reach;
        # fp64_pipe_frac is the executed-instruction view of the same launch.
        # The sufficient-statistics form (k_sinefold<MOM>): 28 per 16-point block + 6 per tile.
        folded = getattr(pop, 'd_fold', None) is not None
        pipe_instr = ((230.0/128.0 if moment else 425.0/128.0) if folded else 6.0) \
            if getattr(pop, 'grid', False) else (19.0 if pop.usig else 20.0)
        kname = (('k_fold_consts + k_sinefold<MOM> + Metropolis epilogue' if moment else 'k_fold_consts + k_sinefold')
                 if folded else
                 'k_sinegrid<USIG=%s>' % ('true' if pop.usig else 'false')) \
            if getattr(pop, 'grid', False) else 'k_model_chisq<SineModel>'
        roof = {'bound': 'fp64' if args.dtype == 'f64' else 'fp32',
                'kernel': kname,
                'fp64_pipe_instr_per_chain_point': pipe_instr,
                'achieved': achieved/1e12, 'peak': best/1e12, 'unit': 'TFLOP/s',
                'frac': achieved/best, 'traffic': prof.get('dram_bytes_per_launch'),
                'traffic_source': prof.get('source'),
                'fp64_pipe_frac': (2.0*pipe_instr*pop.nlocal*n/(kms*1e-3))/best
                if args.dtype == 'f64' else None,
                'peak_source': 'measured live: mc3b_fma_peak register-resident FMA chains',
                'ms_per_launch': kms,
                'note': ('frac = SURVEY 8(d) algorithmic flops (10 per chain-point) over the measured FMA peak; '
                         'this kernel executes %.2f FP64 instructions per chain-point, so frac may exceed 1 '
                         '(fp64_pipe_frac is the executed-instruction view)' % pipe_instr),
                'guard_hits': int(pop.guard_hits.item()) if moment else None,
                'algorithmic_flops_per_chain_point': w['flops_per_point'],
                'hbm_stream_GBs': 24.0*n/(kms*1e-3)/1e9,
                'hbm_peak_GBs': _measured_peaks().get('hbm_gbs')}

    ck = None
    if rank == 0:
        t_end = time.perf_counter() + 0.5
        while len(clocks.rows) < 3 and time.perf_counter() < t_end:
            pop.data_chisq(pop.nextp[pop.chain0:pop.chain0 + pop.nlocal])   # same kernel, untimed
            torch.cuda.synchronize(dev)
        ck = clocks.stop()
        ck['window'] = 'warm-up + timed generations + kernel-alone timing (10 ms NVML polls)'

    # ---- end to end through the public hub call, host buffers ------------
    barrier()
    host = {k: np.array(w[k]) for k in ('data', 'uncert', 'x', 'params', 'pstep', 'pmin',
                                       'pmax', 'prior', 'priorlow', 'priorup')}
    quiet = mc3.Log(verb=-1)

    def hub(ngen, seed):
        with contextlib.redirect_stdout(sys.stderr):      # keep stdout to the one JSON line
            return _hub(ngen, seed)

    def _hub(ngen, seed):
        return mcmc(host['data'], host['uncert'], model, host['params'], [host['x']], {},
                    host['pmin'], host['pmax'], host['pstep'], host['prior'],
                    host['priorlow'], host['priorup'], nchains, None, nchains*ngen,
                    w['sampler'], False, None, False, 0.0, 0.5, 0, 1, 1.0, w['fepsilon'],
                    10, 'normal', None, False, quiet, None, None, seed=seed,
                    dtype=args.dtype, rank=rank, world=world)
    hub(W, 76)                                   # warm-up of the whole public path (W generations)
    e2e_runs = []
    out = None
    for rep in range(3):                         # host-side time is noisy on a shared box: best of 3
        out = None                               # release the previous run's pinned result blocks
        barrier()
        t0 = time.perf_counter()
        out = hub(K, 77 + rep)
        barrier()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_runs.append(float(te.item()))
    e2e_s = min(e2e_runs)
    nfree = 5
    h2d = 3*8*n + 8*10*8                                  # x, data, uncert + small vectors
    d2h = out['posterior'].nbytes + out['log_post'].nbytes + out['zchain'].size*4
    e2e = {'value': nchains*K/e2e_s, 'unit': METRIC,
           'h2d_bytes_per_step': h2d/K, 'd2h_bytes_per_step': d2h/K,
           'seconds': e2e_s, 'seconds_all_calls': e2e_runs,
           'includes': 'H2D of data, initial population (10 x nchains evaluations), '
                       'K generations, report reads, D2H of posterior, host post-statistics'}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_reference_run(args.cpu_steps, 1)
        cpu = {'value': r['value'], 'unit': METRIC, 'cores': r['cores'], 'kind': r['kind'],
               'sample': _cpu_sample_text(r, args.cpu_steps)}
    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': METRIC, 'n_gpus': world,
            'steps': K, 'warmup': W, 'ms_per_step': ms_total/K,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': args.dtype, 'data': 'synthetic',
            'config': {'workload': w['name'], 'nchains': nchains,
                       'nchains_per_gpu': NCHAINS_PER_GPU, 'ndata': n,
                       'sampler': w['sampler'], 'model': w['model'],
                       'l2': 'flushed between timed steps (256 MB write, untimed)',
                       'parallelism': (f'chains partitioned over {world} GPU(s); '
                                       + ('next states stored into every device over NVLink by the '
                                          'Metropolis epilogue, generation flags instead of a collective'
                                          if pop.p2p is not None else
                                          'NCCL all-gather of the population per generation'))
                                      if world > 1 else 'single GPU'},
            'chisq_evals_per_s': value*n,
            'acceptance_rate_pct': 100.0*acc/(nchains*(W + K)),
            'e2e': e2e, 'gpu_launches': launches, 'clocks': ck,
            'roofline': roof, 'cpu_baseline': cpu,
        }
        if parity is not None:
            line['multi_gpu_parity'] = parity
        _emit(line)
    if world > 1:
        # captured graphs first (they may hold NCCL kernels), then the process group
        dist.barrier()
        pop.close()
        del pop
        torch.cuda.synchronize(dev)
        dist.destroy_process_group()


def dump_outputs(pop, counters, rank, outdir):
    """Write what the last timed generation computed, as a caller of Population.run()
    reads it: the history rows it wrote (posterior sample, log-posterior and chi-squared
    of every chain) and the best parameters so far.  The inputs are seeded, so two
    builds run with the same arguments can be compared array for array."""
    posterior, _, log_post, chisq = pop.history_host(dst=0)    # collective at world > 1
    if rank != 0:
        return
    n = pop.nchains                      # thinning 1: one row per chain and generation
    out = {'posterior': posterior[-n:], 'log_post': log_post[-n:], 'chisq': chisq[-n:],
           'bestp': counters['bestp']}
    os.makedirs(outdir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(outdir, name + '.npy'), np.asarray(a, dtype=np.float64))


def multi_gpu_parity(args, w, model, rank, world, dev):
    """Driver-visible check that N devices compute what one device computes: a short
    fixed-seed config-2 population (4096 chains in total, N=1e5: TMA path, decreasing
    split schedule) run on all ranks and on rank 0 alone, launch shape planned for the
    whole population; history compared byte for byte, and sampled rows' chi-squared
    against the oracle (used here as the checker only)."""
    import torch
    import torch.distributed as dist
    import mc3_b200 as mc3
    from mc3_b200.mcmc_driver import mcmc
    nch, ngen = 4096, 6
    quiet = mc3.Log(verb=-1)

    def run(rk, wd):
        with contextlib.redirect_stdout(sys.stderr):
            return mcmc(w['data'], w['uncert'], model, w['params'], [w['x']], {},
                        w['pmin'], w['pmax'], w['pstep'], w['prior'], w['priorlow'],
                        w['priorup'], nch, None, nch*ngen, w['sampler'], False, None, True, 0.0,
                        0.5, 0, 1, 1.0, w['fepsilon'], 2, 'normal', None, False, quiet, None, None,
                        seed=4242, dtype=args.dtype, rank=rk, world=wd, plan_chains=nch)
    multi = run(rank, world)
    dist.barrier()
    res = None
    if rank == 0:
        single = run(0, 1)
        eq = {k: bool(np.array_equal(multi[k], single[k])) for k in ('posterior', 'zchain', 'log_post')}
        from oracle import kernels as ok
        from oracle import models as om
        rs = np.random.RandomState(1)
        rows = rs.choice(multi['posterior'].shape[0], 4, replace=False)
        worst = 0.0
        for r in rows:
            p = np.array(w['params'], float)
            p[:] = multi['posterior'][r]                 # all five parameters are free
            want = ok.chisq(om.sinusoid(p, w['x']), w['data'], w['uncert'], p, w['prior'],
                            w['priorlow'], w['priorup'])
            got = -2.0*multi['log_post'][r]
            worst = max(worst, abs(got - want)/abs(want))
        res = {'bitwise_equal_to_1gpu': all(eq.values()), 'equal': eq,
               'oracle_rel_err': worst, 'nchains': nch, 'generations': ngen, 'ndata': int(w['x'].size),
               'rows_checked_against_oracle': [int(r) for r in rows],
               'exchange': 'peer-memory stores + generation flags' if os.environ.get('MC3B_P2P', '1') != '0'
                           else 'NCCL all-gather'}
    dist.barrier()
    torch.cuda.synchronize(dev)
    return res


_OUT = None


def _emit(line):
    out = _OUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def _profile_summary():
    """dram bytes per launch of the dominant kernel from the committed ncu capture."""
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', 'r2c_model_chisq.json')))
    except Exception:
        return {}


def _measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--dtype', default='f64', choices=['f64', 'f32'])
    ap.add_argument('--cpu-steps', type=int, default=2000)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    # stdout carries exactly one JSON line: everything libraries print on fd 1 while
    # the run lasts (NCCL's version banner, the hub's greeting) goes to stderr.
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
