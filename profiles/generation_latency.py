"""Where the time of one config-2 generation goes (4096 chains, N = 1e5, fp64, DEMC), with the
protocol of bench.py: a 256 MB fill of a scratch buffer before every timed item (untimed), so that
each item starts from an L2 that holds none of its lines and has to evict dirty ones.  Each item is
timed K = 200 times with CUDA events around it, flushed and warm (warm: the same item back to back,
CUDA events around each call, the call enqueued behind a 50 us device-side spin so that host
launch overhead is not charged to the device time):

  step              pop.run(1, use_graph=True), exactly as bench.py calls it (host work included)
  graph_replay      pop._graph.replay(): one captured generation
  propose           mc3b_propose alone, device-driven as in the graph
  chisq_fused       pop.data_chisq(P, fuse=...): the chi-squared kernel + fused Metropolis epilogue
  graph_replay_no_record   graph_replay of a generation captured without the guard record ring
                    (mc3b_moment_t.record = NULL): the cost of the record's store.  Timed in the
                    order with, without, without, with (the _2 entries)

    python profiles/generation_latency.py [--out FILE] [--label NAME]

Writes (or adds the entry `label` to) the JSON file `out`, default profiles/r4_generation_latency.json,
together with the card name, power limit and SM clocks read in the same process.  Needs a GPU."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import mc3_b200 as mc3  # noqa: E402
from mc3_b200 import _lib, workloads  # noqa: E402
from mc3_b200.engine import Population  # noqa: E402

K = 200


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm',
                        '--format=csv,noheader'], capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else 'unknown'


def measure(pop, fn, flush, spin):
    """mean us per call of fn over K calls, L2 flushed before each, and warm."""
    out = {}
    for mode in ('l2_flushed', 'warm'):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for k in range(K):
            if mode == 'l2_flushed':
                flush.fill_(k & 0xFF)
            else:
                spin()
            ev[k][0].record()
            fn()
            ev[k][1].record()
        torch.cuda.synchronize()
        t = np.array([a.elapsed_time(b) for a, b in ev])*1e3
        out[mode] = {'mean_us': float(t.mean()), 'median_us': float(np.median(t)), 'min_us': float(t.min())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                  'r4_generation_latency.json'))
    ap.add_argument('--label', default='current')
    args = ap.parse_args()

    w = workloads.config2()
    pop = Population(w['data'], w['uncert'], mc3.models.BUILTIN[w['model']], w['params'], [w['x']], {},
                     w['pstep'], w['pmin'], w['pmax'], w['prior'], w['priorlow'], w['priorup'],
                     nchains=4096, sampler=w['sampler'], fepsilon=w['fepsilon'], thinning=1,
                     nzchain=10*K + 64, seed=1234)
    pop.init_population('normal')
    pop.run(3, use_graph=True)                   # warm-up (captures the generation graph)
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=pop.dev)
    sleeper = torch.cuda._sleep                  # device-side spin: the host runs ahead of the device
    cycles = int(50e-6*1.9e9)

    def spin():
        sleeper(cycles)

    st = _lib.stream_ptr()
    c0, c1 = pop.chain0, pop.chain0 + pop.nlocal
    P = pop.nextp[c0:c1]

    def step():
        pop.run(1, use_graph=True)

    def replay():
        pop._graph.replay()

    def propose():
        _lib.call('mc3b_propose', ctypes.byref(pop.S), -1, 0, c0, c1, st)

    def chisq_fused():
        pop.data_chisq(P, fuse=(c0, pop.gen, -1, False))

    res = {'spectral': pop.spectral is not None, 'use_moment': bool(getattr(pop, 'use_moment', False))}
    res['step'] = measure(pop, step, flush, spin)
    pop.gen_dev.fill_(pop.gen)
    ring = pop.moment.record
    pop.moment.record = None
    plain, _ = pop._capture(1)
    pop.moment.record = ring
    # A B B A: with and without the record store, alternated against drift
    res['graph_replay'] = measure(pop, replay, flush, spin)
    res['graph_replay_no_record'] = measure(pop, plain.replay, flush, spin)
    res['graph_replay_no_record_2'] = measure(pop, plain.replay, flush, spin)
    res['graph_replay_2'] = measure(pop, replay, flush, spin)
    del plain
    res['propose'] = measure(pop, propose, flush, spin)
    res['chisq_fused'] = measure(pop, chisq_fused, flush, spin)
    pop.gen += 8*K                               # the four graph_replay items, flushed and warm
    pop.gen_dev.fill_(pop.gen)
    torch.cuda.synchronize()
    res['gpu'] = gpu_info()
    res['guard_hits'] = int(pop.guard_hits.item())

    doc = {}
    if os.path.exists(args.out):
        doc = json.load(open(args.out))
    doc.setdefault('workload', 'config 2: DEMC, 4096 chains, sinusoid + line, N = 1e5, fp64, one sigma')
    doc.setdefault('protocol', f'CUDA events around each of K = {K} calls; l2_flushed: a 256 MB fill '
                   'before each call (untimed); warm: a 50 us device spin before each call (untimed), '
                   'no flush; gpu: name, power limit, SM clock, max SM clock')
    doc[args.label] = res
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(doc, open(args.out, 'w'), indent=1)
    print(json.dumps({args.label: res}, indent=1))


if __name__ == '__main__':
    main()
