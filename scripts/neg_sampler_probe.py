"""Times the negative edge sampler: the reference's host sampler against tpnet_b200.NegativeEdgeSampler.

    python scripts/neg_sampler_probe.py --part host   [--calls 30] [--out profiles/neg_sampler_host.json]
    python scripts/neg_sampler_probe.py --part device [--out profiles/neg_sampler_probe_b200.json]

host   : the reference's NegativeEdgeSampler where oracle/_ref/TPNet is installed, otherwise the literal restatement
         of oracle/negative_sampler.py (the same set code); the JSON says which.  Per-call seconds of ``sample`` over
         the first ``--calls`` test batches of B = 200, and the constructor.  A CPU program timed on the CPU.
device : construction and ``sample`` (CUDA events) on the same shapes at B = 200, and at B = 100,000 on a power-law
         graph whose tables are far larger than the 126 MB L2; the card's name and power limit are read in the same run.
Shapes: the Flights-shaped 400,000-edge replica and the full Reddit shape (tpnet_b200.synth), test split = last 15 %,
inductive last_observed_time = the end of the 70 % training split.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200.synth import SHAPES, GraphShape, edge_stream  # noqa: E402

REF = os.path.join(ROOT, 'oracle', '_ref', 'TPNet')
CASES = (('flights', 400_000), ('reddit', SHAPES['reddit'].num_edges))


def stream(shape, edges, batch=1000, seed=0):
    parts = list(edge_stream(shape, batch, edges // batch, seed=seed))
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


def reference_class():
    if os.path.isfile(os.path.join(REF, 'utils', 'utils.py')):
        sys.path.insert(0, REF)
        from utils.utils import NegativeEdgeSampler
        return NegativeEdgeSampler, 'reference utils.utils.NegativeEdgeSampler'
    from oracle.negative_sampler import LiteralNegativeSampler
    return LiteralNegativeSampler, 'oracle.negative_sampler.LiteralNegativeSampler (the reference is not installed)'


def host(calls: int):
    cls, kind = reference_class()
    out = {'timed': kind, 'batch': 200, 'calls_timed': calls, 'cases': []}
    for name, edges in CASES:
        src, dst, t = stream(SHAPES[name], edges)
        lot = float(t[int(0.70 * len(t))])
        first = int(0.85 * len(t))
        n_pairs = len(np.unique(src)) * len(np.unique(dst))
        for strategy in ('historical', 'inductive'):
            rec = {'shape': name, 'edges': int(edges), 'strategy': strategy, 'unique_src_x_unique_dst': n_pairs}
            if n_pairs <= 20_000_000:
                t0 = time.perf_counter()
                smp = cls(src, dst, t, lot, strategy, seed=0)
                rec['construct_s'] = time.perf_counter() - t0
            else:                         # the constructor's set of S x D tuples is not built: not measured
                rec['construct_s'] = None
                smp = cls.__new__(cls)
                smp.__dict__.update(seed=0, negative_sample_strategy=strategy, src_node_ids=src, dst_node_ids=dst,
                                    interact_times=t, earliest_time=t.min(), last_observed_time=lot,
                                    random_state=np.random.RandomState(0))
                if strategy == 'inductive':
                    sel = t <= lot
                    smp.observed_edges = set(zip(src[sel].tolist(), dst[sel].tolist()))
            secs = []
            for c in range(calls):
                i = first + 200 * c
                j = i + 200
                t0 = time.perf_counter()
                smp.sample(200, src[i:j], dst[i:j], t[i], t[j - 1])
                secs.append(time.perf_counter() - t0)
            rec['sample_s_mean'] = float(np.mean(secs))
            rec['sample_s_max'] = float(np.max(secs))
            rec['test_batches'] = (len(t) - first + 199) // 200
            rec['test_split_sample_s_estimate'] = rec['sample_s_mean'] * rec['test_batches']
            out['cases'].append(rec)
            print(json.dumps(rec), flush=True)
    return out


def device():
    import torch
    from tpnet_b200 import NegativeEdgeSampler
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    out = {'gpu': q.stdout.strip(), 'cases': []}

    def timed(fn, reps=1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            r = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / 1e3 / reps, r

    def case(name, src, dst, t, B, strategies=('historical', 'inductive', 'random'), max_calls=300):
        lot = float(t[int(0.70 * len(t))])
        first = int(0.85 * len(t))
        src_d, dst_d, t_d = (torch.from_numpy(x).cuda() for x in (src, dst, t))
        spans = [(i, min(i + B, len(t))) for i in range(first, len(t), B)][:max_calls]
        for strategy in strategies:
            NegativeEdgeSampler(src, dst, t, lot, strategy, seed=0, device='cuda:0')        # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            smp = NegativeEdgeSampler(src, dst, t, lot, strategy, seed=0, device='cuda:0')
            construct = time.perf_counter() - t0                # includes the host checks and the uploads
            for i, j in spans[:3]:                              # warm-up of every shape
                smp.sample(j - i, src_d[i:j], dst_d[i:j], t_d[i], t_d[j - 1], as_tensors=True)
            smp.reset_random_state()
            torch.cuda.synchronize()

            def run():
                for i, j in spans:
                    smp.sample(j - i, src_d[i:j], dst_d[i:j], t_d[i], t_d[j - 1], as_tensors=True)
            total, _ = timed(run)
            rec = {'shape': name, 'edges': int(len(t)), 'strategy': strategy, 'batch': B, 'calls': len(spans),
                   'construct_wall_s': construct, 'sample_s_mean': total / len(spans),
                   'distinct_edges': smp.num_unique_edges}
            out['cases'].append(rec)
            print(json.dumps(rec), flush=True)
            del smp
            torch.cuda.empty_cache()

    for name, edges in CASES:
        src, dst, t = stream(SHAPES[name], edges)
        case(name, src, dst, t, 200)
    pl = GraphShape('powerlaw-replica', 10_000_000, 0, 50_000_000, 3, 1e-7, 1.5e6, False, 1.2)
    src, dst, t = stream(pl, 50_000_000, batch=1_000_000, seed=3)
    case('powerlaw-replica (10M nodes)', src, dst, t, 100_000, strategies=('historical', 'inductive'), max_calls=20)
    out['note'] = ('powerlaw tables: T 20 B + F 16 B + mark 4 B per edge = 2.0 GB for 50M edges, far beyond the L2; '
                   'sample times are CUDA events around back-to-back calls with device-resident batches')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--part', choices=['host', 'device'], required=True)
    ap.add_argument('--calls', type=int, default=30)
    ap.add_argument('--out', default='')
    a = ap.parse_args()
    res = host(a.calls) if a.part == 'host' else device()
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, 'w').write(line + '\n')


if __name__ == '__main__':
    main()
