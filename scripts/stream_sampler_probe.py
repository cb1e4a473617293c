"""Time of the streaming `recent` sampler (StreamingRecentSampler, tpn_stream_sampler_*).

    python scripts/stream_sampler_probe.py --out DIR [--batches 40] [--tpnet-batch 100000] [--tpnet-steps 4]

Three measurements, one JSON file (DIR/stream_sampler_probe.json) with the device name and power limit read in the
same run:

1. power_law: the power-law stream (synth.edge_stream(SHAPES['powerlaw'], 100,000, ...), full N = 10,000,001,
   max_neighbors = 20).  After --warm batches, CUDA events around every push and around the 3B queries of its batch
   (src, dst and negatives at the batch's times, K = 20), summed over --batches batches.  The sampler's tables
   (9.8 GB) are far larger than L2.  Algorithmic bytes are counted below from the shapes and each batch's distinct
   nodes (the fold rewrites two lists per node that the previous batch touched).
2. tpnet_step: the whole projection side of one TPNet batch in the full shape (p = 8K + 2 = 162 pair encodes per
   edge, BASELINE.md §2) at N = 10,000,001, d = 210, L = 3, lazy decay, as ONE CUDA graph per batch (StepGraphs with
   a custom step): push -> the 3B queries -> two structured encoder calls (positive and negative rows) with the
   head -> two decoder calls -> update.  CUDA events around every replay after one warm-up replay.
3. reddit: the Reddit shape, the query time of RecentNeighborSampler (CSR of the whole stream) and of the streaming
   sampler on the same 3B queries of every batch, side by side (everything L2-resident at this size).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import RandomProjectionModule, synth  # noqa: E402
from tpnet_b200.neighbor_sampler import RecentNeighborSampler, StreamingRecentSampler  # noqa: E402
from tpnet_b200.pipeline import EpochBatches, StepGraphs  # noqa: E402

K = 20


def device_info(dev):
    out = {'device': torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(dev.index or 0), '--query-gpu=power.limit,clocks.max.sm',
                            '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
        out['power_limit_and_max_sm_clock'] = q
    except (OSError, subprocess.SubprocessError) as e:
        out['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return out


def push_bytes(B, prev_nodes, N, C):
    """HBM bytes one push moves: inputs; the radix passes (key + value read and written) and the pending arrays
    written; the fold of the previous batch (pending entries read; per node it touched, ALL read and written, OLD
    written, the counts and newest time)."""
    E = 2 * B
    passes = max(1, math.ceil(N.bit_length() / 8))
    sort = passes * E * 16 + E * 8
    pending = E * (4 + 24)
    fold = E * (4 + 24) + prev_nodes * (3 * 24 * C + 16)
    return 32 * B + sort + pending + fold


def query_bytes(n, C, K_):
    """n queries: id and time read, three [n, K] outputs written, at most K list entries read, per node the counts
    and newest time."""
    return n * (16 + 24 * K_ + 24 * K_ + 16)


def events_time(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    return a, b


def power_law(args, dev):
    shape = synth.SHAPES['powerlaw']
    N, B = shape.node_num, 100_000
    rng = np.random.default_rng(5)
    s = StreamingRecentSampler(N, K, dev, max_batch=B)
    n = args.warm + args.batches
    pushes, queries, pbytes, qbytes = [], [], 0, 0
    prev_nodes = 0
    for i, (src, dst, t) in enumerate(synth.edge_stream(shape, B, n, seed=1)):
        eid = np.arange(i * B + 1, (i + 1) * B + 1, dtype=np.int64)
        neg = rng.integers(1, N, B).astype(np.int64)
        d = [torch.from_numpy(a).to(dev) for a in (src, dst, eid, t)]
        qn = torch.from_numpy(np.concatenate([src, dst, neg])).to(dev)
        qt = torch.from_numpy(np.tile(t, 3)).to(dev)
        torch.cuda.synchronize(dev)
        p = events_time(lambda: s.push(*d))
        q = events_time(lambda: s.get_historical_neighbors(qn, qt, K, as_tensors=True))
        nodes = len(np.unique(np.concatenate([src, dst])))
        if i >= args.warm:
            pushes.append(p)
            queries.append(q)
            pbytes += push_bytes(B, prev_nodes, N, K)
            qbytes += query_bytes(3 * B, K, K)
        prev_nodes = nodes
    torch.cuda.synchronize(dev)
    s.check_errors()
    pt = sum(a.elapsed_time(b) for a, b in pushes) / 1e3
    qt_ = sum(a.elapsed_time(b) for a, b in queries) / 1e3
    nb = len(pushes)
    out = {'num_nodes': N, 'batch': B, 'max_neighbors': K, 'K': K, 'timed_batches': nb, 'warm_batches': args.warm,
           'table_bytes': N * (48 * K + 16),
           'push_ms': 1e3 * pt / nb, 'queries_3B_ms': 1e3 * qt_ / nb,
           'push_plus_queries_ms': 1e3 * (pt + qt_) / nb,
           'push_algorithmic_bytes': pbytes // nb, 'queries_algorithmic_bytes': qbytes // nb,
           'push_GBps': pbytes / pt / 1e9, 'queries_GBps': qbytes / qt_ / 1e9}
    del s
    torch.cuda.empty_cache()
    return out


def tpnet_step(args, dev):
    shape = synth.SHAPES['powerlaw']
    N, B = shape.node_num, args.tpnet_batch
    n = args.tpnet_steps + 1
    rng = np.random.default_rng(7)
    parts = list(synth.edge_stream(shape, B, n, seed=2))
    src = np.concatenate([p[0] for p in parts])
    dst = np.concatenate([p[1] for p in parts])
    t = np.concatenate([p[2] for p in parts])
    neg = rng.integers(1, N, len(src)).astype(np.int64)
    eid = np.arange(1, len(src) + 1, dtype=np.int64)
    m = RandomProjectionModule(node_num=N, edge_num=shape.edge_num, dim_factor=shape.dim_factor,
                               num_layer=shape.num_layer, time_decay_weight=shape.time_decay_weight, device=str(dev),
                               use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=-1,
                               decay_mode='lazy', init_p0=False, state_device=dev).to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    with torch.no_grad():
        p0 = m.random_projections[0]
        for lo in range(0, N, 1 << 20):
            hi = min(lo + (1 << 20), N)
            p0[lo:hi].copy_(torch.randn(hi - lo, m.dim, device=dev, generator=g) / math.sqrt(m.dim))
    s = StreamingRecentSampler(N, K, dev, max_batch=B)
    batches = EpochBatches(src, dst, t, B, dev, extra={'eid': eid, 'neg': neg})
    F = m.pair_wise_feature_dim
    out = {'enc_pos': torch.empty(2 * B, K, 2 * F, device=dev), 'enc_neg': torch.empty(2 * B, K, 2 * F, device=dev),
           'pos': torch.empty(B, F, device=dev), 'neg': torch.empty(B, F, device=dev)}

    def step(module, b, o):
        s.push(b.src, b.dst, b.extra['eid'], b.t)
        rows = torch.cat([b.src, b.dst, b.extra['neg']])
        nbr, _, _ = s.get_historical_neighbors(rows, torch.cat([b.t, b.t, b.t]), K, as_tensors=True)
        n_ = len(b)
        s2 = torch.cat([b.src, b.src])
        module.get_neighbor_pair_wise_feature(nbr[:2 * n_], s2, torch.cat([b.dst, b.dst]), out=o['enc_pos'])
        module.get_neighbor_pair_wise_feature(torch.cat([nbr[:n_], nbr[2 * n_:]]), s2,
                                              torch.cat([b.extra['neg'], b.extra['neg']]), out=o['enc_neg'])
        module.get_pair_wise_feature(b.src, b.dst, out=o['pos'])
        module.get_pair_wise_feature(b.src, b.extra['neg'], out=o['neg'])
        module.update(b.src, b.dst, b.t, next_time=b.t_last)

    with torch.no_grad():
        graphs = StepGraphs(m, list(batches), step=step, out=out, max_batch=B)
        times = []
        for i in range(len(graphs)):
            a, b_ = events_time(lambda: graphs.replay(i))
            if i >= 1:
                times.append((a, b_))
        torch.cuda.synchronize(dev)
    s.check_errors()
    m.check_errors()
    sec = sum(a.elapsed_time(b_) for a, b_ in times) / 1e3
    pairs = 8 * B * K + 2 * B
    res = {'num_nodes': N, 'dim': m.dim, 'num_layer': m.num_layer, 'decay_mode': 'lazy', 'batch': B, 'K': K,
           'pair_encodes_per_edge': pairs // B, 'timed_steps': len(times), 'step_ms': 1e3 * sec / len(times),
           'edges_per_s': B * len(times) / sec, 'pair_encodes_per_s': pairs * len(times) / sec}
    del graphs, m, s, batches, out
    torch.cuda.empty_cache()
    return res


def reddit(args, dev):
    shape = synth.SHAPES['reddit']
    B, n = 600, args.reddit_batches
    rng = np.random.default_rng(3)
    parts = list(synth.edge_stream(shape, B, n, seed=4))
    src = np.concatenate([p[0] for p in parts])
    dst = np.concatenate([p[1] for p in parts])
    t = np.concatenate([p[2] for p in parts])
    eid = np.arange(1, len(src) + 1, dtype=np.int64)
    N = shape.node_num
    csr = RecentNeighborSampler(src, dst, eid, t, dev, num_nodes=N)
    s = StreamingRecentSampler(N, K, dev, max_batch=B)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    t_csr, t_stream = [], []
    for i in range(n):
        lo, hi = i * B, (i + 1) * B
        s.push(up(src[lo:hi]), up(dst[lo:hi]), up(eid[lo:hi]), up(t[lo:hi]))
        qn = up(np.concatenate([src[lo:hi], dst[lo:hi], rng.integers(1, N, B)]))
        qt = up(np.tile(t[lo:hi], 3))
        a = events_time(lambda: csr.get_historical_neighbors(qn, qt, K, as_tensors=True))
        b = events_time(lambda: s.get_historical_neighbors(qn, qt, K, as_tensors=True))
        if i >= args.warm:
            t_csr.append(a)
            t_stream.append(b)
    torch.cuda.synchronize(dev)
    s.check_errors()
    c = sum(x.elapsed_time(y) for x, y in t_csr) / len(t_csr)
    st = sum(x.elapsed_time(y) for x, y in t_stream) / len(t_stream)
    return {'num_nodes': N, 'batch': B, 'queries_per_call': 3 * B, 'K': K, 'timed_calls': len(t_csr),
            'csr_query_us': 1e3 * c, 'stream_query_us': 1e3 * st}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--warm', type=int, default=10)
    ap.add_argument('--batches', type=int, default=40)
    ap.add_argument('--tpnet-batch', type=int, default=100_000)
    ap.add_argument('--tpnet-steps', type=int, default=4)
    ap.add_argument('--reddit-batches', type=int, default=400)
    ap.add_argument('--skip', default='', help='comma-separated parts to skip: power_law,tpnet_step,reddit')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('stream_sampler_probe measures on a CUDA device; none found')
    dev = torch.device('cuda', torch.cuda.current_device())
    skip = set(filter(None, args.skip.split(',')))
    res = {'device_info': device_info(dev)}
    for name, fn in (('reddit', reddit), ('power_law', power_law), ('tpnet_step', tpnet_step)):
        if name not in skip:
            res[name] = fn(args, dev)
            print(name, json.dumps(res[name]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'stream_sampler_probe.json'), 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
