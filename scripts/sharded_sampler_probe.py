"""Time and memory of the node-sharded streaming sampler (ShardedStreamingSampler, tpn_stream_shard_*).

    python scripts/sharded_sampler_probe.py --out DIR [--batches 12] [--warm 4] [--worlds 2,4]
    python -m torch.distributed.run --nproc-per-node 8 scripts/sharded_sampler_probe.py --out DIR    # real ranks

The power-law stream (synth.SHAPES['powerlaw']: N = 10,000,001, B = 100,000 edges per batch), C = K = 20, 3B queries
per batch (src, dst and negatives at the batch's times).  One JSON file (DIR/sharded_sampler_probe.json, or
sharded_sampler_probe_world{G}.json under torchrun) with the device name and power limit read in the same run.

1. world1: StreamingRecentSampler and a world-1 ShardedStreamingSampler fed the same stream, timed batch by batch in
   alternating order (CUDA events around push and around the 3B queries); means and the spread of the per-round means.
2. in_process (one GPU, LocalPeerGroup): at each world in --worlds, every rank's push (sort + fold) and its
   route + pull + query of its slice, each rank timed alone on the GPU, and the cache rows it pulled.  The ranks share
   one GPU's HBM, so the pulls are local copies: this measures the kernels, not NVLink.
3. torchrun: the same per-rank times with real ranks (NVLink pulls, flag barriers); each rank's timings are gathered
   on rank 0.
Device memory per rank: the bytes the rank's tables, cache, pending arrays, workspace and mark table hold, against
the replicated sampler's num_nodes * (48 C + 16).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import _lib, synth  # noqa: E402
from tpnet_b200.neighbor_sampler import ShardedStreamingSampler, StreamingRecentSampler  # noqa: E402

K = 20
B = 100_000


def device_info(dev):
    out = {'device': torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(dev.index or 0), '--query-gpu=power.limit,clocks.max.sm',
                            '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
        out['power_limit_and_max_sm_clock'] = q
    except (OSError, subprocess.SubprocessError) as e:
        out['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return out


def stream(n, dev, seed=1):
    shape = synth.SHAPES['powerlaw']
    rng = np.random.default_rng(seed + 4)
    for i, (src, dst, t) in enumerate(synth.edge_stream(shape, B, n, seed=seed)):
        eid = np.arange(i * B + 1, (i + 1) * B + 1, dtype=np.int64)
        neg = rng.integers(1, shape.node_num, B).astype(np.int64)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
        yield [up(a) for a in (src, dst, eid, t)], up(np.concatenate([src, dst, neg])), up(np.tile(t, 3))


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    return (a, b), r


def ms(pairs):
    return [a.elapsed_time(b) for a, b in pairs]


def sampler_bytes(s):
    ts = list(s._lists.values()) + [s._all_cnt, s._old_cnt, s._newest, s._ws] + list(s._pend.values())
    ts += [getattr(s, k) for k in ('_mark', '_need') if hasattr(s, k)]
    return int(sum(t.numel() * t.element_size() for t in ts))


def world1(args, dev):
    N = synth.SHAPES['powerlaw'].node_num
    plain = StreamingRecentSampler(N, K, dev, max_batch=B)
    one = ShardedStreamingSampler(N, K, dev, max_batch=B)
    times = {'plain': ([], []), 'sharded_world1': ([], [])}
    same = True
    for i, (d, qn, qt) in enumerate(stream(args.warm + args.batches, dev)):
        order = (('plain', plain), ('sharded_world1', one))
        for name, s in (order if i % 2 == 0 else order[::-1]):
            torch.cuda.synchronize(dev)
            p, _ = timed(lambda: s.push(*d))
            q, res = timed(lambda: s.get_historical_neighbors(qn, qt, K, as_tensors=True))
            if i >= args.warm:
                times[name][0].append(p)
                times[name][1].append(q)
            if name == 'plain':
                want = res
            else:
                got = res[1:]
        torch.cuda.synchronize(dev)
        same &= all(torch.equal(a, b) for a, b in zip(got, want))
    plain.check_errors()
    one.check_errors()
    out = {'num_nodes': N, 'batch': B, 'K': K, 'queries_per_batch': 3 * B, 'timed_batches': args.batches,
           'answers_bit_equal': bool(same)}
    rounds = 4
    for name, (p, q) in times.items():
        tot = np.array(ms(p)) + np.array(ms(q))
        per_round = [float(np.mean(c)) for c in np.array_split(tot, rounds)]
        out[name] = {'push_ms': float(np.mean(ms(p))), 'queries_3B_ms': float(np.mean(ms(q))),
                     'push_plus_queries_ms': float(np.mean(tot)), 'round_means_ms': per_round,
                     'round_spread_ms': max(per_round) - min(per_round), 'device_bytes': sampler_bytes(
                         plain if name == 'plain' else one)}
    del plain, one
    torch.cuda.empty_cache()
    return out


def per_rank_summary(push, query, pulled):
    return {'push_ms': float(np.mean(push)), 'route_pull_query_ms': float(np.mean(query)),
            'cache_rows_pulled_per_batch': float(np.mean(pulled))}


def in_process(args, dev, world):
    from tpnet_b200.peer import LocalPeerGroup
    N = synth.SHAPES['powerlaw'].node_num
    groups = LocalPeerGroup.create(world)
    ranks = [ShardedStreamingSampler(N, K, dev, max_batch=B, peers=groups[r], cache_rows=args.cache_rows)
             for r in range(world)]
    for s in ranks:
        s.connect()
    push = [[] for _ in ranks]
    query = [[] for _ in ranks]
    pulled = [[] for _ in ranks]
    for i, (d, qn, qt) in enumerate(stream(args.warm + args.batches, dev)):
        pe = []
        for s in ranks:                       # each rank alone on the GPU: its own kernels' time
            e, _ = timed(lambda: s.push(*d))
            torch.cuda.synchronize(dev)
            pe.append(e)
        qe = []
        for s in ranks:
            e, _ = timed(lambda: s.get_historical_neighbors(qn, qt, K, as_tensors=True))
            torch.cuda.synchronize(dev)
            qe.append(e)
        if i >= args.warm:
            for r, s in enumerate(ranks):
                push[r].append(pe[r][0].elapsed_time(pe[r][1]))
                query[r].append(qe[r][0].elapsed_time(qe[r][1]))
                pulled[r].append(int(s._counters[_lib.SHARD_CTR_NEED].item()))
    for s in ranks:
        s.check_errors()
    out = {'world': world, 'num_nodes': N, 'batch': B, 'K': K, 'cache_rows': args.cache_rows,
           'replicated_table_bytes': N * (48 * K + 16),
           'ranks': [dict(per_rank_summary(push[r], query[r], pulled[r]), rank=r, n_local=s.n_local,
                          table_bytes=(s.n_local + s.cache_rows) * (48 * K + 16), device_bytes=sampler_bytes(s))
                     for r, s in enumerate(ranks)]}
    del ranks
    torch.cuda.empty_cache()
    return out


def distributed(args):
    import torch.distributed as dist
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    world, rank = dist.get_world_size(), dist.get_rank()
    N = synth.SHAPES['powerlaw'].node_num
    s = ShardedStreamingSampler(N, K, dev, max_batch=B, cache_rows=args.cache_rows)
    push, query, pulled = [], [], []
    for i, (d, qn, qt) in enumerate(stream(args.warm + args.batches, dev)):
        dist.barrier()
        p, _ = timed(lambda: s.push(*d))
        q, _ = timed(lambda: s.get_historical_neighbors(qn, qt, K, as_tensors=True))
        torch.cuda.synchronize(dev)
        if i >= args.warm:
            push.append(p[0].elapsed_time(p[1]))
            query.append(q[0].elapsed_time(q[1]))
            pulled.append(int(s._counters[_lib.SHARD_CTR_NEED].item()))
    s.check_errors()
    mine = dict(per_rank_summary(push, query, pulled), rank=rank, n_local=s.n_local,
                table_bytes=(s.n_local + s.cache_rows) * (48 * K + 16), device_bytes=sampler_bytes(s))
    allr = [None] * world
    dist.all_gather_object(allr, mine)
    s.close()
    if rank == 0:
        res = {'device_info': device_info(dev), 'torchrun': {
            'world': world, 'num_nodes': N, 'batch': B, 'K': K, 'cache_rows': args.cache_rows,
            'note': 'push includes the rank barrier before the fold; route_pull_query includes the barrier after it',
            'replicated_table_bytes': N * (48 * K + 16), 'ranks': allr}}
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f'sharded_sampler_probe_world{world}.json'), 'w') as fh:
            json.dump(res, fh, indent=1)
        print(json.dumps(res))
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--warm', type=int, default=4)
    ap.add_argument('--batches', type=int, default=12)
    ap.add_argument('--worlds', default='2,4')
    ap.add_argument('--cache-rows', type=int, default=1 << 18)
    ap.add_argument('--skip', default='', help='comma-separated parts to skip: world1,in_process')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('sharded_sampler_probe measures on a CUDA device; none found')
    if int(os.environ.get('WORLD_SIZE', '1')) > 1:
        return distributed(args)
    dev = torch.device('cuda', torch.cuda.current_device())
    skip = set(filter(None, args.skip.split(',')))
    res = {'device_info': device_info(dev)}
    if 'world1' not in skip:
        res['world1'] = world1(args, dev)
        print('world1', json.dumps(res['world1']), flush=True)
    if 'in_process' not in skip:
        res['in_process'] = [in_process(args, dev, int(w)) for w in args.worlds.split(',')]
        print('in_process', json.dumps(res['in_process']), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'sharded_sampler_probe.json'), 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
