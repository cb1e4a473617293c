"""Time of the encoder's structured call (TPNet.py:313-324, head included, under no_grad) on the sharded state.

    python scripts/sharded_encoder_probe.py --out DIR                    # one GPU
    python -m torch.distributed.run --nproc-per-node 2 scripts/sharded_encoder_probe.py --out DIR --torchrun

One GPU: the plain RandomProjectionModule, ShardedRandomProjection at world 1 (alternated with the plain module,
--repeats times, to show the run-to-run spread), and in-process ranks at world 2 and 4 (LocalPeerGroup, all ranks on
the one GPU: their pulls read local HBM, not NVLink; what they measure is the routing and pull overhead of a rank and
the balance of the positional split), each rank's call split into route + pull and the kernels (pair-wise gram +
head).  --torchrun: one rank per GPU, real NVLink pulls, the call with gather=True (all_gather of the slices) and
without.  Every timed call starts a new cache generation (as the first call after an update does), so it pulls
all the remote rows it reads; the rows pulled per call are counters[NEED].

Shapes: 'reddit' (N = 10,985, d = 140, L = 3, m = 400, K = 20; the state fits L2, so L2 is overwritten with a
256 MiB memset between timed calls, outside the events) and 'large' (a 1,000,001-node power-law replica, d = 210,
L = 3, m = 20,000, K = 20; the rows one call reads, ~1.5 GB, are far larger than L2).  Each timing is CUDA events
around every call, summed over a window of at least --window seconds after warm-up.  Writes DIR/sharded_encoder_probe
.json (one per rank 0 of a --torchrun job) with the device name and power limit read in the same run."""
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

SHAPES = {
    'reddit': dict(N=10985, d=140, L=3, m=400, K=20, B=200, updates=60),
    'large': dict(N=1000001, d=210, L=3, m=20000, K=20, B=100000, updates=8),
}


def device_info(dev):
    out = {'device': torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(dev.index or 0), '--query-gpu=power.limit,clocks.max.sm',
                            '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
        out['power_limit_and_max_sm_clock'] = q
    except (OSError, subprocess.SubprocessError) as e:
        out['power_limit_and_max_sm_clock'] = f'not read: {e}'
    return out


def stream_batches(rng, N, B, n):
    t = 0.0
    for _ in range(n):
        s = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
        d = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
        ts = np.sort(t + rng.random(B) * 100.0)
        t = ts[-1]
        yield s, d, ts


def encoder_inputs(rng, N, m, K, dev):
    # neighbours drawn like the sampler's: popular nodes recur (power law), id 0 pads
    nbr = 1 + (rng.zipf(1.3, (m, K)) - 1) % (N - 1)
    nbr[rng.random((m, K)) < 0.1] = 0
    src = rng.integers(1, N, m)
    dst = rng.integers(1, N, m)
    g = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(dev)      # noqa: E731
    return g(nbr), g(src), g(dst)


def module_kw(sh, dev):
    return dict(node_num=sh['N'], edge_num=10 * sh['N'], dim_factor=1, num_layer=sh['L'], time_decay_weight=1e-6,
                device=str(dev), use_matrix=False, beginning_time=np.float64(0.0), not_scale=False,
                enforce_dim=sh['d'])


def plain_module(sh, dev):
    from tpnet_b200 import RandomProjectionModule
    m = RandomProjectionModule(decay_mode='lazy', init_p0=False, state_device=dev, **module_kw(sh, dev)).to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    with torch.no_grad():
        p0 = m.random_projections[0]
        for lo in range(0, sh['N'], 1 << 20):
            hi = min(lo + (1 << 20), sh['N'])
            p0[lo:hi].copy_(torch.randn(hi - lo, m.dim, device=dev, generator=g) / np.sqrt(m.dim))
    return m


def ext_rows_for(sh, world):
    per = -(-sh['m'] // world)
    return max(per * (sh['K'] + 2), 2 * sh['B']) + 4096


def sharded_module(sh, dev, world=1, rank=0, peers=None):
    from tpnet_b200.sharded import ShardedRandomProjection
    m = ShardedRandomProjection(decay_mode='lazy', ext_rows=ext_rows_for(sh, world), p0='device', state_device=dev,
                                exchange='peer' if world > 1 else 'auto', peers=peers, **module_kw(sh, dev)).to(dev)
    m.init_p0_on_device(seed=0)
    return m


class L2Flush:
    def __init__(self, dev, on):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if on else None

    def __call__(self):
        if self.buf is not None:
            self.buf.zero_()


def timed(calls, flush, window, warmup=5):
    """calls: list of (name, fn, before) — before() runs outside the events.  Returns name -> list of ms per call."""
    for _ in range(warmup):
        for _, fn, before in calls:
            before()
            fn()
    torch.cuda.synchronize()
    res = {name: [] for name, _, _ in calls}
    total = 0.0
    while total < window * 1e3 or len(res[calls[0][0]]) < 20:
        evs = []
        for name, fn, before in calls:
            flush()
            before()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((name, a, b))
        torch.cuda.synchronize()
        for name, a, b in evs:
            ms = a.elapsed_time(b)
            res[name].append(ms)
            total += ms
    return res


def stats(ms):
    a = np.asarray(ms)
    return {'calls': int(a.size), 'mean_ms': float(a.mean()), 'median_ms': float(np.median(a)),
            'p10_ms': float(np.percentile(a, 10)), 'p90_ms': float(np.percentile(a, 90))}


def single_gpu(shape_name, args, dev):
    from tpnet_b200.peer import LocalPeerGroup
    from tpnet_b200 import _lib
    sh = SHAPES[shape_name]
    rng = np.random.default_rng(1)
    batches = list(stream_batches(rng, sh['N'], sh['B'], sh['updates']))
    nbr, src, dst = encoder_inputs(rng, sh['N'], sh['m'], sh['K'], dev)
    flush = L2Flush(dev, shape_name == 'reddit')
    out = {'shape': dict(sh), 'l2': 'overwritten between calls (256 MiB memset)' if flush.buf is not None
           else 'rows read per call far exceed L2'}
    torch.manual_seed(0)
    plain = plain_module(sh, dev)
    one = sharded_module(sh, dev)
    one.mlp.load_state_dict(plain.mlp.state_dict())
    for s, d, t in batches:
        plain.update(s, d, t)
        one.update(s, d, t)
    torch.cuda.synchronize()
    with torch.no_grad():
        a = plain.get_neighbor_pair_wise_feature(nbr, src, dst)
        b = one.get_neighbor_pair_wise_feature(nbr, src, dst)[1]
    out['world1_equals_plain'] = bool(torch.equal(a, b))
    nothing = lambda: None      # noqa: E731
    reps = []
    for r in range(args.repeats):            # alternated: the spread between repeats is the run-to-run noise
        with torch.no_grad():
            res = timed([('plain', lambda: plain.get_neighbor_pair_wise_feature(nbr, src, dst), nothing),
                         ('sharded_world1', lambda: one.get_neighbor_pair_wise_feature(nbr, src, dst), nothing)],
                        flush, args.window)
        reps.append({k: stats(v) for k, v in res.items()})
    out['plain_vs_world1'] = reps
    del plain, one
    torch.cuda.empty_cache()

    for world in (2, 4):
        groups = LocalPeerGroup.create(world)
        ranks = [sharded_module(sh, dev, world, r, groups[r]) for r in range(world)]
        for m in ranks:
            for name in ('state', 'stamps', 'flags'):
                if name in m._peer_bufs:
                    m._peers.publish(name, m._peer_bufs[name])
        for m in ranks:
            m.connect()
        for s, d, t in batches:
            pend = [m.update_begin(s, d, t) for m in ranks]
            torch.cuda.synchronize()
            for m, p in zip(ranks, pend):
                m.update_end(p)
            torch.cuda.synchronize()
        calls, store = [], {}
        k = sh['K']
        for m in ranks:
            per, lo, hi = m._row_split(sh['m'])
            n = hi - lo
            ids = torch.cat([nbr[lo:hi].reshape(-1), src[lo:hi], dst[lo:hi]])

            def route(m=m, ids=ids):
                store[m.rank] = m._route_node_rows(ids)

            def kernels(m=m, n=n):
                rows = store[m.rank]
                nk = n * k
                g = m._nbr_gram_rows((rows[:nk], rows[nk:nk + n], rows[nk + n:]), n, k)
                m._head(g.view(n * k * 2, -1))

            calls.append((f'rank{m.rank}_route_and_pull', route, m._state_written))
            calls.append((f'rank{m.rank}_kernels', kernels, nothing))
            calls.append((f'rank{m.rank}_whole_call', lambda m=m: m.get_neighbor_pair_wise_feature(nbr, src, dst),
                          m._state_written))
        with torch.no_grad():
            res = timed(calls, flush, args.window)
        pulled = []
        for m in ranks:                       # rows pulled by one call (fresh generation)
            m._state_written()
            with torch.no_grad():
                m.get_neighbor_pair_wise_feature(nbr, src, dst)
            torch.cuda.synchronize()
            pulled.append(int(m._shard_tensors['counters'][_lib.SHARD_CTR_NEED].item()))
            m.check_errors()
        out[f'in_process_world{world}'] = {
            'note': 'all ranks on one GPU, one after the other: pulls read local HBM, not NVLink',
            'rows_per_rank': [m._row_split(sh['m'])[2] - m._row_split(sh['m'])[1] for m in ranks],
            'rows_pulled_per_call': pulled, 'times': {k2: stats(v) for k2, v in res.items()}}
        del ranks, calls, store
        torch.cuda.empty_cache()
    return out


def torchrun(shape_name, args, dev):
    import torch.distributed as dist
    from tpnet_b200 import _lib
    sh = SHAPES[shape_name]
    world, rank = dist.get_world_size(), dist.get_rank()
    rng = np.random.default_rng(1)
    batches = list(stream_batches(rng, sh['N'], sh['B'], sh['updates']))
    nbr, src, dst = encoder_inputs(rng, sh['N'], sh['m'], sh['K'], dev)
    flush = L2Flush(dev, shape_name == 'reddit')
    m = sharded_module(sh, dev, world, rank)
    for s, d, t in batches:
        m.update(s, d, t)
    torch.cuda.synchronize()
    with torch.no_grad():
        res = timed([('call', lambda: m.get_neighbor_pair_wise_feature(nbr, src, dst), m._state_written),
                     ('call_gather', lambda: m.get_neighbor_pair_wise_feature(nbr, src, dst, gather=True),
                      m._state_written)], flush, args.window)
        m._state_written()
        m.get_neighbor_pair_wise_feature(nbr, src, dst)
    torch.cuda.synchronize()
    pulled = int(m._shard_tensors['counters'][_lib.SHARD_CTR_NEED].item())
    m.check_errors()
    mine = torch.tensor([np.mean(res['call']), np.mean(res['call_gather']), pulled], dtype=torch.float64, device=dev)
    allr = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allr, mine)
    m.close()
    return {'shape': dict(sh), 'world': world,
            'per_rank': [{'call_mean_ms': float(x[0]), 'call_gather_mean_ms': float(x[1]),
                          'rows_pulled_per_call': int(x[2])} for x in allr]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out', required=True)
    ap.add_argument('--shapes', default='reddit,large')
    ap.add_argument('--window', type=float, default=1.0, help='seconds of timed calls per measurement (at least)')
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--torchrun', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device: there is nothing to measure without one')
    rank = 0
    if args.torchrun:
        import torch.distributed as dist
        local = int(os.environ['LOCAL_RANK'])
        torch.cuda.set_device(local)
        dev = torch.device('cuda', local)
        dist.init_process_group('nccl', device_id=dev)
        rank = dist.get_rank()
    else:
        dev = torch.device('cuda', 0)
    result = {'what': 'encoder structured call with head, no_grad, sharded state', **device_info(dev), 'shapes': {}}
    for name in args.shapes.split(','):
        result['shapes'][name] = (torchrun if args.torchrun else single_gpu)(name, args, dev)
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, 'sharded_encoder_probe' + ('_torchrun' if args.torchrun else '') + '.json')
        with open(path, 'w') as fh:
            json.dump(result, fh, indent=1)
        print(json.dumps(result, indent=1))
    if args.torchrun:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
