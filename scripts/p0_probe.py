"""Cost of drawing P_0 at the 10M-node scale: the counter-based tpn_init_projection against the torch draws.

    python scripts/p0_probe.py [--out profiles/p0_probe_b200.json]

Workload: N = 10,000,001 nodes, d = 210, L = 3 (P_0 is 8.4 GB of fp32, inside a 34.6 GB packed state).  Timed with
CUDA events, 10 calls after 2 warm-up calls each:
  - tpn_init_projection of the whole P_0 (what a reset of a ``p0_seed`` module writes; the one-GPU layout);
  - the in-place device ``normal_`` the one-GPU reset does at this size (torch's RNG);
  - ``ShardedRandomProjection.init_p0_on_device`` at world 1 (p0='device');
and, by wall clock on the host, the ``torch.normal`` of ``p0='global'`` at 1,000,001 nodes (one tenth of the graph:
every rank draws the whole matrix in that mode).  Bandwidth = fp32 bytes of P_0 written over the time.  The card's
name and power limit are read in the same run.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import RandomProjectionModule  # noqa: E402
from tpnet_b200.sharded import ShardedRandomProjection  # noqa: E402

N, D, L = 10_000_001, 210, 3
HOST_N = 1_000_001
WARMUP, CALLS = 2, 10


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'torch_device_name': torch.cuda.get_device_name(0), 'nvidia_smi': r.stdout.strip().splitlines()}


def time_device(fn):
    for _ in range(WARMUP):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(CALLS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def summary(ms, nbytes):
    ms = np.asarray(ms, dtype=np.float64)
    return {'ms_mean': float(ms.mean()), 'ms_min': float(ms.min()), 'ms_max': float(ms.max()), 'ms_all': ms.tolist(),
            'bytes_written': int(nbytes), 'GB_per_s_mean': float(nbytes / (ms.mean() * 1e-3) / 1e9)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'p0_probe_b200.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('p0_probe needs a CUDA device')
    dev = torch.device('cuda:0')
    kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=1e-4, device=str(dev),
              use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=D, decay_mode='eager')
    p0_bytes = N * D * 4
    res = {'workload': {'nodes': N, 'dim': D, 'num_layer': L, 'p0_bytes': p0_bytes, 'warmup': WARMUP, 'calls': CALLS},
           'gpu': gpu_info()}

    m = RandomProjectionModule(state_device=dev, p0_seed=1, **kw)
    draws = iter(range(1, 10 ** 6))

    def counter():
        m.p0_draw = next(draws)
        m._write_counter_p0()
    res['tpn_init_projection'] = summary(time_device(counter), p0_bytes)
    p0 = m.random_projections[0]
    std = 1 / math.sqrt(D)
    with torch.no_grad():
        res['torch_normal_inplace_reset'] = summary(time_device(lambda: p0.normal_(mean=0, std=std)), p0_bytes)
    del m, p0
    torch.cuda.empty_cache()

    sh = ShardedRandomProjection(ext_rows=1024, state_device=dev, p0='device', **kw)
    seeds = iter(range(1, 10 ** 6))
    res['init_p0_on_device'] = summary(time_device(lambda: sh.init_p0_on_device(next(seeds))), p0_bytes)
    del sh
    torch.cuda.empty_cache()

    torch.normal(0, std, (HOST_N, D))
    wall = []
    for _ in range(CALLS):
        t0 = time.perf_counter()
        torch.normal(0, std, (HOST_N, D))
        wall.append((time.perf_counter() - t0) * 1e3)
    res['host_torch_normal_global'] = dict(summary(wall, HOST_N * D * 4), nodes=HOST_N,
                                           host_threads=torch.get_num_threads())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: (v.get('ms_mean'), v.get('GB_per_s_mean')) for k, v in res.items() if 'ms_mean' in v}))
    print(res['gpu'])


if __name__ == '__main__':
    main()
