#!/usr/bin/env python
"""bench.py — temporal edges/sec through the walk-projection hot path (update + pair-wise
encode) on synthetic graphs of the BASELINE.json shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload powerlaw|reddit|wikipedia|flights] [--dump-outputs DIR]

Primary workload (all N): BASELINE.json configs[3], the one its metric ("... at 1/2/4/8 B200;
% HBM roofline") is quoted on — a power-law temporal graph with 10M nodes, d=210, L=3, lazy
decay, batches of 100,000 edges, p=2 pair-encodes per edge (the decoder shape of
models/modules.py:112: (src,dst) and (src,neg)), `self.mlp` included.  It fits one GPU (34.6 GB
state).  The roofline fraction uses SURVEY.md 8(d)'s ALGORITHMIC bytes (no credit for duplicate
rows); with zipf endpoints most duplicate rows are L2 hits, so the measured DRAM traffic
(`roofline.traffic`, ncu) is far below that figure — see DESIGN.md section 6.
N>1: the state is sharded by node id (tpnet_b200/sharded.py): routing, NVLink pulls of remote rows and
rank barriers all run on the device, the whole step is one CUDA graph per rank; weak scaling by default —
every GPU brings 100,000 edges per step, the job's batch is 100,000 x N (`--scaling strong` splits one
100,000-edge batch instead).  The N>1 line ends with a `parity` block: a down-scaled replica updated
sharded and on one GPU, compared bit for bit.
At N=1 the line also carries `also.{reddit,wikipedia,flights}`: BASELINE.json configs[1], [0], [2]
(TPNet-batch shapes, B=200, K=20, p=162 — latency-bound, state L2-resident).

One JSON line on stdout (driver contract).  `value`: inputs resident in HBM, CUDA-event time, the
same work as the reference arm (pair-wise encode incl. `self.mlp` + update).  `e2e`: the public numpy API
with pinned H2D of the step's inputs and a scalar result read back per step.  `--impl reference`: the
UNMODIFIED reference class from oracle/_ref/TPNet (installed by oracle/make_ref.py) on the host cores;
the torch-CPU port (oracle/cpu_port.py) only if that copy is missing.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from tpnet_b200.synth import (SHAPES, RecentNeighbors, edge_stream, tpnet_neighbor_batch,  # noqa: E402
                               tpnet_pair_lists)

BATCH = 200                 # TPNet batch (configs[0..2])
NUM_NEIGHBORS = 20
WARM_BATCHES = 400          # untimed: populates P_1..P_L and the neighbour table
PL_BATCH = 100_000          # power-law batch (configs[3])
PL_WARM = 12
METRIC = 'temporal edges/sec (update+pairwise encode)'
REF_THREADS = 3             # the reference pins torch to 3 intra-op threads (train_link_prediction.py:124)
NVLINK_GBS = 900.0          # per direction and GPU (NVLink 5)
CHUNKED_NOTE = ('accumulation=chunked (opt-in, NOT the reference order): a row receiving >= 2048 messages in one update sums '
                'them in chunks of 1024 in order, then the chunk sums in order; deterministic, bit-identical to the oracle\'s '
                'restatement of that order; it removes the hub\'s sequential add chain.  It differs from the reference\'s '
                'sequential fp32 order by up to ~3e-4 of a hub row\'s magnitude on this workload — which is the reference '
                'order\'s own rounding error: against the exact (f64) result the sequential order is off by 2.4e-4, the '
                'chunked one by 3e-6 (profiles/r02_accumulation_order_error.txt)')
REF_DIR = os.path.join(ROOT, 'oracle', '_ref', 'TPNet')
DUMP_BYTES = 64_000_000     # --dump-outputs: at most this much in all
DUMP_STATE_ROWS = 2048


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=None)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='powerlaw', choices=['powerlaw', 'reddit', 'wikipedia', 'flights'])
    ap.add_argument('--decay-mode', default='auto', choices=['auto', 'eager', 'lazy'])
    ap.add_argument('--accumulation', default='reference', choices=['chunked', 'reference'],
                    help='power-law: order in which the messages of one row are added (tpn_state_t::giant_chunk)')
    ap.add_argument('--no-flush', action='store_true', help='small shapes: keep L2 warm between steps')
    ap.add_argument('--no-graphs', action='store_true', help='power-law: launch the steps eagerly instead of as CUDA graphs')
    ap.add_argument('--no-also', action='store_true', help='N=1: skip the secondary measurements')
    ap.add_argument('--e2e-sync-read', action='store_true',
                    help='e2e: read every step\'s result with a blocking .item() instead of the pinned 2-slot ring')
    ap.add_argument('--no-feature-overlap', action='store_true',
                    help='N=1: both decoder calls on one stream (default: the (src, neg) call on the module\'s feature stream)')
    ap.add_argument('--no-prepare', action='store_true',
                    help='N=1: do not start the state-independent half of the update (update_prepare) ahead of the '
                         'pair-wise calls of the same batch')
    ap.add_argument('--no-parity', action='store_true', help='N>1: skip the sharded-vs-single-GPU parity leg')
    ap.add_argument('--exchange', default='auto', choices=['auto', 'peer', 'nccl'], help='N>1: data plane of the sharded state')
    ap.add_argument('--cpu-sample-steps', type=int, default=None)
    ap.add_argument('--no-cpu', action='store_true', help='A/B runs: skip the cpu_baseline leg (the line is then not a bench line)')
    ap.add_argument('--cpu-threads', type=int, default=None, help='--impl reference: host threads (default: all cores)')
    ap.add_argument('--warm-batches', type=int, default=None, help='untimed batches that fill the state')
    ap.add_argument('--pl-nodes', type=int, default=None, help='override the power-law node count (debug)')
    ap.add_argument('--pl-batch', type=int, default=PL_BATCH, help='power-law: edges per step and GPU')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='N > 1: weak = pl_batch edges per GPU and step (job batch pl_batch x N), strong = pl_batch in total')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='power-law, one GPU: after the timed steps, write what the last timed step computed as '
                         'DIR/<name>.npy (float32 / float64), so that two builds can be compared output for output.  '
                         'The other arms (the reddit / wikipedia / flights workloads, the sharded N > 1 path, '
                         '--impl reference) write nothing and refuse the option')
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs is not None and (args.impl != 'ours' or args.workload != 'powerlaw'):
        ap.error('--dump-outputs applies to the power-law workload of --impl ours')
    return args


def peak_gbs():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (burst copy)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def algorithmic_bytes(shape):
    L, d = shape.num_layer, shape.dim
    per_edge = 24 * L * d + 24                                   # SURVEY.md §8(d)
    per_pair = 2 * (L + 1) * d * 4 + (2 * L + 2) ** 2 * 4 + 16
    return per_edge, per_pair


def traffic_note(key):
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(p):
        return json.load(open(p)).get(key)
    return None


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '50', '-i', str(index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = [r for ts, r in self.rows if t0 - 0.15 <= ts <= t1 + 0.15] or [r for _, r in self.rows[-3:]]
        for r in rows:
            p = [x.strip() for x in r.split(',')]
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


# ============================================================================= the reference arm (CPU)
def load_reference_class():
    """The UNMODIFIED reference class from oracle/_ref/TPNet (oracle/make_ref.py), or None."""
    if not os.path.isfile(os.path.join(REF_DIR, 'models', 'TPNet.py')):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    from models.TPNet import RandomProjectionModule as Ref          # the reference's own module
    return Ref


class CpuArm:
    """update / pair_wise of the reference on the host cores: the real class when it is installed
    (kind 'reference'), else the torch-CPU port of its op sequence (kind 'port')."""

    def __init__(self, shape, node_num, t0, with_mlp=True, device='cpu'):
        Ref = load_reference_class() if device == 'cpu' else None
        torch.manual_seed(0)
        if Ref is not None:
            self.kind = 'reference'
            self.m = Ref(node_num=node_num, edge_num=shape.edge_num, dim_factor=shape.dim_factor,
                         num_layer=shape.num_layer, time_decay_weight=shape.time_decay_weight, device='cpu',
                         use_matrix=False, beginning_time=np.float64(t0), not_scale=False, enforce_dim=-1)
            if not with_mlp:
                self.m.mlp = torch.nn.Identity()
            self.update = self.m.update
            self.pair_wise = self.m.get_pair_wise_feature
        else:
            from oracle.cpu_port import CpuWalkProjection          # baseline leg only (see oracle/__init__.py)
            self.kind = 'port'
            self.m = CpuWalkProjection(node_num, shape.dim, shape.num_layer, shape.time_decay_weight, float(t0),
                                       not_scale=False, with_mlp=with_mlp, seed=0, device=device)
            self.update = self.m.update
            self.pair_wise = self.m.pair_wise


# ============================================================================= TPNet-batch workloads (configs[0..2])
def make_steps(shape, n_steps, seed, warm=WARM_BATCHES):
    """Returns (warm_batches, steps).  Each step holds the numpy inputs of one batch."""
    rng = np.random.default_rng(seed + 17)
    nbr = RecentNeighbors(shape.node_num, NUM_NEIGHBORS)
    stream = edge_stream(shape, BATCH, warm + n_steps, seed=seed)
    warm_batches, steps = [], []
    lo, hi = (shape.num_src + 1, shape.num_src + shape.num_dst + 1) if shape.num_dst else (1, shape.num_src + 1)
    for i, (s, d, t) in enumerate(stream):
        if i < warm:
            warm_batches.append((s, d, t))
        else:
            neg = rng.integers(lo, hi, BATCH).astype(np.int64)          # random negative sampling
            pa, pb = tpnet_pair_lists(nbr, s, d)
            na, nb = tpnet_pair_lists(nbr, s, neg)
            steps.append(dict(src=s, dst=d, t=t, neg=neg, enc_pos=(pa, pb), enc_neg=(na, nb),
                              nbr_pos=tpnet_neighbor_batch(nbr, s, d), nbr_neg=tpnet_neighbor_batch(nbr, s, neg)))
        nbr.insert(s, d)
    return warm_batches, steps


def pairs_per_step():
    return 8 * BATCH * NUM_NEIGHBORS + 2 * BATCH


def cpu_tpnet(shape, warm_batches, steps, n_warm, n_timed, threads, with_mlp=True):
    """Times the reference's CPU path on the host cores: same step shape.  Returns (seconds per step, kind)."""
    torch.set_num_threads(threads)
    arm = CpuArm(shape, shape.node_num, float(warm_batches[0][2][0]), with_mlp=with_mlp)
    for s, d, t in warm_batches[-40:]:                      # a short warm stream is enough to fill the rows
        arm.update(s, d, t)

    def one(st):
        with torch.no_grad():
            arm.pair_wise(*st['enc_pos'])
            arm.pair_wise(*st['enc_neg'])
            pos = arm.pair_wise(st['src'], st['dst'])
            neg = arm.pair_wise(st['src'], st['neg'])
            arm.update(st['src'], st['dst'], st['t'])
            res = pos.sum() - neg.sum()
        return float(res)

    for st in steps[:n_warm]:
        one(st)
    t0 = time.perf_counter()
    for st in steps[n_warm:n_warm + n_timed]:
        one(st)
    return (time.perf_counter() - t0) / n_timed, arm.kind


def build_module(shape, device, decay_mode, t0):
    from tpnet_b200 import RandomProjectionModule
    torch.manual_seed(0)
    m = RandomProjectionModule(node_num=shape.node_num, edge_num=shape.edge_num, dim_factor=shape.dim_factor,
                               num_layer=shape.num_layer, time_decay_weight=shape.time_decay_weight,
                               device=str(device), use_matrix=False, beginning_time=np.float64(t0), not_scale=False,
                               enforce_dim=-1, decay_mode=decay_mode)
    return m.to(device)


def to_dev(st, device):
    g = lambda a, dt: torch.from_numpy(a).to(device=device, dtype=dt)     # noqa: E731
    return dict(src=g(st['src'], torch.int64), dst=g(st['dst'], torch.int64), t=g(st['t'], torch.float64),
                neg=g(st['neg'], torch.int64), t_last=float(st['t'][-1]),
                nbr_pos=tuple(g(a, torch.int64) for a in st['nbr_pos']),
                nbr_neg=tuple(g(a, torch.int64) for a in st['nbr_neg']))


def resident_step(m, ds):
    """One step with device-resident inputs, the same work as the reference arm: encoder + decoder pair-wise
    features incl. `self.mlp`, then the update.  The feature tensors are dropped at once: inside a capture their
    memory returns to the graph pool."""
    with torch.no_grad():
        m.get_neighbor_pair_wise_feature(*ds['nbr_pos'])   # encoder: [2B, K, 2F] = 4BK pair blocks (TPNet.py:313-324)
        m.get_neighbor_pair_wise_feature(*ds['nbr_neg'])
        m.get_pair_wise_feature(ds['src'], ds['dst'])
        m.get_pair_wise_feature(ds['src'], ds['neg'])
        m.update(ds['src'], ds['dst'], ds['t'], next_time=ds['t_last'])


READBACK_NOTE = {
    True: '(blocking .item() per step)',
    False: '(D2H copy into a pinned slot every step; the host reads the value of step k after step k+1 is enqueued)',
}


class ResultReader:
    """Device -> host read of every step's scalar result through a 2-slot pinned ring: the value of step k is read on
    the host after step k+1 has been enqueued (how a loop that accumulates its metric uses it), so the read-back of one
    step does not drain the GPU before the next step's staging starts.  Every step still pays its D2H copy and its
    host-side read inside the timed region; `drain()` reads the last one.  `--e2e-sync-read` restores `.item()`."""

    def __init__(self):
        self.buf = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.ev = [torch.cuda.Event() for _ in range(2)]
        self.k = 0
        self.pending = None
        self.total = 0.0

    def push(self, r):
        i = self.k & 1
        self.buf[i].copy_(r.reshape(1), non_blocking=True)
        self.ev[i].record()
        self.drain()
        self.pending = i
        self.k += 1

    def drain(self):
        if self.pending is not None:
            self.ev[self.pending].synchronize()
            self.total += float(self.buf[self.pending][0])
            self.pending = None


def api_step(m, st, reader=None):
    """One step through the public numpy API, head included, scalar result read back."""
    with torch.no_grad():
        m.get_neighbor_pair_wise_feature(*st['nbr_pos'])       # encoder features (feed the Mixer in TPNet)
        m.get_neighbor_pair_wise_feature(*st['nbr_neg'])
        pos = m.get_pair_wise_feature(st['src'], st['dst'])    # decoder features -> the step's scalar result
        neg = m.get_pair_wise_feature(st['src'], st['neg'])
        m.update(st['src'], st['dst'], st['t'])
        res = pos.sum() - neg.sum()
    if reader is not None:
        reader.push(res)                                       # D2H copy now, host read one step later
        return None
    return float(res.item())                                   # D2H read of the step's result


def time_sampler(shape, warm_batches, steps, device):
    """SURVEY.md 8(f) N2: one TPNet batch samples K recent neighbours for 2B (pos) + 2B (neg) nodes."""
    from tpnet_b200.neighbor_sampler import RecentNeighborSampler
    src = np.concatenate([b[0] for b in warm_batches])
    dst = np.concatenate([b[1] for b in warm_batches])
    t = np.concatenate([b[2] for b in warm_batches])
    eid = np.arange(1, len(src) + 1)
    gs = RecentNeighborSampler(src, dst, eid, t, device, num_nodes=shape.node_num)
    st = steps[0]
    q = np.concatenate([st['src'], st['dst'], st['src'], st['neg']])
    qt = np.tile(st['t'], 4)
    dq, dqt = torch.from_numpy(q).to(device), torch.from_numpy(qt).to(device)
    for _ in range(5):
        gs.get_historical_neighbors(dq, dqt, NUM_NEIGHBORS, as_tensors=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 200
    a.record()
    for _ in range(reps):
        gs.get_historical_neighbors(dq, dqt, NUM_NEIGHBORS, as_tensors=True)
    b.record()
    torch.cuda.synchronize()
    dev_us = a.elapsed_time(b) * 1e3 / reps
    t0 = time.perf_counter()
    for _ in range(50):
        gs.get_historical_neighbors(q, qt, NUM_NEIGHBORS)              # numpy in, numpy out (the reference's interface)
    api_us = (time.perf_counter() - t0) * 1e6 / 50
    out = {'queries_per_batch': int(len(q)), 'num_neighbors': NUM_NEIGHBORS, 'edges_in_graph': int(len(src)),
           'device_us_per_batch': dev_us, 'numpy_api_us_per_batch': api_us}
    cpu_us, kind = None, None
    try:
        if load_reference_class() is not None:
            from utils.DataLoader import Data                        # the reference's own sampler (utils/utils.py:160-224)
            from utils.utils import get_neighbor_sampler
            data = Data(src, dst, t, eid, np.zeros(len(src)))
            q = np.minimum(q, int(max(src.max(), dst.max())))       # its adjacency list ends at the largest id seen
            cs = get_neighbor_sampler(data=data, sample_neighbor_strategy='recent', seed=0)
            kind = 'reference'
        else:
            from oracle.neighbor_sampler import RecentSamplerOracle
            cs = RecentSamplerOracle(src, dst, eid, t)
            kind = 'port'
        cs.get_historical_neighbors(q, qt, NUM_NEIGHBORS)
        t0 = time.perf_counter()
        for _ in range(10):
            cs.get_historical_neighbors(q, qt, NUM_NEIGHBORS)
        cpu_us = (time.perf_counter() - t0) * 1e6 / 10
    except Exception as e:                                           # a baseline leg must never sink the bench line
        kind = f'unavailable: {type(e).__name__}: {e}'
    out['cpu_us_per_batch'] = cpu_us
    out['cpu_kind'] = kind
    return out


def run_tpnet_shape(args, shape, device, K, W, with_cpu=True, sampler_leg=False):
    """Single-GPU TPNet-batch workload (Reddit / Wikipedia / Flights shapes)."""
    per_edge_B, per_pair_B = algorithmic_bytes(shape)
    pps = pairs_per_step()
    warm_n = args.warm_batches if args.warm_batches is not None else WARM_BATCHES
    warm_batches, steps = make_steps(shape, 2 * (K + W), seed=0, warm=warm_n)
    m = build_module(shape, device, args.decay_mode, warm_batches[0][2][0])
    for s, d, t in warm_batches:
        m.update(s, d, t)
    torch.cuda.synchronize()

    from tpnet_b200.pipeline import StepGraphs
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    dsteps = [to_dev(st, device) for st in steps[:K + W]]
    # the product's per-batch CUDA graphs (tpnet_b200/pipeline.py, SURVEY.md 8(f) N3) around this workload's step
    sg = StepGraphs(m, dsteps, step=lambda mod, ds, out: resident_step(mod, ds), out={}, max_batch=BATCH)
    side = torch.cuda.Stream(device)
    pool = torch.cuda.graph_pool_handle()
    for i in range(W):
        sg.replay(i)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    wall0 = time.perf_counter()
    for k in range(K):
        if not args.no_flush:
            flush.zero_()                                   # evict the 126 MB L2 between steps (untimed)
        ev[k][0].record()
        sg.replay(W + k)
        ev[k][1].record()
    torch.cuda.synchronize()
    wall1 = time.perf_counter()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    m.check_errors()

    # dominant kernel (the 4BK-pair encoder launch): each launch alone in a CUDA graph so that no
    # host launch latency sits between the two events; L2 flushed before each
    n_pair = min(K, 100)
    pair_graphs = []
    with torch.cuda.stream(side):
        for k in range(n_pair):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool, stream=side):
                m.neighbor_pair_wise_gram(*dsteps[W + k]['nbr_pos'])
            pair_graphs.append(g)
    torch.cuda.synchronize()
    pev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_pair)]
    for k in range(n_pair):
        flush.zero_()
        pev[k][0].record()
        pair_graphs[k].replay()
        pev[k][1].record()
    torch.cuda.synchronize()
    pair_ms = float(np.mean([a.elapsed_time(b) for a, b in pev]))
    pairs_per_launch = 2 * dsteps[0]['nbr_pos'][0].numel()        # two pair blocks per (row, neighbour)

    api = steps[K + W:]
    reader = None if args.e2e_sync_read else ResultReader()
    for st in api[:W]:
        api_step(m, st, reader)
    if reader is not None:
        reader.drain()
    torch.cuda.synchronize()
    e0 = time.perf_counter()
    for st in api[W:W + K]:
        api_step(m, st, reader)
    if reader is not None:
        reader.drain()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - e0) * 1e3
    h2d = 2 * ((2 * BATCH * NUM_NEIGHBORS + 4 * BATCH) * 8) + 2 * (2 * BATCH * 8) + 3 * BATCH * 8

    peak, peak_src = peak_gbs()
    achieved = pairs_per_launch * per_pair_B / (pair_ms * 1e-3) / 1e9
    step_bytes = BATCH * per_edge_B + pps * per_pair_B
    heads = 4 if shape.num_layer == 3 else 0                 # the fused head exists for F = 64 (L = 3); else cuBLAS via nn.Sequential
    kernels_per_step = 4 + heads + 3                          # 4 pair-wise (+ 4 head) + prep(+sweep) + snapshot + walk
    out = {
        'value': BATCH * K / (dev_ms * 1e-3), 'unit': 'edges/s', 'steps': K, 'warmup': W, 'ms_per_step': dev_ms / K,
        'config': {'workload': (f'{shape.name}-shaped synthetic graph ({shape.num_nodes} nodes, {shape.num_edges} '
                                f'edges), d={shape.dim}, L={shape.num_layer}, batch {BATCH}, K={NUM_NEIGHBORS}, '
                                f'{pps // BATCH} pair-encodes per edge incl. self.mlp, random negatives'),
                   'batch': BATCH, 'num_neighbors': NUM_NEIGHBORS, 'pairs_per_step': pps, 'dim': shape.dim,
                   'num_layer': shape.num_layer, 'node_num': shape.node_num, 'parallelism': 'single GPU',
                   'decay_mode': 'lazy' if m.lazy else 'eager',
                   'l2': 'warm (no flush)' if args.no_flush else 'flushed between steps (256 MiB memset, untimed)',
                   'timing': 'CUDA events per step, one CUDA graph per step (tpnet_b200.pipeline.StepGraphs)',
                   'algorithmic_bytes_per_step': step_bytes,
                   'wall_ms_per_step_incl_flush': (wall1 - wall0) * 1e3 / K},
        'pairs_per_s': pps * K / (dev_ms * 1e-3),
        'algorithmic_GBps_step': step_bytes * K / (dev_ms * 1e-3) / 1e9,
        'roofline': {'bound': 'hbm', 'kernel': 'tpn::pairwise_nbr_kernel (encoder launch: 2B rows x K neighbours = 4BK pair blocks)',
                     'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic_note('reddit_pairwise_dram_bytes_per_launch') if shape.name == 'reddit' else None,
                     'peak_source': peak_src,
                     'launch_us': pair_ms * 1e3, 'pairs_per_launch': pairs_per_launch,
                     'note': 'state (%.1f MB) is L2-resident: algorithmic bytes are served from L2 after first '
                             'touch, so this is a fraction of the HBM copy peak reached out of L2, not DRAM use' %
                             (shape.node_num * (shape.num_layer + 1) * m.row_stride * 4 / 1e6)},
        'e2e': {'value': BATCH * K / (e2e_ms * 1e-3), 'unit': 'edges/s', 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': 4, 'ms_per_step': e2e_ms / K,
                'path': 'RandomProjectionModule.get_pair_wise_feature/update with numpy ids, self.mlp included, scalar '
                        'result read back ' + READBACK_NOTE[bool(args.e2e_sync_read)]},
        'gpu_launches': kernels_per_step * K,
    }
    if sampler_leg:
        out['sampler'] = time_sampler(shape, warm_batches, steps, device)
    if with_cpu:
        threads = os.cpu_count() or 1
        n_cpu = args.cpu_sample_steps or 20
        sec, kind = cpu_tpnet(shape, warm_batches, steps, 2, n_cpu, threads)
        sec3, _ = cpu_tpnet(shape, warm_batches, steps, 2, max(n_cpu // 2, 3), REF_THREADS)
        sec_id, _ = cpu_tpnet(shape, warm_batches, steps, 2, max(n_cpu // 2, 3), threads, with_mlp=False)
        out['cpu_baseline'] = {'value': BATCH / sec, 'unit': 'edges/s', 'cores': threads, 'kind': kind,
                               'sample': f'{n_cpu} steps of the same workload on the host ({kind}, self.mlp included, '
                                         f'{sec * 1e3:.1f} ms/step)',
                               'mlp_identity': {'value': BATCH / sec_id, 'note': 'same, with mlp = nn.Identity() '
                                                                                 '(BASELINE.md section 2)'},
                               'at_reference_threads': {'value': BATCH / sec3, 'cores': REF_THREADS,
                                                        'note': 'torch.set_num_threads(3), the reference\'s own setting '
                                                                '(train_link_prediction.py:124)'}}
    del sg, pair_graphs, m, flush
    torch.cuda.empty_cache()
    return out


# ============================================================================= power-law (sharded) workload
def powerlaw_shape(args):
    shape = SHAPES['powerlaw']
    if args.pl_nodes:
        shape = dataclasses.replace(shape, num_src=int(args.pl_nodes))
    return shape


def powerlaw_steps(shape, B, n, seed=1234):
    """Replicated on every rank (same seed): (src, dst, t, neg) per step."""
    rng = np.random.default_rng(seed)
    out = []
    for s, d, t in edge_stream(shape, B, n, seed=seed):
        neg = rng.integers(1, shape.num_src + 1, B).astype(np.int64)
        out.append((s, d, t, neg))
    return out


def cpu_port_powerlaw(shape, B, n_warm, n_timed, threads, scale_down, device='cpu', with_mlp=True):
    """The reference's CPU path on a down-scaled replica (its eager decay is N-proportional).  device='cpu': the
    reference arm / CPU baseline (the real class when oracle/_ref is installed).  A CUDA device: the port's stock
    ATen op sequence on the GPU (scripts/aten_gpu_baseline.py).  Returns (seconds per step, nodes, kind)."""
    torch.set_num_threads(threads)
    small = dataclasses.replace(shape, num_src=max(shape.num_src // scale_down, 1000))
    arm = CpuArm(dataclasses.replace(small, num_edges=shape.num_edges), small.node_num, 0.0, with_mlp=with_mlp,
                 device=device)
    steps = powerlaw_steps(small, B, n_warm + n_timed)

    def one(st):
        s, d, t, neg = st
        with torch.no_grad():
            pos = arm.pair_wise(s, d)
            ng = arm.pair_wise(s, neg)
            arm.update(s, d, t)
            return float(pos.sum() - ng.sum())

    for st in steps[:n_warm]:
        one(st)
    if device != 'cpu':
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    for st in steps[n_warm:]:
        one(st)                      # ends in float(...): the device is idle again when it returns
    return (time.perf_counter() - t0) / n_timed, small.node_num, arm.kind


def sharded_parity(args, rank, world, device):
    """N > 1: a down-scaled replica (100,001 nodes, same d / L / decay / accumulation, job batches of pl_batch x N
    edges) updated sharded — this very data plane — and, on rank 0, by the plain single-GPU module; the gathered
    sharded state must equal the single-GPU state BIT FOR BIT; routed pair-wise features within fp32 tolerance."""
    import torch.distributed as dist
    from tpnet_b200 import RandomProjectionModule
    from tpnet_b200.sharded import ShardedRandomProjection
    shape = dataclasses.replace(SHAPES['powerlaw'], num_src=100_000)
    B = args.pl_batch * world
    kw = dict(node_num=shape.node_num, edge_num=shape.edge_num, dim_factor=shape.dim_factor, num_layer=shape.num_layer,
              time_decay_weight=shape.time_decay_weight, device=str(device), use_matrix=False,
              beginning_time=np.float64(0.0), not_scale=False, enforce_dim=-1)
    torch.manual_seed(5)
    sh = ShardedRandomProjection(decay_mode='lazy', ext_rows=shape.node_num + 1024, p0='global', state_device=device,
                                 exchange=args.exchange, accumulation=args.accumulation, **kw).to(device)
    ref = None
    if rank == 0:
        torch.manual_seed(5)
        ref = RandomProjectionModule(decay_mode='lazy', accumulation=args.accumulation, **kw).to(device)
    steps = powerlaw_steps(shape, B, 3, seed=99)
    pair_diff = 0.0
    for s, d, t, neg in steps:
        keep, feat = sh.pair_wise_gram(s, neg)
        if ref is not None:
            keep_t = keep if isinstance(keep, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(keep)).to(device)
            want = ref.pair_wise_gram(s, neg)[keep_t]
            pair_diff = max(pair_diff, float((feat - want).abs().max().item()) if feat.numel() else 0.0)
        sh.update(s, d, t)
        if ref is not None:
            ref.update(s, d, t)
    full = sh.gather_global()
    sh.check_errors()
    sh.close()
    out = None
    if rank == 0:
        ref.materialize()
        diff = max(float((full[i] - ref.random_projections[i].data).abs().max().item())
                   for i in range(shape.num_layer + 1))
        equal = all(torch.equal(full[i], ref.random_projections[i].data) for i in range(shape.num_layer + 1))
        out = {'world': world, 'max_abs_diff': diff, 'bit_equal': bool(equal),
               'checked_rows': int(shape.node_num * (shape.num_layer + 1)), 'batches': len(steps), 'batch': B,
               'pairwise_max_abs_diff': pair_diff, 'exchange': sh.exchange,
               'what': 'sharded state (gather_global) vs the single-GPU module on a 100,001-node replica, same '
                       'd/L/decay/accumulation; pair-wise features of the routed call vs the single-GPU call'}
    del sh, ref, full
    torch.cuda.empty_cache()
    dist.barrier()
    return out


def dump_outputs(out_dir, m, feats, step):
    """What one step computed, as .npy files that two builds can be compared on: the decoder features of its calls
    (`feats`: name -> [B, F], self.mlp included) and all L+1 layers of a sample of the rows its update wrote, decay
    applied (get_random_projections).  Samples are drawn with fixed seeds from the step's own ids, so the same inputs
    give the same files; the features are sampled too (with their row indices) only if they would not fit DUMP_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    touched = np.unique(np.concatenate([step[0], step[1]]))
    ids = np.sort(np.random.default_rng(0).choice(touched, min(DUMP_STATE_ROWS, len(touched)), replace=False))
    arrays = {'state_row_ids': ids.astype(np.float64),
              'state_rows': torch.stack(m.get_random_projections(ids)).cpu().numpy()}     # [L+1, rows, d]
    n = len(step[0])
    row_bytes = sum(f.shape[1] for f in feats.values()) * 4
    room = (DUMP_BYTES - 4096 - sum(a.nbytes for a in arrays.values())) // row_bytes
    rows = None
    if n > room:
        rows = np.sort(np.random.default_rng(1).choice(n, room * row_bytes // (row_bytes + 8), replace=False))
        arrays['feature_rows'] = rows.astype(np.float64)
    for name, f in feats.items():
        arrays[name + '_features'] = (f if rows is None else f[torch.from_numpy(rows).to(f.device)]).cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def run_powerlaw(args, rank, world, device, K, W, sampler, accumulation=None, with_e2e=True, dump=None):
    import torch.distributed as dist
    from tpnet_b200.sharded import ShardedRandomProjection
    accumulation = accumulation or args.accumulation
    shape = powerlaw_shape(args)
    # weak scaling (default): every GPU brings its own 100,000 edges per step, so the batch of the whole job is
    # pl_batch x N; strong: the same 100,000-edge batch split over the ranks
    weak = args.scaling == 'weak'
    B = args.pl_batch * (world if weak else 1)
    per_edge_B, per_pair_B = algorithmic_bytes(shape)
    warm_n = args.warm_batches if args.warm_batches is not None else PL_WARM
    n_phase = min(K, 8)
    steps = powerlaw_steps(shape, B, warm_n + 2 * (K + W) + n_phase + 1)
    torch.manual_seed(0)
    # remote rows cached per generation (two pair calls + the update of one batch): at most the owned pairs of
    # both calls plus the owned dst-role messages; sized from the per-rank launch capacity (3.5 / world of a call)
    cap_pairs = min(B, int(B * min(1.0, 3.5 / world)) + 1024)
    ext_rows = 3 * cap_pairs + 4096 if world > 1 else 1024
    m = ShardedRandomProjection(node_num=shape.node_num, edge_num=shape.edge_num, dim_factor=shape.dim_factor,
                                num_layer=shape.num_layer, time_decay_weight=shape.time_decay_weight,
                                device=str(device), use_matrix=False, beginning_time=np.float64(0.0),
                                not_scale=False, enforce_dim=-1, decay_mode='lazy', ext_rows=ext_rows,
                                p0='device', state_device=device, exchange=args.exchange, accumulation=accumulation)
    m = m.to(device)
    m.init_p0_on_device(seed=0)
    peer = world > 1 and m.exchange == 'peer'
    for s, d, t, _ in steps[:warm_n]:
        m.update(s, d, t)
    torch.cuda.synchronize()
    m.check_errors()

    def g(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(device)

    def stage(st):
        """Resident inputs of one step: the (replicated) edge batch as device tensors."""
        s, d, t, neg = st
        return dict(src=g(s), dst=g(d), t=g(t), neg=g(neg), t_last=float(t[-1]), host=st)

    def dev_plan(plan):
        plan.first_rows, plan.second_rows, plan.send_rows = g(plan.first_rows), g(plan.second_rows), g(plan.send_rows)
        return plan

    def stage_nccl(st):
        s, d, t, neg = st
        up, tmsg = m.plan_update(s, d, t)
        return dict(src=s, dst=d, t=t, up=(dev_plan(up), torch.from_numpy(tmsg).to(device)),
                    pos=dev_plan(m.plan_pairs(s, d)), neg=dev_plan(m.plan_pairs(s, neg)))

    nccl = world > 1 and not peer
    res = [(stage_nccl if nccl else stage)(st) for st in steps[warm_n:warm_n + K + W]]

    def resident_pairs(st, which, keep=None):
        with torch.no_grad():
            if world == 1:
                feat = m.get_pair_wise_feature(st['src'], st['dst' if which == 'pos' else 'neg'])[1]
            elif peer:
                feat = m.routed_pair_wise_feature(st['src'], st['dst' if which == 'pos' else 'neg']).feat
            else:
                _, feat = m.pair_wise_gram(None, None, plan=st[which])
                feat = m._head(feat)
        if keep is not None:
            keep[which] = feat

    def resident_update(st):
        if nccl:
            m.update(st['src'], st['dst'], st['t'], plan=st['up'])
        else:
            m.update(st['src'], st['dst'], st['t'], next_time=st['t_last'])

    def resident(st, keep=None):
        if world == 1 and not args.no_prepare:
            # the half of the update that does not write the state starts now, on the module's side stream
            m.update_prepare(st['src'], st['dst'], st['t'], next_time=st['t_last'])
        if world == 1 and not args.no_feature_overlap:
            # the two decoder calls are independent: the head of one overlaps the row gather of the other
            cur, fs = torch.cuda.current_stream(device), m.feature_stream()
            fs.wait_stream(cur)
            with torch.cuda.stream(fs):
                resident_pairs(st, 'neg', keep)
            resident_pairs(st, 'pos', keep)
            cur.wait_stream(fs)
        else:
            resident_pairs(st, 'pos', keep)
            resident_pairs(st, 'neg', keep)
        resident_update(st)

    # Every step is captured once into a CUDA graph and replayed once, in order (the host-side launch latency of
    # the ~20-40 small kernels of a step would otherwise show up as idle gaps).  N > 1, peer data plane: routing,
    # pulls and barriers are kernels too, so the whole sharded step is one graph per rank; the NCCL data plane stays eager.
    use_graphs = not nccl and not args.no_graphs
    side = torch.cuda.Stream(device)
    pool = torch.cuda.graph_pool_handle() if use_graphs else None

    def capture(fn, *a):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, pool=pool, stream=side):
            fn(*a)
        return gr

    # --dump-outputs: the last timed step keeps its decoder features (in its graph's memory pool when captured)
    last = {} if dump else None
    keep = lambda i: last if i == len(res) - 1 else None     # noqa: E731
    if use_graphs:
        with torch.cuda.stream(side):
            graphs = [capture(resident, st, keep(i)) for i, st in enumerate(res)]
        torch.cuda.synchronize()
        run_step = lambda i: graphs[i].replay()              # noqa: E731
    else:
        run_step = lambda i: resident(res[i], keep(i))       # noqa: E731
    if world > 1:
        dist.barrier()
    for i in range(W):
        run_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    wall0 = time.perf_counter()
    for k in range(K):
        ev[k][0].record()
        run_step(W + k)
        ev[k][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall1 = time.perf_counter()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    m.check_errors()
    if dump:
        dump_outputs(dump, m, last, steps[warm_n + K + W - 1])
    del res, last
    if use_graphs:
        del graphs

    # per-phase device time (events around each call) for the roofline of the dominant kernel
    pool = torch.cuda.graph_pool_handle() if use_graphs else None      # the step graphs' pool died with them
    t_pair, t_upd = [], []
    for st in steps[warm_n + K + W:warm_n + K + W + n_phase]:
        r = (stage_nccl if nccl else stage)(st)
        if world > 1:
            dist.barrier()
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        if use_graphs:
            with torch.cuda.stream(side):
                gp, gu = capture(resident_pairs, r, 'pos'), capture(resident_update, r)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            a.record()
            gp.replay()
            b.record()
            gu.replay()
            c.record()
        else:
            a.record()
            resident_pairs(r, 'pos')
            b.record()
            resident_update(r)
            c.record()
        torch.cuda.synchronize()
        t_pair.append(a.elapsed_time(b))
        t_upd.append(b.elapsed_time(c))
    pair_ms, upd_ms = float(np.mean(t_pair)), float(np.mean(t_upd))

    # one instrumented eager step (N > 1, peer): how many remote rows were pulled, and how fast
    exch = None
    if peer:
        st = stage(steps[warm_n + K + W + n_phase])
        ctr = m._shard_tensors['counters']
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        dist.barrier()
        with torch.no_grad():
            m.routed_pair_wise_feature(st['src'], st['dst'])
            m.routed_pair_wise_feature(st['src'], st['neg'])
        rows_pairs = int(ctr[0].item())
        # the pull of the pos call alone, timed (fresh generation: force one by a no-op reload-free reset of the cache)
        m._state_written()
        torch.cuda.synchronize()
        dist.barrier()
        lib_ptrs = m._global_ids_to_device([st['src'], st['dst']], ['id', 'id'])
        from tpnet_b200 import _lib as tl
        lib = tl.load()
        rb = m._route_buffers('pairs', B)
        keep = torch.empty(B, dtype=torch.int64, device=device)
        cnt = torch.zeros(1, dtype=torch.int32, device=device)
        lib.tpn_route_pairs(m._c_shard(), lib_ptrs[0], lib_ptrs[1], B, rb['first'].data_ptr(), rb['second'].data_ptr(),
                            keep.data_ptr(), cnt.data_ptr(), rb['ws'].data_ptr(), rb['ws'].numel(), m._stream())
        m._barrier()
        m._dirty = False
        evs[0].record()
        lib.tpn_pull_rows(m._c_state(), m._c_shard(), m._stream())
        evs[1].record()
        torch.cuda.synchronize()
        rows_pos = int(ctr[0].item())
        pull_ms = evs[0].elapsed_time(evs[1])
        block_bytes = (shape.num_layer + 1) * m.row_stride * 4
        m._state_written()
        dist.barrier()
        # where an eager update spends its time: routing + pull | barrier | rank-local kernels
        ue = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        with torch.no_grad():
            m.routed_pair_wise_feature(st['src'], st['dst'])          # as in a step: the update finds its rows cached
        torch.cuda.synchronize()
        dist.barrier()
        ue[0].record()
        pending = m.update_begin(st['src'], st['dst'], st['t'], st['t_last'])
        ue[1].record()
        m._barrier()
        ue[2].record()
        m.update_end(pending)
        ue[3].record()
        m._barrier()
        ue[4].record()
        torch.cuda.synchronize()
        upd_parts = [ue[i].elapsed_time(ue[i + 1]) for i in range(4)]
        dist.barrier()
        tt = torch.tensor([rows_pairs, rows_pos, pull_ms] + upd_parts, dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        rows_pairs, rows_pos, pull_ms, *upd_parts = [float(x) for x in tt.tolist()]
        exch = {'data_plane': 'device-side routing + NVLink pulls out of the owners\' HBM (IPC-mapped peer memory) + '
                              'flag barriers; no NCCL in the step',
                'rows_cached_per_rank_per_step': rows_pairs, 'bytes_per_rank_per_step': rows_pairs * block_bytes,
                'pull_of_one_pair_call': {'rows': rows_pos, 'ms': pull_ms,
                                          'achieved_GBps': rows_pos * block_bytes / (pull_ms * 1e-3) / 1e9,
                                          'peak_GBps': NVLINK_GBS,
                                          'note': 'upper bound on bytes: never-written rows are not fetched'},
                'eager_update_ms': {'route_and_pull': upd_parts[0], 'barrier': upd_parts[1], 'rank_local_kernels': upd_parts[2],
                                    'barrier_back_to_back': upd_parts[3]},
                'barriers_per_step': 2}

    # end to end: numpy API, routing inside the timed region, head + scalar read-back
    e2e_ms, n_api = float('nan'), 0
    if with_e2e:
        api = steps[warm_n + K + W + n_phase + 1:][:K + W]

        def api_one(st):
            s, d, t, neg = st
            with torch.no_grad():
                if world == 1 and not args.no_prepare:
                    m.update_prepare(s, d, t)
                if peer:
                    pos = m.routed_pair_wise_feature(s, d).feat          # zero rows past the count
                    ng = m.routed_pair_wise_feature(s, neg).feat
                else:
                    # (the two calls on two streams, as in `value`, were measured here too: 0.754 vs 0.723 ms per step —
                    # this path is bound by the host's staging and launch work, not by the device; profiles/r02_ab_variants.txt)
                    _, pos = m.get_pair_wise_feature(s, d)
                    _, ng = m.get_pair_wise_feature(s, neg)
                m.update(s, d, t)
                r = pos.sum() - ng.sum()
            if reader is not None:
                reader.push(r)
                return None
            return float(r.item())

        reader = None if args.e2e_sync_read else ResultReader()
        for st in api[:W]:
            api_one(st)
        if reader is not None:
            reader.drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0 = time.perf_counter()
        n_api = len(api) - W
        for st in api[W:]:
            api_one(st)
        if reader is not None:
            reader.drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e2e_ms = (time.perf_counter() - e0) * 1e3
        m.check_errors()
    wall_end = time.perf_counter()

    tt = torch.tensor([dev_ms, e2e_ms if with_e2e else 0.0, pair_ms, upd_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, pair_ms, upd_ms = [float(x) for x in tt.tolist()]
    barriers = m.barriers
    row_stride = m.row_stride
    m.close()
    del m
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    peak, peak_src = peak_gbs()
    # per rank: B/world * ... under weak scaling every rank owns ~pl_batch pairs per call and ~2*pl_batch messages
    n_pairs_rank, n_msgs_rank = B // world, 2 * B // world
    pair_gbs = n_pairs_rank * per_pair_B / (pair_ms * 1e-3) / 1e9
    upd_gbs = n_msgs_rank * (per_edge_B / 2) / (upd_ms * 1e-3) / 1e9
    # the dominant launch group of a step is the longest single call: the update (one per step) unless one pair-wise
    # call alone takes longer
    dominant_is_update = upd_ms >= pair_ms
    step_bytes = B * per_edge_B + 2 * B * per_pair_B
    block_bytes = (shape.num_layer + 1) * row_stride * 4
    state_gb = shape.node_num * block_bytes / 1e9
    front = 'routing + NVLink pull + barriers + ' if world > 1 else ''
    step_gbs = (step_bytes / world) * K / (dev_ms * 1e-3) / 1e9          # per GPU
    roof = {'bound': 'hbm', 'peak': peak, 'unit': 'GB/s', 'peak_source': peak_src,
            'phases': {'pairwise': {'what': front + 'tpn::pairwise_tma_kernel + tpn::head_tc_kernel (self.mlp on tcgen05), ~%d '
                                            'pairs per rank; the gather kernel alone: profiles/r02m_ncu_full_step_kernels.txt'
                                            % n_pairs_rank, 'ms': pair_ms, 'achieved': pair_gbs, 'frac': pair_gbs / peak},
                       'update': {'what': front + 'sort front end + snapshot + tpn::walk_small_kernel || tpn::walk_hub2_kernel || '
                                          'tpn::walk_stream_kernel (+ combine_giants), ~%d messages per rank' % n_msgs_rank,
                                  'ms': upd_ms, 'achieved': upd_gbs, 'frac': upd_gbs / peak},
                       'step': {'what': 'whole step (two pair-wise calls incl. head + one update, overlapped as in `value`), '
                                        'algorithmic bytes per GPU / step time', 'ms': dev_ms / K, 'achieved': step_gbs,
                                'frac': step_gbs / peak}}}
    tkey = 'powerlaw_update_dram_bytes_per_call' if dominant_is_update else 'powerlaw_pairwise_dram_bytes_per_launch'
    if accumulation == 'chunked' and dominant_is_update:
        tkey = 'powerlaw_update_chunked_dram_bytes_per_call'
    if dominant_is_update:
        roof.update(kernel='update path (sort front end + snapshot + walk_small || walk_hub2 || walk_stream)', achieved=upd_gbs,
                    frac=upd_gbs / peak)
    else:
        roof.update(kernel='tpn::pairwise_tma_kernel (+ head)', achieved=pair_gbs, frac=pair_gbs / peak)
    # ncu DRAM bytes are a property of the N=1 launch: not carried over to the sharded runs
    roof['traffic'] = traffic_note(tkey) if world == 1 else None
    h2d = 3 * B * 8 + 2 * (2 * B * 8)
    upd_launches = 1 + 1 + 1 + 1 + 1 + 1 + 1 + 1                # fused front end (prep + radix passes), payload, giant ordering,
    #                                                             snapshot, walk_stream, hub2, small, stamps
    if accumulation == 'chunked':
        upd_launches -= 1                                       # no giant ordering, no walk_stream; + combine_giants
    per_step = 2 * 2 + upd_launches if world == 1 else (2 * (4 + 1 + 2) + 1 + 4 + 1 + 1 + upd_launches)
    line = {
        'metric': METRIC, 'value': B * K / (dev_ms * 1e-3), 'unit': 'edges/s', 'n_gpus': world, 'steps': K,
        'warmup': W, 'ms_per_step': dev_ms / K, 'higher_is_better': True, 'scaling': 'weak' if weak else 'strong',
        'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': (f'power-law temporal graph, {shape.num_nodes} nodes / {shape.num_edges} edges '
                                f'(BASELINE configs[3]), d={shape.dim}, L={shape.num_layer}, batch {B}, 2 pair-encodes '
                                f'per edge incl. self.mlp (decoder shape), lazy decay'),
                   'batch': B, 'pairs_per_step': 2 * B, 'dim': shape.dim, 'num_layer': shape.num_layer,
                   'node_num': shape.node_num, 'state_GB': state_gb,
                   'accumulation': CHUNKED_NOTE if accumulation == 'chunked' else
                   'reference: one message at a time per row, the order of CPU scatter_add_ (TPNet.py:93-96), bit for bit',
                   'parallelism': 'single GPU' if world == 1 else
                   (f'state sharded by node id over {world} GPUs; per call: device-side routing, remote rows pulled over '
                    f'NVLink from peer memory, {2} flag barriers per step; the step is ONE CUDA graph per rank'
                    if peer else f'state sharded by node id over {world} GPUs, host plan + one all_to_all per call (NCCL)'),
                   'l2': f'no flush needed: {state_gb:.1f} GB state >> 126 MB L2',
                   'timing': ('CUDA events per step, one CUDA graph per step' + (', max over ranks; routing is inside the step'
                                                                                 if world > 1 else '')) if use_graphs else
                             'CUDA events per step, max over ranks; host routing plans are resident inputs',
                   'algorithmic_bytes_per_step': step_bytes, 'wall_ms_per_step': (wall1 - wall0) * 1e3 / K},
        'pairs_per_s': 2 * B * K / (dev_ms * 1e-3),
        'algorithmic_GBps_step': step_bytes * K / (dev_ms * 1e-3) / 1e9,
        'roofline': roof,
        'gpu_launches': K * per_step,
        'exchange': exch,
        'clocks': sampler.window(wall0, wall_end) if sampler else None,
    }
    if with_e2e:
        line['e2e'] = {'value': B * n_api / (e2e_ms * 1e-3), 'unit': 'edges/s', 'h2d_bytes_per_step': h2d,
                       'd2h_bytes_per_step': 4, 'ms_per_step': e2e_ms / n_api,
                       'path': ('ShardedRandomProjection.routed_pair_wise_feature/update with numpy ids: every rank stages '
                                '1/N of each array, the slices are all-gathered over NVLink, routing on the device; '
                                if peer else 'ShardedRandomProjection.get_pair_wise_feature/update with numpy ids; ')
                               + 'self.mlp included, scalar result read back ' + READBACK_NOTE[bool(args.e2e_sync_read)]}
        line['barriers_total'] = barriers
    return line


# ============================================================================= main
def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    threads = args.cpu_threads or os.cpu_count() or 1

    # ---------------- reference arm: the reference's CPU implementation on the host cores, rank 0 only
    if args.impl == 'reference':
        if rank != 0:
            return
        if args.workload == 'powerlaw':
            K = args.steps or 3
            W = min(args.warmup if args.warmup is not None else 1, 2)
            shape = powerlaw_shape(args)
            sec, n_small, kind = cpu_port_powerlaw(shape, args.pl_batch, W, K, threads, scale_down=10)
            val = args.pl_batch / sec
            sample = (f'{K} batches of {args.pl_batch} edges + 2 pair-encodes per edge (self.mlp included) on a '
                      f'{n_small}-node replica (10x fewer nodes: the reference\'s eager decay is N-proportional, so this '
                      f'flatters it)')
            cfg = {'workload': f'power-law temporal graph (BASELINE configs[3]) d={shape.dim} L={shape.num_layer} '
                               f'batch {args.pl_batch}, CPU arm on a 10x down-scaled node set', 'batch': args.pl_batch}
        else:
            shape = SHAPES[args.workload]
            K, W = args.steps or 30, max(args.warmup or 3, 1)
            warm_batches, steps = make_steps(shape, K + W, seed=0, warm=60)
            sec, kind = cpu_tpnet(shape, warm_batches, steps, W, K, threads)
            val = BATCH / sec
            sample = f'{K} steps of the same workload (self.mlp included)'
            cfg = {'workload': f'{shape.name}-shaped synthetic graph, batch {BATCH}, K={NUM_NEIGHBORS}', 'batch': BATCH}
        what = ('the unmodified reference class (oracle/_ref/TPNet, models/TPNet.py:9-157)' if kind == 'reference'
                else 'torch-CPU port of the reference (oracle/cpu_port.py)')
        print(json.dumps({'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'edges/s', 'n_gpus': args.gpus,
                          'steps': K, 'warmup': W, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
                          'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
                          'cpu_baseline': {'value': val, 'unit': 'edges/s', 'cores': threads, 'kind': kind,
                                           'sample': sample + '; ' + what},
                          'e2e': {'value': val, 'unit': 'edges/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return

    # ---------------- our arm
    if not torch.cuda.is_available():
        raise SystemExit('bench.py (impl=ours) needs a CUDA device: there is no CPU fallback')
    if args.dump_outputs is not None and world > 1:
        raise SystemExit('--dump-outputs writes the outputs of a single-GPU run')
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
    from tpnet_b200 import _lib
    _lib.load()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    time.sleep(0.3 if sampler else 0)

    if args.workload == 'powerlaw':
        K, W = args.steps or 20, max(args.warmup if args.warmup is not None else 3, 3)
        line = run_powerlaw(args, rank, world, device, K, W, sampler, dump=args.dump_outputs)
        if world > 1 and not args.no_parity:
            parity = sharded_parity(args, rank, world, device)
            if rank == 0:
                line['parity'] = parity
        if rank == 0:
            if world == 1 and args.no_cpu:
                line['cpu_baseline'] = None
            elif world == 1:
                n_cpu = args.cpu_sample_steps or 3
                shape = powerlaw_shape(args)
                sec, n_small, kind = cpu_port_powerlaw(shape, args.pl_batch, 1, n_cpu, threads, scale_down=10)
                sec3, _, _ = cpu_port_powerlaw(shape, args.pl_batch, 1, 1, REF_THREADS, scale_down=10)
                sec_id, _, _ = cpu_port_powerlaw(shape, args.pl_batch, 1, 1, threads, scale_down=10, with_mlp=False)
                line['cpu_baseline'] = {'value': args.pl_batch / sec, 'unit': 'edges/s', 'cores': threads,
                                        'kind': kind,
                                        'sample': f'{n_cpu} batches on a {n_small}-node replica (10x fewer nodes than '
                                                  f'the GPU run; {kind}, self.mlp included, {sec:.2f} s/step)',
                                        'mlp_identity': {'value': args.pl_batch / sec_id,
                                                         'note': 'same, with mlp = nn.Identity() (BASELINE.md section 2); 1 batch'},
                                        'at_reference_threads': {'value': args.pl_batch / sec3, 'cores': REF_THREADS,
                                                                 'note': 'torch.set_num_threads(3), the reference\'s own '
                                                                         'setting (train_link_prediction.py:124); 1 batch'}}
                if not args.no_also:
                    also = {}
                    other = 'chunked' if args.accumulation == 'reference' else 'reference'
                    alt = run_powerlaw(args, rank, world, device, min(K, 10), W, None, accumulation=other, with_e2e=False)
                    also[other + '_order'] = {k: alt[k] for k in ('value', 'ms_per_step', 'roofline')}
                    also[other + '_order']['note'] = CHUNKED_NOTE if other == 'chunked' else (
                        'same workload with accumulation=reference (strictly sequential adds per row, bit-identical to '
                        'CPU scatter_add_)')
                    also['reddit'] = run_tpnet_shape(args, SHAPES['reddit'], device, 300, 10, with_cpu=True, sampler_leg=True)
                    for name in ('wikipedia', 'flights'):
                        a2 = argparse.Namespace(**vars(args))
                        a2.cpu_sample_steps = args.cpu_sample_steps or 10
                        also[name] = run_tpnet_shape(a2, SHAPES[name], device, 200, 10, with_cpu=True)
                    line['also'] = also
            else:
                line['cpu_baseline'] = None
    else:
        if world > 1:
            raise SystemExit('the TPNet-batch shapes are single-GPU workloads (state 13-32 MB): use --workload powerlaw')
        K, W = args.steps or 300, max(args.warmup if args.warmup is not None else 10, 3)
        t0 = time.perf_counter()
        body = run_tpnet_shape(args, SHAPES[args.workload], device, K, W, with_cpu=True,
                               sampler_leg=args.workload == 'reddit')
        line = {'metric': METRIC, 'n_gpus': 1, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic'}
        line.update(body)
        line['clocks'] = sampler.window(t0, time.perf_counter()) if sampler else None
    if sampler:
        sampler.stop()
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
