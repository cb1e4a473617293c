#!/usr/bin/env python
"""Times tpn_pairwise alone at the flagship shape: the pipelined kernel (default) against the one-shot TMA kernel
(TPN_DEBUG_LEGACY_PAIRWISE), alternated in one process.

The state is bench.py's power-law state (10,000,001 nodes, d = 210, L = 3, lazy decay, ~35 GB: far larger than L2),
after the same warm-up updates.  The pairs are the (src, dst) and (src, neg) decoder calls of bench.py's batches
(zipf ids of tpnet_b200.synth.edge_stream), so L2 hits are what the bench sees.  Per kernel and round: CUDA events
around `--calls` back-to-back 100,000-pair calls, cycling over the batches.

Prints one JSON object: us per call (median and spread over the rounds), algorithmic GB/s (bench.py's per-pair
bytes), unique-block GB/s (node blocks of distinct ids per call + the outputs), and the card, power limit and max SM
clock read in the same run.  ``--nodes`` shrinks the state for a quick check.
"""
import argparse
import dataclasses
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from tpnet_b200 import _lib  # noqa: E402
from tpnet_b200.sharded import ShardedRandomProjection  # noqa: E402

LEGACY = 128                      # TPN_DEBUG_LEGACY_PAIRWISE (include/tpnet_b200.h)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(','))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:        # the numbers are still reported, without their context
        return dict(name=torch.cuda.get_device_name(0), error=str(e))


def timeline(m, steps, flags):
    """Kernel durations and the step span of bench.py's step, captured as bench.py captures it (one CUDA graph per
    step: update_prepare on the side stream, the (src, neg) decoder call on the feature stream, the (src, dst) call,
    then update), replayed under torch.profiler.  Per kernel: mean device time per step; `span_us`: first kernel
    start to last kernel end of a step."""
    import time
    dev = torch.device('cuda:0')
    g = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
    res = [dict(src=g(s), dst=g(d), t=g(t), neg=g(neg), t_last=float(t[-1])) for s, d, t, neg in steps]

    def resident(st):
        with torch.no_grad():
            m.update_prepare(st['src'], st['dst'], st['t'], next_time=st['t_last'])
            cur, fs = torch.cuda.current_stream(dev), m.feature_stream()
            fs.wait_stream(cur)
            with torch.cuda.stream(fs):
                m.get_pair_wise_feature(st['src'], st['neg'])
            m.get_pair_wise_feature(st['src'], st['dst'])
            cur.wait_stream(fs)
            m.update(st['src'], st['dst'], st['t'], next_time=st['t_last'])

    lib = _lib.load()
    side = torch.cuda.Stream(dev)
    pool = torch.cuda.graph_pool_handle()
    old = lib.tpn_set_debug_flags(flags)          # the launch choice is baked in at capture
    try:
        graphs = []
        with torch.cuda.stream(side):
            for st in res:
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr, pool=pool, stream=side):
                    resident(st)
                graphs.append(gr)
        torch.cuda.synchronize()
    finally:
        lib.tpn_set_debug_flags(old)
    for gr in graphs:                             # warm replays
        gr.replay()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for gr in graphs:
            gr.replay()
            torch.cuda.synchronize()
            time.sleep(0.002)                     # a gap that separates the steps in the trace
    ev = sorted(((e.time_range.start, e.time_range.end, e.name) for e in prof.events()
                 if str(e.device_type).endswith('CUDA') and e.time_range.end > e.time_range.start), key=lambda x: x[0])
    groups, last_end = [], None
    for st, en, name in ev:
        if last_end is None or st - last_end > 1000:
            groups.append([])
        groups[-1].append((st, en, name))
        last_end = en if last_end is None else max(last_end, en)
    per = {}
    for g in groups:
        for st, en, name in g:
            n2 = re.sub(r'^void ', '', name.replace('(anonymous namespace)::', ''))
            short = re.match(r'([\w:]*)', n2).group(1).split('::')[-1] or n2[:60]
            per[short] = per.get(short, 0.0) + (en - st)
    n = max(len(groups), 1)
    return dict(steps=len(groups), span_us=round(float(np.mean([max(x[1] for x in g) - g[0][0] for g in groups])), 1),
                kernel_us_per_step={k: round(v / n, 1) for k, v in sorted(per.items(), key=lambda kv: -kv[1])})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--calls', type=int, default=200)
    ap.add_argument('--batches', type=int, default=8)
    ap.add_argument('--nodes', type=int, default=0, help='sources of the power-law shape (default: the bench shape)')
    ap.add_argument('--timeline', type=int, default=0,
                    help='also trace this many bench steps (StepGraphs replays) per kernel with torch.profiler')
    args = ap.parse_args()

    dev = torch.device('cuda:0')
    shape = bench.SHAPES['powerlaw']
    if args.nodes:
        shape = dataclasses.replace(shape, num_src=args.nodes)
    B = bench.PL_BATCH
    steps = bench.powerlaw_steps(shape, B, bench.PL_WARM + args.batches)
    torch.manual_seed(0)
    m = ShardedRandomProjection(node_num=shape.node_num, edge_num=shape.edge_num, dim_factor=shape.dim_factor,
                                num_layer=shape.num_layer, time_decay_weight=shape.time_decay_weight,
                                device=str(dev), use_matrix=False, beginning_time=np.float64(0.0), not_scale=False,
                                enforce_dim=-1, decay_mode='lazy', ext_rows=1024, p0='device', state_device=dev)
    m = m.to(dev)
    m.init_p0_on_device(seed=0)
    for s, d, t, _ in steps[:bench.PL_WARM]:
        m.update(s, d, t)
    torch.cuda.synchronize()
    m.check_errors()

    lib = _lib.load()
    st = m._c_state()
    stream = torch.cuda.current_stream().cuda_stream
    F = m.pair_wise_feature_dim
    out = torch.empty(B, F, dtype=torch.float32, device=dev)
    calls = []
    uniq = []
    for s, d, _, neg in steps[bench.PL_WARM:]:
        for b in (d, neg):
            calls.append((torch.from_numpy(s).to(dev), torch.from_numpy(b).to(dev)))
            uniq.append(len(np.unique(s)) + len(np.unique(b)))
    _, per_pair = bench.algorithmic_bytes(shape)
    block = (shape.num_layer + 1) * m.row_stride * 4
    uniq_bytes = float(np.mean(uniq)) * block + B * F * 4

    def run(flags, n_calls):
        old = lib.tpn_set_debug_flags(flags)
        try:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n_calls):
                a, b = calls[i % len(calls)]
                rc = lib.tpn_pairwise(st, a.data_ptr(), b.data_ptr(), B, None, 1, out.data_ptr(), stream)
                if rc:
                    _lib.check(rc, 'tpn_pairwise')
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e3 / n_calls
        finally:
            lib.tpn_set_debug_flags(old)

    for flags in (0, LEGACY):
        run(flags, 20)                                       # warm-up: modules, attributes, L2
    rounds = {'pipelined': [], 'legacy': []}
    for _ in range(args.rounds):
        rounds['pipelined'].append(run(0, args.calls))
        rounds['legacy'].append(run(LEGACY, args.calls))
    m.check_errors()

    res = dict(what='tpn_pairwise alone, 100,000-pair zipf decoder calls at the bench shape',
               shape=dict(nodes=shape.node_num, dim=shape.dim, layers=shape.num_layer, row_stride=m.row_stride,
                          decay='lazy', pairs_per_call=B),
               card=card(), rounds=args.rounds, calls_per_round=args.calls,
               algorithmic_bytes_per_call=per_pair * B, unique_block_bytes_per_call=uniq_bytes)
    for k, v in rounds.items():
        us = float(np.median(v))
        res[k] = dict(us_per_call_median=round(us, 2), us_per_call_min=round(min(v), 2),
                      us_per_call_max=round(max(v), 2), us_per_round=[round(x, 2) for x in v],
                      algorithmic_gbs=round(per_pair * B / us / 1e3, 1), unique_block_gbs=round(uniq_bytes / us / 1e3, 1))
    res['speedup'] = round(res['legacy']['us_per_call_median'] / res['pipelined']['us_per_call_median'], 3)
    if args.timeline:
        res['timeline'] = {}
        for name, flags in (('pipelined', 0), ('legacy', LEGACY)):
            try:
                res['timeline'][name] = timeline(m, steps[bench.PL_WARM:bench.PL_WARM + args.timeline], flags)
            except Exception as e:              # the call timings above stand without it
                res['timeline'][name] = dict(error=repr(e))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
