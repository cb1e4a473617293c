"""Time and host memory of save_sampler / load_sampler (tpnet_b200/checkpoint.py) at the power-law shape.

    python scripts/sampler_checkpoint_probe.py --out DIR [--batches 4] [--chunk-mib 64,256] [--tmp TMPDIR]

A StreamingRecentSampler over synth.SHAPES['powerlaw'] (N = 10,000,001, C = 20: 9.76 GB of tables) is fed --batches
batches of 100,000 edges and queried; then, per chunk size, it is saved to a fresh directory under --tmp and loaded
into a second sampler, whose answers to the last batch's queries must be bit-equal to the first one's.  One JSON file,
DIR/sampler_checkpoint_probe.json, with the device name and power limit read in the same run.

Times are host wall clock around each call, which ends with its last device copy done and its last write returned.
The save writes to the page cache (no fsync) and the load then reads the same files back, most likely from that
cache: these are the rates of the format's copies and of the host's file cache, not of a disk.  Peak host memory is
the largest resident set sampled every 2 ms during the call, minus the resident set before it.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import checkpoint as ck, synth  # noqa: E402
from tpnet_b200.neighbor_sampler import StreamingRecentSampler  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, 'scripts'))
from sharded_sampler_probe import B, K, device_info, stream  # noqa: E402


def rss_bytes() -> int:
    with open('/proc/self/statm') as fh:
        return int(fh.read().split()[1]) * os.sysconf('SC_PAGE_SIZE')


def measured(fn):
    """(seconds, peak resident bytes above the start, result) of fn()."""
    base, peak, done = rss_bytes(), [0], threading.Event()

    def sample():
        while not done.is_set():
            peak[0] = max(peak[0], rss_bytes())
            time.sleep(0.002)

    th = threading.Thread(target=sample)
    th.start()
    t0 = time.perf_counter()
    try:
        r = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        done.set()
        th.join()
    return dt, max(peak[0], rss_bytes()) - base, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--batches', type=int, default=4)
    ap.add_argument('--chunk-mib', default='64,256')
    ap.add_argument('--tmp', default=None, help='directory for the checkpoint files (default: the system temp dir)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('sampler_checkpoint_probe measures on a CUDA device; none found')
    dev = torch.device('cuda', torch.cuda.current_device())
    N = synth.SHAPES['powerlaw'].node_num
    a = StreamingRecentSampler(N, K, dev, max_batch=B)
    for d, qn, qt in stream(args.batches, dev):
        a.push(*d)
        want = a.get_historical_neighbors(qn, qt, K, as_tensors=True)
    a.check_errors()
    b = StreamingRecentSampler(N, K, dev, max_batch=B)
    table_bytes = N * ck.sampler_row_bytes(K)
    res = {'device_info': device_info(dev), 'num_nodes': N, 'capacity': K, 'batch': B, 'batches_pushed': args.batches,
           'table_bytes': table_bytes, 'runs': []}
    for mib in (int(x) for x in args.chunk_mib.split(',')):
        d = tempfile.mkdtemp(prefix='sampler_ckpt_', dir=args.tmp)
        try:
            ts, hs, path = measured(lambda: ck.save_sampler(a, d, chunk_bytes=mib << 20))
            files = os.path.getsize(path) + os.path.getsize(ck.lists_path(path))
            tl, hl, _ = measured(lambda: ck.load_sampler(b, d, chunk_bytes=mib << 20))
            got = b.get_historical_neighbors(qn, qt, K, as_tensors=True)
            same = all(torch.equal(x, y) for x, y in zip(got, want))
        finally:
            shutil.rmtree(d, ignore_errors=True)
        run = {'chunk_bytes': mib << 20, 'file_bytes': files, 'save_s': ts, 'save_GBps': files / ts / 1e9,
               'save_peak_host_bytes_above_start': hs, 'load_s': tl, 'load_GBps': files / tl / 1e9,
               'load_peak_host_bytes_above_start': hl, 'answers_bit_equal_after_load': bool(same)}
        res['runs'].append(run)
        print(json.dumps(run), flush=True)
    b.check_errors()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'sampler_checkpoint_probe.json'), 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
