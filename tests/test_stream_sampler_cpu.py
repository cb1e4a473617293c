"""CPU suite of the streaming `recent` sampler (tpn_stream_sampler_*, StreamingRecentSampler).

`TwoListModel` is the rule the kernels implement, in numpy: per node ALL (last C folded entries) and OLD (last C
folded entries strictly older than the node's newest folded time), plus the latest batch pending.  It is pinned here
against RecentNeighborOracle over the pushed prefix, on zipf streams with ragged batches and timestamps quantised so
that equal times cross batch boundaries all the time."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.neighbor_sampler import RecentNeighborOracle
from tpnet_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class TwoListModel:
    def __init__(self, num_nodes: int, capacity: int):
        self.C = capacity
        self.all = [[] for _ in range(num_nodes)]        # entries (nbr, eid, t), oldest first
        self.old = [[] for _ in range(num_nodes)]
        self.newest = np.full(num_nodes, -np.inf)
        self.pending = {}                                 # node -> its entries of the latest batch, in sorted order

    def push(self, src, dst, eid, t):
        for u, seg in self.pending.items():              # fold: only the last 2C entries of a segment are read
            tnew = seg[-1][2]
            if tnew > self.newest[u]:
                older = [e for e in seg if e[2] < tnew]
                self.old[u] = (self.all[u] + older[-self.C:])[-self.C:]
                self.newest[u] = tnew
            self.all[u] = (self.all[u] + seg[-self.C:])[-self.C:]
        self.pending = {}
        for j in range(len(src)):                         # stable sort by node of (src: dst), (dst: src)
            for owner, other in ((src[j], dst[j]), (dst[j], src[j])):
                self.pending.setdefault(int(owner), []).append((int(other), int(eid[j]), float(t[j])))

    def query(self, nodes, times, K):
        out = np.zeros((len(nodes), K, 3))
        for q, (u, tq) in enumerate(zip(nodes, times)):
            if tq > self.newest[u]:
                lst = self.all[u] + [e for e in self.pending.get(int(u), []) if e[2] < tq]
            elif tq == self.newest[u]:
                lst = self.old[u]
            else:
                raise AssertionError('query before the node\'s newest folded time')
            lst = lst[-K:]
            if lst:
                out[q, K - len(lst):] = np.array(lst, dtype=np.float64)
        return out[..., 0].astype(np.int64), out[..., 1].astype(np.int64), out[..., 2]


@pytest.mark.parametrize('seed', range(30))
def test_two_list_model_matches_oracle_on_tied_ragged_streams(seed):
    rng = np.random.default_rng(seed)
    N = int(rng.integers(5, 60))
    C = int(rng.integers(1, 8))
    E = int(rng.integers(200, 900))
    src = (rng.zipf(1.4, E) - 1) % N
    dst = (rng.zipf(1.4, E) - 1) % N
    loops = rng.random(E) < 0.03                           # self-loops: both directions land in one list
    dst[loops] = src[loops]
    t = np.sort(np.floor(rng.random(E) * 60.0))           # 60 distinct values: ties across batch boundaries
    eid = np.arange(1, E + 1)
    model = TwoListModel(N, C)
    lo = 0
    while lo < E:
        hi = min(E, lo + int(rng.integers(1, 301)))
        model.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        bt = t[lo:hi]
        rnd = rng.integers(0, N, 40)
        qn = np.concatenate([src[lo:hi], dst[lo:hi], rnd])
        qt = np.concatenate([bt, bt, np.full(40, bt[-1]) + rng.integers(0, 3, 40)])
        # only queries the contract covers: time >= the node's newest time before this push
        ok = qt >= model.newest[qn]
        for K in sorted({1, C}):
            got = model.query(qn[ok], qt[ok], K)
            ref = o.get_historical_neighbors(qn[ok], qt[ok], K)
            for g, r in zip(got, ref):
                assert np.array_equal(g, r), (seed, lo, K)
        lo = hi


def test_stream_struct_layout_matches_header(tmp_path):
    fields = [f[0] for f in _lib.TpnStreamSampler._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tpnet_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(tpn_stream_sampler_t));']
    lines += [f'  printf("{f} %zu\\n", offsetof(tpn_stream_sampler_t, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'layout'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(_lib.TpnStreamSampler)
    for f in fields:
        assert int(out[f]) == getattr(_lib.TpnStreamSampler, f).offset, f


def test_stream_entry_points_validate_without_gpu():
    lib = _lib.load()
    INVALID = -1
    s = _lib.TpnStreamSampler(num_nodes=100, capacity=20, max_batch=10)       # every table pointer is null
    ref = ctypes.byref(s)
    assert lib.tpn_stream_sampler_push(None, None, None, None, None, 4, None, 0, None) == INVALID
    assert lib.tpn_stream_sampler_query(None, None, None, 4, 5, None, None, None, None) == INVALID
    assert lib.tpn_stream_sampler_reset(None, None) == INVALID
    assert lib.tpn_stream_sampler_reset(ref, None) == INVALID                   # null tables
    assert lib.tpn_stream_sampler_push(ref, None, None, None, None, 4, None, 0, None) == INVALID
    assert lib.tpn_stream_sampler_query(ref, None, None, 4, 5, None, None, None, None) == INVALID
    assert lib.tpn_stream_sampler_push(ref, None, None, None, None, 11, None, 0, None) == INVALID   # > max_batch
    assert lib.tpn_stream_sampler_query(ref, None, None, 4, 21, None, None, None, None) == INVALID  # K > C
    assert lib.tpn_stream_sampler_query(ref, None, None, 4, 0, None, None, None, None) == INVALID
    assert lib.tpn_stream_sampler_push(ref, None, None, None, None, 0, None, 0, None) == _lib.TPN_OK
    assert lib.tpn_stream_sampler_query(ref, None, None, 0, 5, None, None, None, None) == _lib.TPN_OK
    bad = _lib.TpnStreamSampler(num_nodes=100, capacity=0, max_batch=10)      # C < 1
    assert lib.tpn_stream_sampler_query(ctypes.byref(bad), None, None, 0, 1, None, None, None, None) == INVALID
    assert lib.tpn_stream_sampler_push(ctypes.byref(bad), None, None, None, None, 0, None, 0, None) == INVALID
    assert lib.tpn_stream_sampler_reset(ctypes.byref(bad), None) == INVALID
    ws = lib.tpn_stream_sampler_workspace_bytes
    assert 0 < ws(1) < ws(100_000) and ws(100_000) >= 4 * 4 * 200_000


def test_streaming_sampler_refuses_cpu():
    from tpnet_b200.neighbor_sampler import StreamingRecentSampler
    with pytest.raises(RuntimeError, match='CUDA only'):
        StreamingRecentSampler(100, 20, 'cpu')
