"""CPU suite of the sharded streaming sampler's C ABI (tpn_stream_shard_*): the ctypes mirror of tpn_stream_shard_t
against the header, and argument validation of the entry points with null tables (nothing reaches a GPU)."""
import ctypes
import os
import subprocess

import pytest

from tpnet_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = -1


def test_stream_shard_struct_layout_matches_header(tmp_path):
    top = [f[0] for f in _lib.TpnStreamShard._fields_]
    shard = [f[0] for f in _lib.TpnShard._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tpnet_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(tpn_stream_shard_t));',
             '  printf("tables %d\\n", TPN_STREAM_PEER_TABLES);']
    lines += [f'  printf("{f} %zu\\n", offsetof(tpn_stream_shard_t, {f}));' for f in top]
    lines += [f'  printf("shard.{f} %zu\\n", offsetof(tpn_stream_shard_t, shard.{f}));' for f in shard]
    lines += ['  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'layout'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(_lib.TpnStreamShard)
    assert int(out['tables']) == len(_lib.STREAM_PEER_TABLES)
    for f in top:
        assert int(out[f]) == getattr(_lib.TpnStreamShard, f).offset, f
    base = _lib.TpnStreamShard.shard.offset
    for f in shard:
        assert int(out[f'shard.{f}']) == base + getattr(_lib.TpnShard, f).offset, f


def _shard(N=100, world=2, rank=1, C=20, max_batch=10, ext=16, routing=True):
    """A descriptor with every table pointer null; `routing` sets fake (never dereferenced) routing pointers."""
    s = _lib.TpnStreamShard()
    s.local = _lib.TpnStreamSampler(num_nodes=N, capacity=C, max_batch=max_batch)
    sh = s.shard
    sh.world, sh.rank, sh.global_nodes, sh.ext_rows = world, rank, N, ext
    sh.num_local_rows = (N - rank + world - 1) // world if world > 0 else N
    if routing:
        sh.mark, sh.counters, sh.need_nodes = 0x1000, 0x2000, 0x3000
    return s


def test_stream_shard_entry_points_validate_without_gpu():
    lib = _lib.load()
    for fn in (lib.tpn_stream_shard_reset, lib.tpn_stream_shard_pull):
        assert fn(None, None) == INVALID
    assert lib.tpn_stream_shard_push(None, None, None, None, None, 4, None, 0, None) == INVALID
    assert lib.tpn_stream_shard_query(None, None, None, None, 4, 5, None, None, None, None) == INVALID
    ok = _shard()
    ref = ctypes.byref(ok)
    # null list / pending tables
    assert lib.tpn_stream_shard_reset(ref, None) == INVALID
    assert lib.tpn_stream_shard_pull(ref, None) == INVALID
    assert lib.tpn_stream_shard_push(ref, None, None, None, None, 4, None, 0, None) == INVALID
    assert lib.tpn_stream_shard_query(ref, None, None, None, 4, 5, None, None, None, None) == INVALID
    assert lib.tpn_stream_shard_push(ref, None, None, None, None, 11, None, 0, None) == INVALID       # > max_batch
    assert lib.tpn_stream_shard_query(ref, None, None, None, 4, 21, None, None, None, None) == INVALID  # K > C
    # empty calls launch nothing
    assert lib.tpn_stream_shard_push(ref, None, None, None, None, 0, None, 0, None) == _lib.TPN_OK
    assert lib.tpn_stream_shard_query(ref, None, None, None, 0, 5, None, None, None, None) == _lib.TPN_OK
    # a shard that does not describe the placement of the sampler's nodes
    bad = [_shard(routing=False), _shard(world=0), _shard(rank=2), _shard(world=65, rank=0)]
    b = _shard()
    b.shard.global_nodes = 99                                                # != local.num_nodes
    bad.append(b)
    b = _shard()
    b.shard.num_local_rows = 51                                              # rank 1 of 2 owns 50 of 100 nodes
    bad.append(b)
    b = _shard()
    b.shard.ext_rows = -1
    bad.append(b)
    bad.append(_shard(N=1 << 31, world=2, rank=0))                          # ids must fit the int32 mark tables
    for s in bad:
        r = ctypes.byref(s)
        assert lib.tpn_stream_shard_reset(r, None) == INVALID
        assert lib.tpn_stream_shard_pull(r, None) == INVALID
        assert lib.tpn_stream_shard_push(r, None, None, None, None, 0, None, 0, None) == INVALID
        assert lib.tpn_stream_shard_query(r, None, None, None, 0, 5, None, None, None, None) == INVALID


def test_sharded_sampler_refuses_cpu_and_the_nccl_plane():
    from tpnet_b200.neighbor_sampler import ShardedStreamingSampler
    from tpnet_b200.peer import LocalPeerGroup
    with pytest.raises(RuntimeError, match='CUDA only'):
        ShardedStreamingSampler(100, 20, 'cpu')
    with pytest.raises(NotImplementedError, match="exchange='peer'"):
        ShardedStreamingSampler(100, 20, 'cuda:0', peers=LocalPeerGroup.create(2)[0], exchange='nccl')
