"""GPU suite: the encoder's structured call and get_random_projections on the sharded state (peer data plane).

All ranks of a sharded state run inside this process (LocalPeerGroup), each on its own stream, read phases before
write phases, exactly as in tests/test_gpu_sharded.py.  Every result is compared with the plain
RandomProjectionModule fed the same batches (that module is pinned to the oracle by the rest of the suite).
The real multi-process run (NVLink pulls, all_gather of the slices) is tests/dist_gpu_encoder_check.py."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'


# ---------------------------------------------------------------- in-process ranks (as in tests/test_gpu_sharded.py)
def _sim_ranks(world, kw, mode, ext_rows, accumulation='reference', chunk=1024):
    from tpnet_b200.peer import LocalPeerGroup
    from tpnet_b200.sharded import ShardedRandomProjection
    groups = LocalPeerGroup.create(world)
    ranks = []
    for r in range(world):
        torch.manual_seed(11)                      # p0='global': every rank draws the same global P_0, keeps its rows
        ranks.append(ShardedRandomProjection(decay_mode=mode, ext_rows=ext_rows, peers=groups[r], exchange='peer',
                                             state_device='cuda:0', accumulation=accumulation, giant_chunk=chunk,
                                             **kw).to('cuda:0'))
    for m in ranks:
        m._peers.publish('state', m._peer_bufs['state'])          # every buffer is published before anyone connects
        if 'stamps' in m._peer_bufs:
            m._peers.publish('stamps', m._peer_bufs['stamps'])
        m._peers.publish('flags', m._peer_bufs['flags'])
    for m in ranks:
        m.connect()
    return ranks, [torch.cuda.Stream() for _ in range(world)]


def _each(ranks, streams, fn):
    """One phase on every rank (each on its own stream), then a device-wide sync: with all ranks on one GPU the
    phases are ordered by the driver instead of tpn_peer_barrier (LocalPeerGroup.host_barriers)."""
    out = []
    for m, s in zip(ranks, streams):
        with torch.cuda.stream(s):
            out.append(fn(m))
    torch.cuda.synchronize()
    return out


def _update_all(ranks, streams, s, d, ts, next_time=None):
    pending = _each(ranks, streams, lambda m: m.update_begin(s, d, ts, next_time))      # reads: routing + pulls
    for m, st, p in zip(ranks, streams, pending):                                     # writes
        with torch.cuda.stream(st):
            m.update_end(p)
    torch.cuda.synchronize()


# ---------------------------------------------------------------- helpers of this file
def _kw(N, dim, L, not_scale):
    return dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=1e-4, device=DEV,
                use_matrix=False, beginning_time=np.float64(0.0), not_scale=not_scale, enforce_dim=dim)


def _setup(world, mode, N, dim, L, not_scale, ext_rows=None):
    from tpnet_b200 import RandomProjectionModule
    kw = _kw(N, dim, L, not_scale)
    ranks, streams = _sim_ranks(world, kw, mode, ext_rows=ext_rows if ext_rows is not None else 2 * N + 64)
    torch.manual_seed(11)
    ref = RandomProjectionModule(decay_mode=mode, **kw).to(DEV)
    for m in ranks:
        m.mlp.load_state_dict(ref.mlp.state_dict())
    return ranks, streams, ref


def _assemble(parts, m):
    """(positions, rows) of every rank -> [m, ...]; every position must be covered exactly once."""
    keep0, feat0 = parts[0]
    got = torch.zeros((m,) + tuple(feat0.shape[1:]), dtype=feat0.dtype, device=DEV)
    seen = torch.zeros(m, dtype=torch.int64, device=DEV)
    for keep, feat in parts:
        assert keep.shape[0] == feat.shape[0]
        got[keep] = feat
        seen[keep] += 1
    assert torch.all(seen == 1), seen
    return got


def _assemble_layers(parts, m, L):
    return [_assemble([(keep, layers[i]) for keep, layers in parts], m) for i in range(L + 1)]


def _encoder_batch(rng, N, m, K):
    nbr = rng.integers(1, N, (m, K)).astype(np.int64)
    nbr[rng.random((m, K)) < 0.2] = 0                  # padding neighbour id 0: an ordinary row
    return nbr, rng.integers(1, N, m).astype(np.int64), rng.integers(1, N, m).astype(np.int64)


def _check_encoder(ranks, streams, ref, nbr, src, dst):
    m = nbr.shape[0]
    parts = _each(ranks, streams, lambda r: r.neighbor_pair_wise_gram(nbr, src, dst))
    want = ref.neighbor_pair_wise_gram(nbr, src, dst)
    torch.cuda.synchronize()
    got = _assemble(parts, m)
    assert torch.equal(got, want), (got - want).abs().max().item()


def _check_rows(ranks, streams, ref, ids, L):
    parts = _each(ranks, streams, lambda r: r.get_random_projections(ids))
    want = ref.get_random_projections(ids)
    torch.cuda.synchronize()
    got = _assemble_layers(parts, len(ids), L)
    for i in range(L + 1):
        assert torch.equal(got[i], want[i]), i


# ---------------------------------------------------------------- parity
@pytest.mark.parametrize('L,not_scale', [(2, True), (3, False)], ids=['L2-not_scale', 'L3-scale'])
@pytest.mark.parametrize('mode', ['eager', 'lazy'])
@pytest.mark.parametrize('world', [2, 4])
def test_encoder_and_rows_equal_single_gpu(world, mode, L, not_scale):
    """Routed encoder calls, routed decoder pairs and routed updates interleaved over several batches, then
    backup -> update -> reload: the encoder features and the gathered rows are bit-equal to the plain module's.
    K = 20 and 7, padding id 0, m not divisible by world, and m < world (ranks with an empty slice)."""
    N, dim = 997, (36 if L == 2 else 140)
    ranks, streams, ref = _setup(world, mode, N, dim, L, not_scale)
    rng = np.random.default_rng(world * 10 + L)
    t = 0.0
    for B in (300, 4000, 1500):
        s = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
        d = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
        ts = np.sort(t + rng.random(B) * 500.0)
        t = ts[-1]
        for m, K in ((2 * 101 + 1, 20), (57, 7), (world - 1, 20)):
            _check_encoder(ranks, streams, ref, *_encoder_batch(rng, N, m, K))
        a = rng.integers(0, N, 501).astype(np.int64)
        b = rng.integers(0, N, 501).astype(np.int64)
        routed = _each(ranks, streams, lambda r: r.routed_pair_wise_gram(a, b))      # decoder pairs, same generation
        want = ref.pair_wise_gram(a, b)
        got = torch.zeros_like(want)
        for r in routed:
            keep, feat = r.trimmed()
            got[keep] = feat
        assert torch.allclose(got, want, rtol=1e-5, atol=2e-5)
        _check_rows(ranks, streams, ref, rng.integers(0, N, 301).astype(np.int64), L)
        _update_all(ranks, streams, s, d, ts)
        ref.update(s, d, ts)
    # backup -> update -> reload: every write starts a new generation of the remote-row caches
    saved = _each(ranks, streams, lambda m: m.backup_random_projections())
    saved_ref = ref.backup_random_projections()
    s = rng.integers(1, N, 500).astype(np.int64)
    d = rng.integers(1, N, 500).astype(np.int64)
    ts = np.sort(t + rng.random(500) * 100.0)
    _update_all(ranks, streams, s, d, ts)
    ref.update(s, d, ts)
    _check_encoder(ranks, streams, ref, *_encoder_batch(rng, N, 64, 20))
    for m, sv, st in zip(ranks, saved, streams):
        with torch.cuda.stream(st):
            m.reload_random_projections(sv)
    torch.cuda.synchronize()
    ref.reload_random_projections(saved_ref)
    _check_encoder(ranks, streams, ref, *_encoder_batch(rng, N, 203, 20))
    _check_rows(ranks, streams, ref, np.arange(N, dtype=np.int64), L)
    for m in ranks:
        m.check_errors()


# ---------------------------------------------------------------- head, device-resident ids
@pytest.mark.parametrize('L', [3, 2], ids=['F64-tensor-core-head', 'F36-cublas-head'])
def test_encoder_features_with_head(L):
    """get_neighbor_pair_wise_feature: the head acts on each block alone, so the fused tensor-core head (F = 64)
    gives the same bits on a rank's slice as on the whole call; the cuBLAS head (F = 36) may pick another algorithm
    for another row count.  CUDA-tensor ids give the same result as numpy ids."""
    N, world = 997, 2
    ranks, streams, ref = _setup(world, 'lazy', N, 140 if L == 3 else 36, L, False)
    rng = np.random.default_rng(5)
    s = rng.integers(1, N, 3000).astype(np.int64)
    d = rng.integers(1, N, 3000).astype(np.int64)
    ts = np.sort(rng.random(3000) * 100.0)
    _update_all(ranks, streams, s, d, ts)
    ref.update(s, d, ts)
    nbr, src, dst = _encoder_batch(rng, N, 401, 20)
    with torch.no_grad():
        parts = _each(ranks, streams, lambda r: r.get_neighbor_pair_wise_feature(nbr, src, dst))
        g = lambda a: torch.from_numpy(a).to(DEV)       # noqa: E731
        parts_dev = _each(ranks, streams, lambda r: r.get_neighbor_pair_wise_feature(g(nbr), g(src), g(dst)))
        want = ref.get_neighbor_pair_wise_feature(nbr, src, dst)
    torch.cuda.synchronize()
    got = _assemble(parts, 401)
    got_dev = _assemble(parts_dev, 401)
    assert got.shape == want.shape == (401, 20, 2 * ref.pair_wise_feature_dim)
    assert torch.equal(got_dev, got)
    if L == 3:
        assert torch.equal(got, want), (got - want).abs().max().item()
    else:
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-6), (got - want).abs().max().item()
    ids = rng.integers(0, N, 257).astype(np.int64)
    rows_np = _each(ranks, streams, lambda r: r.get_random_projections(ids))
    rows_dev = _each(ranks, streams, lambda r: r.get_random_projections(g(ids)))
    for a, b in zip(_assemble_layers(rows_np, 257, L), _assemble_layers(rows_dev, 257, L)):
        assert torch.equal(a, b)
    for m in ranks:
        m.check_errors()


def test_single_rank_takes_the_plain_kernels():
    """World 1: the plain kernels on the whole call, ids checked against the GLOBAL node count (not the row count of
    the buffer, which includes the extension rows)."""
    from tpnet_b200 import RandomProjectionModule
    from tpnet_b200.sharded import ShardedRandomProjection
    N, L = 301, 3
    kw = _kw(N, 64, L, False)
    torch.manual_seed(3)
    sh = ShardedRandomProjection(decay_mode='lazy', ext_rows=64, **kw).to(DEV)
    torch.manual_seed(3)
    ref = RandomProjectionModule(decay_mode='lazy', **kw).to(DEV)
    rng = np.random.default_rng(2)
    s = rng.integers(1, N, 2000).astype(np.int64)
    d = rng.integers(1, N, 2000).astype(np.int64)
    ts = np.sort(rng.random(2000) * 100.0)
    sh.update(s, d, ts)
    ref.update(s, d, ts)
    nbr, src, dst = _encoder_batch(rng, N, 33, 20)
    keep, feat = sh.neighbor_pair_wise_gram(nbr, src, dst)
    assert torch.equal(keep.cpu(), torch.arange(33)) and torch.equal(feat, ref.neighbor_pair_wise_gram(nbr, src, dst))
    with torch.no_grad():
        keep, feat = sh.get_neighbor_pair_wise_feature(nbr, src, dst)
        assert torch.equal(feat, ref.get_neighbor_pair_wise_feature(nbr, src, dst))
        assert torch.equal(sh.get_neighbor_pair_wise_feature(nbr, src, dst, gather=True), feat)
    ids = rng.integers(0, N, 100).astype(np.int64)
    for a, b in zip(sh.get_random_projections(ids), ref.get_random_projections(ids)):       # the reference's list
        assert torch.equal(a, b)
    # ids in [N, N + ext_rows) are rows of the buffer but not nodes of the graph
    with pytest.raises(IndexError):
        sh.get_random_projections(np.array([1, N + 3], dtype=np.int64))
    bad = nbr.copy()
    bad[5, 2] = N
    with pytest.raises(IndexError):
        sh.neighbor_pair_wise_gram(bad, src, dst)
    sh.check_errors()


# ---------------------------------------------------------------- errors
def test_errors_of_the_routed_calls():
    N, world, L = 301, 2, 3
    ranks, streams, _ = _setup(world, 'lazy', N, 64, L, False)
    rng = np.random.default_rng(7)
    nbr, src, dst = _encoder_batch(rng, N, 40, 7)
    # host ids: validated against the global node count before anything is launched, on the rank whose slice holds
    # the id (rows [0, 20) are rank 0's)
    bad = nbr.copy()
    bad[3, 1] = N + 1
    with pytest.raises(IndexError):
        ranks[0].neighbor_pair_wise_gram(bad, src, dst)
    with pytest.raises(IndexError):
        ranks[0].get_random_projections(np.array([N, 2], dtype=np.int64))
    # device-resident ids: flagged by the routing kernel, raised by check_errors
    dbad = torch.from_numpy(bad).to(DEV)
    _each(ranks, streams, lambda r: r.neighbor_pair_wise_gram(dbad, torch.from_numpy(src).to(DEV),
                                                              torch.from_numpy(dst).to(DEV)))
    with pytest.raises(IndexError):
        ranks[0].check_errors()
    ranks[1].check_errors()                               # its slice was clean
    # extension rows too small for one call
    small, sstreams, _ = _setup(world, 'lazy', N, 64, L, False, ext_rows=8)
    _each(small, sstreams, lambda r: r.neighbor_pair_wise_gram(nbr, src, dst))
    with pytest.raises(RuntimeError, match='extension rows'):
        small[0].check_errors()


def test_nccl_data_plane_refuses_the_node_calls():
    from tpnet_b200.peer import LocalPeerGroup
    from tpnet_b200.sharded import ShardedRandomProjection
    groups = LocalPeerGroup.create(2)
    m = ShardedRandomProjection(decay_mode='eager', ext_rows=16, peers=groups[0], exchange='nccl', **_kw(101, 16, 2, False))
    m = m.to(DEV)
    ids = np.arange(4, dtype=np.int64)
    for call in (lambda: m.neighbor_pair_wise_gram(ids.reshape(2, 2), ids[:2], ids[:2]),
                 lambda: m.get_neighbor_pair_wise_feature(ids.reshape(2, 2), ids[:2], ids[:2]),
                 lambda: m.get_random_projections(ids)):
        with pytest.raises(NotImplementedError, match="exchange='peer'"):
            call()


# ---------------------------------------------------------------- the routing kernel itself
def test_route_nodes_kernel_invariants():
    """tpn_route_nodes, one rank's view (no peers needed): owned ids -> id // world; every remote id -> a slot s
    with need_nodes[s] == id, shared by repeated ids; a second call in the same generation reuses the slots and hands
    out only new ones ([PREV, NEED) is exactly the new ones); an id outside the graph is flagged and maps to row 0."""
    from tpnet_b200 import _lib
    from tpnet_b200.sharded import rows_on_rank
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    N, world, rank = 5003, 3, 1
    n_local = rows_on_rank(N, world, rank)
    ext = 4096
    mark = torch.zeros(N, dtype=torch.int32, device=DEV)
    ctr = torch.zeros(8, dtype=torch.int32, device=DEV)
    need = torch.zeros(ext, dtype=torch.int64, device=DEV)
    sh = _lib.TpnShard()
    sh.world, sh.rank, sh.global_nodes, sh.num_local_rows, sh.ext_rows = world, rank, N, n_local, ext
    sh.mark, sh.counters, sh.need_nodes = mark.data_ptr(), ctr.data_ptr(), need.data_ptr()
    rng = np.random.default_rng(0)

    def route(ids):
        d = torch.from_numpy(ids).to(DEV)
        rows = torch.full((len(ids),), -7, dtype=torch.int64, device=DEV)
        assert lib.tpn_route_nodes(ctypes.byref(sh), d.data_ptr(), len(ids), rows.data_ptr(), stream) == 0
        torch.cuda.synchronize()
        return rows.cpu().numpy()

    def check(ids, rows):
        own = ids % world == rank
        assert np.array_equal(rows[own], ids[own] // world)
        slots = rows[~own] - n_local
        assert np.all((slots >= 0) & (slots < int(ctr[0].item())))
        nodes = need.cpu().numpy()
        assert np.array_equal(nodes[slots], ids[~own])
        for u in np.unique(ids[~own]):                      # repeated ids share one slot
            assert len(np.unique(rows[ids == u])) == 1

    ids1 = (1 + (rng.zipf(1.3, 3000) - 1) % (N - 1)).astype(np.int64)      # many repeats (power law)
    rows1 = route(ids1)
    check(ids1, rows1)
    remote1 = np.unique(ids1[ids1 % world != rank])
    assert int(ctr[0].item()) == len(remote1) and int(ctr[1].item()) == 0 and int(ctr[2].item()) == 0
    ids2 = np.concatenate([ids1[:500], rng.integers(0, N, 2000)]).astype(np.int64)
    rows2 = route(ids2)
    check(ids2, rows2)
    assert np.array_equal(rows2[:500], rows1[:500])                          # reused in the same generation
    new = np.setdiff1d(np.unique(ids2[ids2 % world != rank]), remote1)
    assert int(ctr[1].item()) == len(remote1) and int(ctr[0].item()) == len(remote1) + len(new)
    assert set(need[len(remote1):int(ctr[0].item())].cpu().numpy().tolist()) == set(new.tolist())
    # an empty list: nothing new to pull
    assert lib.tpn_route_nodes(ctypes.byref(sh), None, 0, None, stream) == 0
    torch.cuda.synchronize()
    assert int(ctr[1].item()) == int(ctr[0].item())
    rows3 = route(np.array([4, N, -1, 7], dtype=np.int64))
    assert rows3[1] == 0 and rows3[2] == 0 and int(ctr[2].item()) == 1


# ---------------------------------------------------------------- wide rows
def test_wide_rows_take_the_pairwise_fallback():
    """Node blocks too wide for the shared-memory staging of tpn_pairwise_neighbors: the translated rows go through
    tpn_pairwise on the expanded lists (no second routing).  Both sides stay under 4096 pairs, so both launch the
    same pair kernel and the features are bit-equal."""
    N, world, L = 64, 2, 3
    ranks, streams, ref = _setup(world, 'eager', N, 6400, L, False)
    rng = np.random.default_rng(9)
    s = rng.integers(1, N, 200).astype(np.int64)
    d = rng.integers(1, N, 200).astype(np.int64)
    ts = np.sort(rng.random(200) * 10.0)
    _update_all(ranks, streams, s, d, ts)
    ref.update(s, d, ts)
    nbr, src, dst = _encoder_batch(rng, N, 31, 7)
    before = [m.launches for m in ranks]
    _check_encoder(ranks, streams, ref, nbr, src, dst)
    assert [m.launches - b for m, b in zip(ranks, before)] == [2, 2]                 # the two tpn_pairwise calls
    for m in ranks:
        m.check_errors()


# ---------------------------------------------------------------- real ranks
def test_encoder_calls_real_ranks():
    """One process per GPU (torchrun), NVLink pulls, gather=True on every rank: tests/dist_gpu_encoder_check.py."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29541', os.path.join(ROOT, 'tests', 'dist_gpu_encoder_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'PASS' in r.stdout
