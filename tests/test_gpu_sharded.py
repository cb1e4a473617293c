"""GPU suite: the sharded path on >= 2 GPUs (skipped on a single-GPU box)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_single_rank_equals_plain_module():
    """world_size 1 (no process group): the message-mode update + extension-row plumbing must
    reproduce the plain module bit for bit."""
    import numpy as np
    from tpnet_b200 import RandomProjectionModule
    from tpnet_b200.sharded import ShardedRandomProjection
    dev = 'cuda:0'
    for mode in ('eager', 'lazy'):
        kw = dict(node_num=301, edge_num=3000, dim_factor=1, num_layer=3, time_decay_weight=1e-4, device=dev,
                  use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=28)
        torch.manual_seed(3)
        sh = ShardedRandomProjection(decay_mode=mode, ext_rows=64, **kw).to(dev)
        torch.manual_seed(3)
        ref = RandomProjectionModule(decay_mode=mode, **kw).to(dev)
        rng = np.random.default_rng(1)
        t = 0.0
        for B in (200, 3000, 40000):
            s = rng.integers(1, 301, B).astype(np.int64)
            d = rng.integers(1, 301, B).astype(np.int64)
            ts = np.sort(t + rng.random(B) * 100.0)
            t = ts[-1]
            sh.update(s, d, ts, plan=sh.plan_update(s, d, ts))      # explicit plan: the message-mode path
            ref.update(s, d, ts)
        sh.materialize(); ref.materialize()
        for i in range(4):
            assert torch.equal(sh.random_projections[i].data[:301], ref.random_projections[i].data), (mode, i)
        a = rng.integers(0, 301, 500).astype(np.int64)
        b = rng.integers(0, 301, 500).astype(np.int64)
        keep, feat = sh.pair_wise_gram(a, b, plan=sh.plan_pairs(a, b))
        assert len(keep) == 500 and torch.equal(feat, ref.pair_wise_gram(a, b))
        keep, feat = sh.pair_wise_gram(a, b)                        # world 1 without a plan: the plain path
        assert len(keep) == 500 and torch.equal(feat, ref.pair_wise_gram(a, b))


@pytest.mark.parametrize('world', [2, 4, 8])
def test_sharded_equals_single_gpu_real_ranks(world):
    """One process per GPU (torchrun), real NVLink pulls and NCCL all_to_all: tests/dist_gpu_check.py."""
    if torch.cuda.device_count() < world:
        pytest.skip(f'needs >= {world} GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world),
           '--master-addr', '127.0.0.1', '--master-port', str(29517 + world), os.path.join(ROOT, 'tests', 'dist_gpu_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'PASS' in r.stdout


# ----------------------------------------------------------------------------------------------------------------
# The routed ("peer") data plane with all ranks inside this process (LocalPeerGroup): device-side routing, pulls
# through peer pointers, flag barriers, device-side counts.  Every rank launches on its own stream, exactly the
# launches a one-process-per-GPU job issues; only the NVLink transport itself needs several GPUs
# (tests/dist_gpu_check.py, bench.py --gpus N `parity`).
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


def _global_layers(ranks, N, L, streams):
    _each(ranks, streams, lambda m: m.materialize())
    torch.cuda.synchronize()
    world = len(ranks)
    full = []
    for i in range(L + 1):
        g = torch.zeros(N, ranks[0].dim, device='cuda:0')
        for r, m in enumerate(ranks):
            g[r::world] = m.random_projections[i].data[:m.n_local]
        full.append(g)
    return full


@pytest.mark.parametrize('world,flags', [(2, 0), (4, 0), (2, 64)], ids=['world2', 'world4', 'world2-stream-all'])
@pytest.mark.parametrize('mode', ['eager', 'lazy'])
def test_peer_data_plane_equals_single_gpu(world, mode, flags):
    """'stream-all' (TPN_DEBUG_STREAM_ALL): every giant segment of the routed message-mode updates takes the streamed
    path of the hub walker (received rows with their own stamps included).
    Sharded over `world` ranks == the plain module, BIT FOR BIT (eager and lazy: a cached remote row carries
    its owner's stamps, so it is read with the same single multiply as on one GPU), through batches that take the
    single-CTA sort, the radix sort, the short-segment walker and the hub walkers; pair-wise features of the
    routed call; reset / backup / reload; error flags."""
    import numpy as np
    from tpnet_b200 import RandomProjectionModule, _lib
    dev = 'cuda:0'
    old_flags = _lib.load().tpn_set_debug_flags(flags)
    try:
        _peer_data_plane_case(world, mode, dev, np, RandomProjectionModule)
    finally:
        _lib.load().tpn_set_debug_flags(old_flags)


def _peer_data_plane_case(world, mode, dev, np, RandomProjectionModule):
    for (N, dim, L, sizes) in [(403, 20, 3, (200, 3000)), (2003, 140, 3, (9000, 200, 25000)), (997, 36, 2, (40000,))]:
        kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=1e-4, device=dev,
                  use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=dim)
        ranks, streams = _sim_ranks(world, kw, mode, ext_rows=2 * N + 64)
        torch.manual_seed(11)
        ref = RandomProjectionModule(decay_mode=mode, **kw).to(dev)
        rng = np.random.default_rng(N + world)
        t = 0.0
        for rnd in range(2):
            for B in sizes:
                s = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
                d = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
                ts = np.sort(t + rng.random(B) * 500.0)
                t = ts[-1]
                n = 3001 if rnd == 0 else 5000
                a = rng.integers(0, N, n).astype(np.int64)
                b = rng.integers(0, N, n).astype(np.int64)
                routed = _each(ranks, streams, lambda m: m.routed_pair_wise_gram(a, b))      # reads ...
                _update_all(ranks, streams, s, d, ts)                                         # ... then the write
                want = ref.pair_wise_gram(a, b)
                ref.update(s, d, ts)
                torch.cuda.synchronize()
                got = torch.zeros_like(want)
                seen = torch.zeros(n, dtype=torch.int64, device=dev)
                for m, r in zip(ranks, routed):
                    keep, feat = r.trimmed()
                    assert torch.all(torch.from_numpy(a).to(dev)[keep] % world == m.rank)
                    assert torch.all(keep[1:] > keep[:-1])                                   # batch order kept
                    got[keep] = feat
                    seen[keep] += 1
                assert torch.all(seen == 1)                                                   # every pair has one owner
                assert torch.allclose(got, want, rtol=1e-5, atol=2e-5)
        full = _global_layers(ranks, N, L, streams)
        ref.materialize()
        for i in range(L + 1):
            assert torch.equal(full[i], ref.random_projections[i].data), (world, mode, N, i)
        # backup -> more updates -> reload: the caches of remote rows are invalidated on every write
        saved = _each(ranks, streams, lambda m: m.backup_random_projections())
        saved_ref = ref.backup_random_projections()
        s = rng.integers(1, N, 500).astype(np.int64); d = rng.integers(1, N, 500).astype(np.int64)
        ts = np.sort(t + rng.random(500) * 100.0)
        _update_all(ranks, streams, s, d, ts); ref.update(s, d, ts)
        for m, sv, st in zip(ranks, saved, streams):
            with torch.cuda.stream(st):
                m.reload_random_projections(sv)
        torch.cuda.synchronize()
        ref.reload_random_projections(saved_ref)
        _update_all(ranks, streams, s, d, ts); ref.update(s, d, ts)
        full = _global_layers(ranks, N, L, streams)
        ref.materialize()
        for i in range(L + 1):
            assert torch.equal(full[i], ref.random_projections[i].data), ('after reload', world, mode, N, i)
        for m in ranks:
            m.check_errors()
            assert m.barriers > 0


def test_peer_barrier_kernel_single_rank():
    """tpn_peer_barrier itself (world 1: the rank signals and waits for its own flag word): the sequence number
    advances, nothing hangs, no error.  Several ranks need one GPU each: tests/dist_gpu_check.py."""
    import ctypes
    from tpnet_b200 import _lib
    from tpnet_b200.peer import PeerBuffer
    lib = _lib.load()
    dev = torch.device('cuda:0')
    flags = PeerBuffer(64, dev)
    table = torch.tensor([flags.ptr], dtype=torch.int64, device=dev)
    mark = torch.zeros(8, dtype=torch.int32, device=dev)
    ctr = torch.zeros(8, dtype=torch.int32, device=dev)
    need = torch.zeros(8, dtype=torch.int64, device=dev)
    seq = torch.zeros(1, dtype=torch.int32, device=dev)
    sh = _lib.TpnShard()
    sh.world, sh.rank, sh.global_nodes, sh.num_local_rows, sh.ext_rows = 1, 0, 8, 8, 0
    sh.mark, sh.counters, sh.need_nodes = mark.data_ptr(), ctr.data_ptr(), need.data_ptr()
    sh.peer_flags, sh.barrier_seq = table.data_ptr(), seq.data_ptr()
    for k in range(1, 4):
        assert lib.tpn_peer_barrier(ctypes.byref(sh), torch.cuda.current_stream().cuda_stream) == 0
        torch.cuda.synchronize()
        assert int(seq.item()) == k and int(flags.tensor((1,), torch.int32).item()) == k and int(ctr[2].item()) == 0


def test_peer_data_plane_chunked_accumulation_and_errors():
    """accumulation='chunked' on the sharded state: the chunk boundaries are positions in the target's own message
    list, which is the same list on the owner rank, so sharded == single GPU bit for bit.  Then the error paths:
    an id outside the graph in a device-resident batch, and extension rows too small for one generation."""
    import numpy as np
    from tpnet_b200 import RandomProjectionModule
    dev = 'cuda:0'
    N, dim, L, world = 301, 64, 3, 2
    kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=1e-5, device=dev,
              use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=dim)
    ranks, streams = _sim_ranks(world, kw, 'lazy', ext_rows=2 * N, accumulation='chunked', chunk=512)
    torch.manual_seed(11)
    ref = RandomProjectionModule(decay_mode='lazy', accumulation='chunked', giant_chunk=512, **kw).to(dev)
    rng = np.random.default_rng(3)
    t = 0.0
    for B in (9000, 12000):
        s = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
        d = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
        assert np.bincount(np.concatenate([s, d])).max() >= 2048
        ts = np.sort(t + rng.random(B) * 500.0)
        t = ts[-1]
        _update_all(ranks, streams, s, d, ts); ref.update(s, d, ts)
    full = _global_layers(ranks, N, L, streams)
    ref.materialize()
    for i in range(L + 1):
        assert torch.equal(full[i], ref.random_projections[i].data), i
    # id outside the graph, device-resident: dropped + flagged on every rank
    bad = torch.tensor([5, N + 7, 9], dtype=torch.int64, device=dev)
    ok = torch.tensor([6, 8, 10], dtype=torch.int64, device=dev)
    tt = torch.full((3,), t + 1.0, dtype=torch.float64, device=dev)
    _update_all(ranks, streams, bad, ok, tt, next_time=t + 1.0)
    for m in ranks:
        with pytest.raises(IndexError):
            m.check_errors()
    # host ids are validated before anything is launched
    with pytest.raises(IndexError):
        ranks[0].update(np.array([N + 1]), np.array([3]), np.array([t + 2.0]))
    # extension rows exhausted
    small, sstreams = _sim_ranks(world, kw, 'lazy', ext_rows=4)
    a = np.arange(0, 200, dtype=np.int64); b = np.arange(1, 201, dtype=np.int64)
    _each(small, sstreams, lambda m: m.routed_pair_wise_gram(a, b))
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match='extension rows'):
        small[0].check_errors()


def test_routing_kernels_match_the_numpy_plan():
    """tpn_route_update / tpn_route_pairs (one rank's view, no peers needed) against make_plan: kept items and their
    order, local rows, and one cache slot per distinct remote node."""
    import ctypes
    import numpy as np
    from tpnet_b200 import _lib
    from tpnet_b200.sharded import make_plan, rows_on_rank, update_messages
    lib = _lib.load()
    dev = 'cuda:0'
    rng = np.random.default_rng(0)
    N = 5003
    stream_ptr = torch.cuda.current_stream().cuda_stream
    for world in (2, 3, 8):
        for rank in (0, world - 1):
            n_local = rows_on_rank(N, world, rank)
            for B in (1, 200, 2049, 30000):
                src = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
                dst = rng.integers(0, N, B).astype(np.int64)
                t = np.sort(rng.random(B))
                ext = 2 * B + 8
                mark = torch.zeros(N, dtype=torch.int32, device=dev)
                ctr = torch.zeros(8, dtype=torch.int32, device=dev)
                need = torch.zeros(ext, dtype=torch.int64, device=dev)
                sh = _lib.TpnShard()
                sh.world, sh.rank, sh.global_nodes, sh.num_local_rows, sh.ext_rows = world, rank, N, n_local, ext
                sh.mark, sh.counters, sh.need_nodes = mark.data_ptr(), ctr.data_ptr(), need.data_ptr()
                d = lambda x: torch.from_numpy(x).to(dev)      # noqa: E731
                ds, dd, dt = d(src), d(dst), d(t)
                first = torch.empty(2 * B, dtype=torch.int64, device=dev)
                second = torch.empty(2 * B, dtype=torch.int64, device=dev)
                tout = torch.empty(2 * B, dtype=torch.float64, device=dev)
                cnt = torch.zeros(1, dtype=torch.int32, device=dev)
                ws = torch.empty(lib.tpn_route_workspace_bytes(2 * B), dtype=torch.uint8, device=dev)
                assert lib.tpn_route_update(ctypes.byref(sh), ds.data_ptr(), dd.data_ptr(), dt.data_ptr(), B,
                                            first.data_ptr(), second.data_ptr(), tout.data_ptr(), cnt.data_ptr(),
                                            ws.data_ptr(), ws.numel(), stream_ptr) == 0
                tgt, oth, tm = update_messages(src, dst, t)
                plan = make_plan(tgt, oth, world, rank, n_local)
                M = int(cnt.item())
                assert M == len(plan.keep)
                assert np.array_equal(first[:M].cpu().numpy(), plan.first_rows)
                assert np.array_equal(tout[:M].cpu().numpy(), tm[plan.keep])
                got2 = second[:M].cpu().numpy()
                remote = plan.second_rows >= n_local
                assert np.array_equal(got2[~remote], plan.second_rows[~remote])
                n_need = int(ctr[0].item())
                assert n_need == plan.num_recv and int(ctr[1].item()) == 0 and int(ctr[2].item()) == 0
                nodes = need[:n_need].cpu().numpy()
                assert len(np.unique(nodes)) == n_need                       # one slot per distinct remote node
                assert np.array_equal(nodes[got2[remote] - n_local], oth[plan.keep][remote])
                # a second call in the same generation re-uses the slots: pairs (src, dst) need nothing new
                keep = torch.empty(B, dtype=torch.int64, device=dev)
                assert lib.tpn_route_pairs(ctypes.byref(sh), ds.data_ptr(), dd.data_ptr(), B, first.data_ptr(),
                                           second.data_ptr(), keep.data_ptr(), cnt.data_ptr(), ws.data_ptr(),
                                           ws.numel(), stream_ptr) == 0
                pplan = make_plan(src, dst, world, rank, n_local)
                Mp = int(cnt.item())
                assert Mp == len(pplan.keep) and np.array_equal(keep[:Mp].cpu().numpy(), pplan.keep)
                assert int(ctr[0].item()) == n_need and int(ctr[1].item()) == n_need
                got2 = second[:Mp].cpu().numpy()
                premote = pplan.second_rows >= n_local
                assert np.array_equal(nodes[got2[premote] - n_local], dst[pplan.keep][premote])
