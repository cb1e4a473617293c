"""GPU suite of the node-sharded streaming sampler (ShardedStreamingSampler, tpn_stream_shard_*).

All ranks run inside this process (LocalPeerGroup), each on its own stream, one phase at a time (push on every rank,
then the queries of every rank), as in tests/test_gpu_sharded_encoder.py.  After every push the slices of all ranks,
put back together by position, are bit-equal in all three arrays to a StreamingRecentSampler fed the same stream (that
sampler is pinned to oracle/neighbor_sampler.py by tests/test_gpu_stream_sampler.py); some streams are also checked
against the oracle directly.  The real multi-process run (NVLink pulls, flag barriers) is
tests/dist_gpu_sampler_check.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.neighbor_sampler import RecentNeighborOracle
from tpnet_b200 import RandomProjectionModule, synth
from tpnet_b200.neighbor_sampler import ShardedStreamingSampler, StreamingRecentSampler

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'


# ---------------------------------------------------------------- in-process ranks
def make_ranks(world, N, C, max_batch, cache_rows):
    from tpnet_b200.peer import LocalPeerGroup
    groups = LocalPeerGroup.create(world)
    ranks = [ShardedStreamingSampler(N, C, DEV, max_batch=max_batch, peers=groups[r], cache_rows=cache_rows)
             for r in range(world)]
    for s in ranks:                       # every rank published its tables in its constructor
        s.connect()
    return ranks, [torch.cuda.Stream() for _ in range(world)]


def each(ranks, streams, fn):
    """One phase on every rank (each on its own stream), then a device-wide sync: with all ranks on one GPU the
    phases are ordered by the driver instead of tpn_peer_barrier (LocalPeerGroup.host_barriers)."""
    out = []
    for s, st in zip(ranks, streams):
        with torch.cuda.stream(st):
            out.append(fn(s))
    torch.cuda.synchronize()
    return out


def push_all(ranks, streams, *batch):
    each(ranks, streams, lambda s: s.push(*batch))


def query_all(ranks, streams, qn, qt, K):
    """Every rank's slice, assembled by position into the [m, K] arrays; every position covered exactly once."""
    parts = each(ranks, streams, lambda s: s.get_historical_neighbors(qn, qt, K, as_tensors=True))
    m = len(qn)
    out = [np.zeros((m, K), dtype=np.int64), np.zeros((m, K), dtype=np.int64), np.zeros((m, K), dtype=np.float64)]
    seen = np.zeros(m, dtype=np.int64)
    for keep, *arrs in parts:
        keep = keep.cpu().numpy()
        seen[keep] += 1
        for o, a in zip(out, arrs):
            assert a.shape == (len(keep), K)
            o[keep] = a.cpu().numpy()
    assert np.all(seen == 1)
    return tuple(out)


def assert_same(got, ref, where=''):
    for g, r, name in zip(got, ref, ('nbr', 'eid', 't')):
        assert g.shape == r.shape and g.dtype == r.dtype, (where, name)
        assert np.array_equal(g, r), (where, name, int((g != r).sum()))


def loop_queries(rng, src, dst, t, N, lo, hi, extra=64):
    """TPNet's queries after pushing edges [lo, hi) (src, dst, negatives at the batch's times), plus random nodes at
    and after the batch's last time."""
    bt = t[lo:hi]
    qn = np.concatenate([src[lo:hi], dst[lo:hi], rng.integers(0, N, hi - lo), rng.integers(0, N, extra)])
    qt = np.concatenate([bt, bt, bt, bt[-1] + np.floor(rng.random(extra) * 3.0)])
    return qn.astype(np.int64), qt


def drive(world, src, dst, eid, t, N, C, cuts, Ks, rng, max_batch, cache_rows=None, oracle=False):
    """Push the stream in `cuts` on the sharded ranks and on one StreamingRecentSampler; after every push the
    assembled slices equal the plain sampler's answers (and the oracle's over the pushed prefix, if asked)."""
    ranks, streams = make_ranks(world, N, C, max_batch, cache_rows if cache_rows is not None else N)
    plain = StreamingRecentSampler(N, C, DEV, max_batch=max_batch)
    lo = 0
    for hi in cuts:
        batch = (src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        push_all(ranks, streams, *batch)
        plain.push(*batch)
        qn, qt = loop_queries(rng, src, dst, t, N, lo, hi)
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N) if oracle else None
        for K in Ks:
            got = query_all(ranks, streams, qn, qt, K)
            assert_same(got, plain.get_historical_neighbors(qn, qt, K), (world, hi, K))
            if o is not None:
                assert_same(got, o.get_historical_neighbors(qn, qt, K), (world, hi, K, 'oracle'))
        lo = hi
    for s in ranks:
        s.check_errors()
    plain.check_errors()
    return ranks, streams


# ---------------------------------------------------------------- streams
@pytest.mark.parametrize('K,C', [(1, 1), (20, 20), (33, 40)])
@pytest.mark.parametrize('world', [1, 2, 3, 4])
def test_ragged_batches_with_ties(world, K, C):
    """Batches of 1 to 100,000 edges, ~740 edges per timestamp (ties cross every batch boundary); the 100,000-edge
    batch grows the pending buffers.  World 3 is also checked against the oracle."""
    rng = np.random.default_rng(K + 100 * world)
    N = 5000
    sizes = [1, 4096, 1, 100_000, 7, 2500, 1, 3000]
    E = sum(sizes)
    src = (rng.zipf(1.3, E) - 1) % N
    dst = (rng.zipf(1.3, E) - 1) % N
    t = np.sort(np.floor(rng.random(E) * 150.0))
    eid = np.arange(1, E + 1)
    drive(world, src, dst, eid, t, N, C, np.cumsum(sizes), sorted({1, K}), rng, max_batch=4096,
          oracle=(world == 3 and K == 20))


@pytest.mark.parametrize('world', [2, 3, 4])
def test_more_than_capacity_at_one_time_and_the_old_list_of_remote_nodes(world):
    """Node 1 gets 9 entries at t=5 split 5 | 4 over two pushes (C = 4).  Queries of node 1 sit in rank 0's slice,
    and rank 0 never owns node 1: every answer is read from a pulled copy, those at t == newest[1] from OLD."""
    C, N = 4, 50
    src = np.array([1, 1, 1] + [1] * 9 + [1, 1, 2, 3], dtype=np.int64)
    dst = np.array([10, 11, 12] + list(range(20, 29)) + [30, 31, 40, 41], dtype=np.int64)
    t = np.array([1.0] * 3 + [5.0] * 9 + [6.0, 6.0, 7.0, 7.0])
    eid = np.arange(1, len(src) + 1)
    ranks, streams = make_ranks(world, N, C, 8, 16)
    plain = StreamingRecentSampler(N, C, DEV, max_batch=8)
    qn = np.array([1] * 5 + [10, 20, 28, 30, 2] * 3, dtype=np.int64)
    assert ranks[0].row_split(len(qn))[2] >= 5 and 1 % world != 0
    for lo, hi in ((0, 8), (8, 12), (12, 14), (14, 16)):
        push_all(ranks, streams, src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        plain.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        qt = np.full(len(qn), t[lo]) + np.tile(np.array([0, 0.5, 1, 2, 100]), 4)
        for K in (1, 3, 4):
            got = query_all(ranks, streams, qn, qt, K)
            assert_same(got, plain.get_historical_neighbors(qn, qt, K), (hi, K))
            assert_same(got, o.get_historical_neighbors(qn, qt, K), (hi, K, 'oracle'))
    # after the third push node 1's newest folded time is 5: at t = 5 the answer is OLD (the three t=1 entries)
    ranks, streams = make_ranks(world, N, C, 8, 16)
    for lo, hi in ((0, 8), (8, 12), (12, 14)):
        push_all(ranks, streams, src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
    got = query_all(ranks, streams, np.ones(world, dtype=np.int64), np.full(world, 5.0), 4)
    assert got[0].tolist() == [[0, 10, 11, 12]] * world and got[2].tolist() == [[0.0, 1.0, 1.0, 1.0]] * world
    for s in ranks:
        s.check_errors()


@pytest.mark.parametrize('world', [1, 2, 3, 4])
def test_power_law_replica_with_a_hub_per_batch(world):
    shape = synth.GraphShape('powerlaw_small', 100_000, 0, 100_000_000, 3, 1e-7, 3.0e6, False, 1.2)
    N, B = shape.node_num, 100_000
    assert N == 100_001
    parts = list(synth.edge_stream(shape, B, 3, seed=11))
    src = np.concatenate([p[0] for p in parts])
    dst = np.concatenate([p[1] for p in parts])
    t = np.concatenate([p[2] for p in parts])
    eid = np.arange(1, len(src) + 1)
    deg = np.bincount(np.concatenate([src[:B], dst[:B]]), minlength=N)
    assert deg.max() > 30_000                                      # a hub's segment of one batch
    drive(world, src, dst, eid, t, N, 20, [B, 2 * B, 3 * B], [20], np.random.default_rng(2), max_batch=B,
          cache_rows=200_000)


@pytest.mark.parametrize('world', [1, 2, 3, 4])
def test_self_loops_unseen_nodes_and_times_after_everything(world):
    """Checked against the oracle directly: self-loops, nodes never pushed (0, 29, 12), times inside the pending
    batch, at its end, and far after it."""
    N, C = 30, 6
    src = np.array([3, 3, 4, 5, 3, 7, 7, 3], dtype=np.int64)
    dst = np.array([3, 4, 4, 3, 3, 8, 7, 9], dtype=np.int64)
    t = np.array([1.0, 1.0, 2.0, 2.0, 3.0, 3.0, 3.0, 4.0])
    eid = np.arange(100, 108)
    ranks, streams = make_ranks(world, N, C, 4, N)
    for lo, hi in ((0, 3), (3, 7), (7, 8)):
        push_all(ranks, streams, src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        qn = np.array([3, 3, 3, 4, 7, 7, 0, 29, 12, 3, 9], dtype=np.int64)
        qt = np.array([t[lo], t[hi - 1], t[hi - 1] + 0.5, t[lo], t[hi - 1], 1e18, 5.0, 1e18, t[lo], np.inf, 1e9])
        for K in (1, 4, 6):
            got = query_all(ranks, streams, qn, qt, K)
            assert_same(got, o.get_historical_neighbors(qn, qt, K), (hi, K))
            assert not got[0][6:9].any()
    for s in ranks:
        s.check_errors()


# ---------------------------------------------------------------- layout, errors, reset
@pytest.mark.parametrize('world', [2, 3, 4])
def test_each_rank_holds_its_rows_and_the_cache(world):
    from tpnet_b200.sharded import rows_on_rank
    N, C, cache = 1001, 7, 123
    ranks, _ = make_ranks(world, N, C, 16, cache)
    for r, s in enumerate(ranks):
        rows = rows_on_rank(N, world, r) + cache
        assert s.n_local == rows_on_rank(N, world, r)
        assert all(v.shape == (rows, C) for v in s._lists.values())
        assert s._all_cnt.shape == s._old_cnt.shape == s._newest.shape == (rows,)
    one = ShardedStreamingSampler(N, C, DEV, max_batch=16)        # world 1: the plain sampler, no cache
    assert one.world == 1 and one._lists['all_nbr'].shape == (N, C)


def test_error_paths():
    world, N, C = 2, 10, 4
    ranks, streams = make_ranks(world, N, C, 4, N)
    d = lambda a: torch.as_tensor(a).to(DEV)               # noqa: E731
    push_all(ranks, streams, np.array([1, 2]), np.array([3, 4]), np.array([1, 2]), np.array([5.0, 6.0]))
    # host ids: checked before anything is launched (the whole call, on every rank)
    for s in ranks:
        with pytest.raises(IndexError):
            s.get_historical_neighbors(np.array([1, N]), np.array([7.0, 7.0]), 2)
        with pytest.raises(IndexError):
            s.push(np.array([1]), np.array([N]), np.array([3]), np.array([7.0]))
        with pytest.raises(ValueError):
            s.get_historical_neighbors(np.array([1]), np.array([7.0]), C + 1)
        s.check_errors()
    # a device-resident bad id in rank 0's slice: flagged there, raised by check_errors
    each(ranks, streams, lambda s: s.get_historical_neighbors(d([N + 3, 1]), d([7.0, 7.0]), 2, as_tensors=True))
    with pytest.raises(IndexError):
        ranks[0].check_errors()
    ranks[0].check_errors()                                              # the flags were cleared
    ranks[1].check_errors()
    # a past query on a remote node: node 1 lives on rank 1, rank 0's slice asks for it before its newest time
    push_all(ranks, streams, np.array([1]), np.array([3]), np.array([3]), np.array([8.0]))    # newest[1] is now 5
    got = each(ranks, streams, lambda s: s.get_historical_neighbors(d([1, 1]), d([4.0, 8.0]), 2, as_tensors=True))
    with pytest.raises(ValueError, match='before the newest time'):
        ranks[0].check_errors()
    ranks[1].check_errors()
    assert not got[0][1].any() and got[1][1].tolist() == [[0, 3]]     # ALL (t = 5); the t = 8 entry is not older
    # decreasing pushed times (device-resident): flagged on every rank
    push_all(ranks, streams, d([1, 2]), d([3, 4]), d([7, 8]), d([9.0, 8.5]))
    for s in ranks:
        with pytest.raises(ValueError, match='decreased'):
            s.check_errors()
    # one generation's remote lists do not fit the cache
    small, sstreams = make_ranks(world, 100, C, 64, 2)
    push_all(small, sstreams, np.arange(1, 41), np.arange(41, 81), np.arange(40), np.arange(40, dtype=np.float64))
    each(small, sstreams, lambda s: s.get_historical_neighbors(d(np.arange(1, 41)), d(np.full(40, 50.0)), 2,
                                                               as_tensors=True))
    with pytest.raises(RuntimeError, match='cache_rows=2'):
        small[0].check_errors()


@pytest.mark.parametrize('world', [2, 3])
def test_reset_matches_a_fresh_sampler(world):
    rng = np.random.default_rng(9)
    N, E, B = 300, 3000, 250
    src = (rng.zipf(1.3, E) - 1) % N
    dst = (rng.zipf(1.3, E) - 1) % N
    t = np.sort(np.floor(rng.random(E) * 30.0))
    eid = np.arange(E)
    used, us = make_ranks(world, N, 8, B, N)
    for lo in range(0, E, B):
        push_all(used, us, src[lo:lo + B], dst[lo:lo + B], eid[lo:lo + B], t[lo:lo + B])
        query_all(used, us, np.arange(N), np.full(N, t[lo + B - 1]), 8)
    each(used, us, lambda s: s.reset())
    fresh, fs = make_ranks(world, N, 8, B, N)
    q = np.arange(N)
    for lo in range(0, 1000, B):
        for rk, st in ((used, us), (fresh, fs)):
            push_all(rk, st, src[lo:lo + B], dst[lo:lo + B], eid[lo:lo + B], t[lo:lo + B])
        qt = np.full(N, t[lo + B - 1])
        assert_same(query_all(used, us, q, qt, 8), query_all(fresh, fs, q, qt, 8))


# ---------------------------------------------------------------- a whole TPNet batch on the sharded pair
def _state_kw(N):
    return dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=3, time_decay_weight=1e-4, device=DEV,
                use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=140)


def _state_ranks(world, N):
    from tpnet_b200.peer import LocalPeerGroup
    from tpnet_b200.sharded import ShardedRandomProjection
    groups = LocalPeerGroup.create(world)
    ranks = []
    for r in range(world):
        torch.manual_seed(11)                      # p0='global': every rank draws the same global P_0, keeps its rows
        ranks.append(ShardedRandomProjection(decay_mode='lazy', ext_rows=2 * N + 64, peers=groups[r], exchange='peer',
                                             state_device=DEV, **_state_kw(N)).to(DEV))
    for m in ranks:
        for name in ('state', 'stamps', 'flags'):
            m._peers.publish(name, m._peer_bufs[name])
    for m in ranks:
        m.connect()
    torch.manual_seed(11)
    ref = RandomProjectionModule(decay_mode='lazy', **_state_kw(N)).to(DEV)
    for m in ranks:
        m.mlp.load_state_dict(ref.mlp.state_dict())
    return ranks, ref


@pytest.mark.parametrize('world', [2, 4])
def test_tpnet_batch_on_the_sharded_pair(world):
    """push -> sliced query -> sliced encoder call (no all-gather) -> both decoder calls -> update, per batch, on the
    sharded sampler + sharded state; against StreamingRecentSampler + RandomProjectionModule.  Encoder features with
    the tensor-core head (F = 64) and the state's rows are bit-equal; the routed decoder features are compared as in
    tests/test_gpu_sharded_encoder.py."""
    N, K, B, nb = 997, 20, 600, 4
    rng = np.random.default_rng(world)
    E = B * nb
    src = (1 + (rng.zipf(1.3, E) - 1) % (N - 1)).astype(np.int64)
    dst = (1 + (rng.zipf(1.3, E) - 1) % (N - 1)).astype(np.int64)
    neg = rng.integers(1, N, E).astype(np.int64)
    t = np.sort(np.floor(rng.random(E) * 40.0) * 10.0)
    eid = np.arange(1, E + 1)
    states, ref = _state_ranks(world, N)
    samplers, _ = make_ranks(world, N, K, B, N)
    streams = [torch.cuda.Stream() for _ in range(world)]
    plain = StreamingRecentSampler(N, K, DEV, max_batch=B)
    pairs = list(zip(samplers, states))
    with torch.no_grad():
        for i in range(nb):
            lo, hi = i * B, (i + 1) * B
            s, d_, n_, ts = src[lo:hi], dst[lo:hi], neg[lo:hi], t[lo:hi]
            rows, times = np.concatenate([s, d_]), np.concatenate([ts, ts])
            each(pairs, streams, lambda p: p[0].push(s, d_, eid[lo:hi], ts))
            plain.push(s, d_, eid[lo:hi], ts)
            sliced = each(pairs, streams, lambda p: p[0].get_historical_neighbors(rows, times, K, as_tensors=True))
            enc = each(pairs, streams, lambda p: p[1].get_neighbor_pair_wise_feature(
                sliced[p[0].rank][1], np.concatenate([s, s]), np.concatenate([d_, d_]), sliced_neighbors=True))
            pos = each(pairs, streams, lambda p: p[1].routed_pair_wise_feature(s, d_))
            negf = each(pairs, streams, lambda p: p[1].routed_pair_wise_feature(s, n_))
            nbr, _, _ = plain.get_historical_neighbors(rows, times, K, as_tensors=True)
            g = lambda a: torch.from_numpy(np.concatenate(a)).to(DEV)        # noqa: E731
            want = ref.get_neighbor_pair_wise_feature(nbr, g([s, s]), g([d_, d_]))
            got = torch.zeros_like(want)
            for (keep, _, _, _), (keep_e, f) in zip(sliced, enc):
                assert torch.equal(keep, keep_e)
                got[keep_e] = f
            assert torch.equal(got, want), (i, (got - want).abs().max().item())
            for routed, (a, b) in ((pos, (s, d_)), (negf, (s, n_))):
                want = ref.get_pair_wise_feature(a, b)
                got = torch.zeros_like(want)
                for r in routed:
                    k, f = r.trimmed()
                    got[k] = f
                assert torch.allclose(got, want, rtol=1e-5, atol=2e-5), (i, (got - want).abs().max().item())
            pending = each(pairs, streams, lambda p: p[1].update_begin(s, d_, ts))
            for (_, m), st, pd in zip(pairs, streams, pending):
                with torch.cuda.stream(st):
                    m.update_end(pd)
            torch.cuda.synchronize()
            ref.update(s, d_, ts)
        ids = np.arange(N, dtype=np.int64)
        parts = each(pairs, streams, lambda p: p[1].get_random_projections(ids))
        want = ref.get_random_projections(ids)
    for layer in range(4):
        got = torch.zeros_like(want[layer])
        for keep, layers in parts:
            got[keep] = layers[layer]
        assert np.array_equal(got.cpu().numpy(), want[layer].cpu().numpy()), layer
    for sm, st in pairs:
        sm.check_errors()
        st.check_errors()
    plain.check_errors()


def test_world_one_step_graph_capture_equals_eager():
    """World 1: a StepGraphs capture of push -> sliced query -> sliced encoder call -> both decoder calls -> update on
    the sharded pair equals the eager run, and the sampled neighbours are the oracle's."""
    from tpnet_b200.pipeline import EpochBatches, StepGraphs
    from tpnet_b200.sharded import ShardedRandomProjection
    rng = np.random.default_rng(1)
    N, E, B, K = 2000, 4096, 512, 20
    src = 1 + (rng.zipf(1.3, E) - 1) % (N - 1)
    dst = 1 + (rng.zipf(1.3, E) - 1) % (N - 1)
    t = np.sort(np.floor(rng.random(E) * 64.0))
    eid = np.arange(1, E + 1)
    batches = EpochBatches(src, dst, t, B, DEV, extra={'eid': eid})

    def make():
        torch.manual_seed(0)
        m = ShardedRandomProjection(node_num=N, edge_num=E + 1, dim_factor=10, num_layer=3, time_decay_weight=1e-6,
                                    device=DEV, use_matrix=False, beginning_time=np.float64(0.0), not_scale=False,
                                    enforce_dim=-1, decay_mode='lazy', ext_rows=64).to(DEV)
        return m, ShardedStreamingSampler(N, K, DEV, max_batch=B)

    def step_for(sampler):
        def step(module, b, out):
            sampler.push(b.src, b.dst, b.extra['eid'], b.t)
            _, nbr, e_, t_ = sampler.get_historical_neighbors(torch.cat([b.src, b.dst]), torch.cat([b.t, b.t]), K,
                                                              as_tensors=True)
            out['nbr'].copy_(nbr)
            out['eid'].copy_(e_)
            out['t'].copy_(t_)
            module.get_neighbor_pair_wise_feature(nbr, torch.cat([b.src, b.src]), torch.cat([b.dst, b.dst]),
                                                  out=out['enc'], sliced_neighbors=True)
            out['pos'].copy_(module.get_pair_wise_feature(b.src, b.dst)[1])
            out['neg'].copy_(module.get_pair_wise_feature(b.src, torch.flip(b.dst, [0]))[1])
            module.update(b.src, b.dst, b.t, next_time=b.t_last)
        return step

    def outs(module):
        f = module.pair_wise_feature_dim
        return {'nbr': torch.zeros(2 * B, K, dtype=torch.int64, device=DEV),
                'eid': torch.zeros(2 * B, K, dtype=torch.int64, device=DEV),
                't': torch.zeros(2 * B, K, dtype=torch.float64, device=DEV),
                'enc': torch.zeros(2 * B, K, 2 * f, device=DEV),
                'pos': torch.zeros(B, f, device=DEV), 'neg': torch.zeros(B, f, device=DEV)}

    m1, s1 = make()
    with torch.no_grad():
        graphs = StepGraphs(m1, list(batches), step=step_for(s1), out=outs(m1), max_batch=B)
        replayed = []
        for i in range(len(graphs)):
            r = graphs.replay(i)
            replayed.append({k: v.clone() for k, v in r.items()})
    m2, s2 = make()
    o2 = outs(m2)
    with torch.no_grad():
        for i, b in enumerate(batches):
            step_for(s2)(m2, b, o2)
            for k in o2:
                assert torch.equal(o2[k], replayed[i][k]), (i, k)
    o = RecentNeighborOracle(src, dst, eid, t, N)
    lo = E - B
    ref = o.get_historical_neighbors(np.concatenate([src[lo:], dst[lo:]]), np.tile(t[lo:], 2), K)
    assert_same(tuple(replayed[-1][k].cpu().numpy() for k in ('nbr', 'eid', 't')), ref)
    for x in (s1, s2, m1, m2):
        x.check_errors()
    for a, b in zip(m1.random_projections, m2.random_projections):
        assert torch.equal(a, b)


# ---------------------------------------------------------------- real ranks
def test_sharded_sampler_real_ranks():
    """One process per GPU (torchrun), NVLink pulls and flag barriers: tests/dist_gpu_sampler_check.py."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', '29543', os.path.join(ROOT, 'tests', 'dist_gpu_sampler_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'PASS' in r.stdout
