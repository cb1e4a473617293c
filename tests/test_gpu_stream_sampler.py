"""GPU suite of the streaming `recent` sampler (StreamingRecentSampler, tpn_stream_sampler_*): after every push its
answers equal RecentNeighborOracle built over the pushed prefix, bit for bit in all three arrays, for the queries
TPNet's loop makes (the batch's src, dst and negatives at the batch's times) and for later times."""
import numpy as np
import pytest
import torch

from oracle.neighbor_sampler import RecentNeighborOracle
from tpnet_b200 import RandomProjectionModule, synth
from tpnet_b200.neighbor_sampler import RecentNeighborSampler, StreamingRecentSampler
from tpnet_b200.pipeline import EpochBatches, StepGraphs

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def assert_same(got, ref, where=''):
    for g, r, name in zip(got, ref, ('nbr', 'eid', 't')):
        g = g.cpu().numpy() if isinstance(g, torch.Tensor) else g
        assert g.shape == r.shape and g.dtype == r.dtype, (where, name)
        assert np.array_equal(g, r), (where, name, int((g != r).sum()))


def loop_queries(rng, src, dst, t, N, lo, hi, extra=64):
    """TPNet's queries after pushing edges [lo, hi): src, dst and negatives at the batch's times, plus random nodes
    at and after the batch's last time."""
    bt = t[lo:hi]
    neg = rng.integers(0, N, hi - lo)
    rnd = rng.integers(0, N, extra)
    qn = np.concatenate([src[lo:hi], dst[lo:hi], neg, rnd]).astype(np.int64)
    qt = np.concatenate([bt, bt, bt, bt[-1] + np.floor(rng.random(extra) * 3.0)])
    return qn, qt


def drive(s, src, dst, eid, t, N, cuts, Ks, rng, max_q=40_000):
    lo = 0
    for hi in cuts:
        s.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        qn, qt = loop_queries(rng, src, dst, t, N, lo, hi)
        if len(qn) > max_q:
            pick = np.sort(rng.choice(len(qn), max_q, replace=False))
            qn, qt = qn[pick], qt[pick]
        for K in Ks:
            assert_same(s.get_historical_neighbors(qn, qt, K), o.get_historical_neighbors(qn, qt, K), (hi, K))
        lo = hi
    s.check_errors()


@pytest.mark.parametrize('K,C', [(1, 1), (20, 20), (33, 40)])
def test_ragged_batches_with_ties_match_oracle(K, C):
    rng = np.random.default_rng(K)
    N = 5000
    sizes = [1, 4096, 1, 100_000, 7, 2500, 1, 3000]
    E = sum(sizes)
    src = (rng.zipf(1.3, E) - 1) % N
    dst = (rng.zipf(1.3, E) - 1) % N
    t = np.sort(np.floor(rng.random(E) * 150.0))            # ~740 edges per timestamp: ties cross every boundary
    eid = np.arange(1, E + 1)
    s = StreamingRecentSampler(N, C, DEV, max_batch=4096)     # the 100,000-edge batch grows the buffers
    drive(s, src, dst, eid, t, N, np.cumsum(sizes), sorted({1, K}), rng)


def test_more_than_capacity_entries_at_one_time_straddling_a_push():
    C = 4
    # node 1: 3 entries at t=1, then 9 at t=5 split 5 | 4 over two pushes, then 2 at t=6
    src = np.array([1, 1, 1] + [1] * 9 + [1, 1, 2, 3], dtype=np.int64)
    dst = np.array([10, 11, 12] + list(range(20, 29)) + [30, 31, 40, 41], dtype=np.int64)
    t = np.array([1.0] * 3 + [5.0] * 9 + [6.0, 6.0, 7.0, 7.0])
    eid = np.arange(1, len(src) + 1)
    N = 50
    s = StreamingRecentSampler(N, C, DEV, max_batch=8)
    qn = np.array([1, 1, 1, 1, 1, 10, 20, 28, 30, 2], dtype=np.int64)
    for lo, hi in ((0, 8), (8, 12), (12, 14), (14, 16)):
        s.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        qt = np.full(len(qn), t[lo]) + np.array([0, 0.5, 1, 2, 100, 0, 0, 1, 3, 0])
        for K in (1, 3, 4):
            assert_same(s.get_historical_neighbors(qn, qt, K), o.get_historical_neighbors(qn, qt, K), (hi, K))
    # at t=5 after the third push node 1's newest folded time is 5: the answer comes from OLD (all three t=1 entries)
    s2 = StreamingRecentSampler(N, C, DEV, max_batch=8)
    for lo, hi in ((0, 8), (8, 12), (12, 14)):
        s2.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
    n_, e_, t_ = s2.get_historical_neighbors(np.array([1]), np.array([5.0]), 4)
    assert n_.tolist() == [[0, 10, 11, 12]] and t_.tolist() == [[0.0, 1.0, 1.0, 1.0]]


def test_flights_shaped_day_quantised_stream():
    shape = synth.SHAPES['flights']
    rng = np.random.default_rng(7)
    parts = list(synth.edge_stream(shape, 3000, 12, seed=3))
    src = np.concatenate([p[0] for p in parts])
    dst = np.concatenate([p[1] for p in parts])
    t = np.concatenate([p[2] for p in parts])
    assert len(np.unique(t)) < 10                                  # whole batches share a day stamp
    eid = np.arange(1, len(src) + 1)
    s = StreamingRecentSampler(shape.node_num, 20, DEV, max_batch=3000)
    drive(s, src, dst, eid, t, shape.node_num, np.arange(3000, len(src) + 1, 3000), [5, 20], rng, max_q=6000)


def test_power_law_replica_with_a_hub_per_batch():
    shape = synth.GraphShape('powerlaw_small', 100_000, 0, 100_000_000, 3, 1e-7, 3.0e6, False, 1.2)
    N, B = shape.node_num, 100_000
    parts = list(synth.edge_stream(shape, B, 3, seed=11))
    src = np.concatenate([p[0] for p in parts])
    dst = np.concatenate([p[1] for p in parts])
    t = np.concatenate([p[2] for p in parts])
    eid = np.arange(1, len(src) + 1)
    deg = np.bincount(np.concatenate([src[:B], dst[:B]]), minlength=N)
    assert deg.max() > 30_000                                      # a hub's segment of one batch
    rng = np.random.default_rng(2)
    s = StreamingRecentSampler(N, 20, DEV, max_batch=B)
    drive(s, src, dst, eid, t, N, [B, 2 * B, 3 * B], [20], rng, max_q=20_000)
    # every one of the loop's 3B queries of the last batch, against the CSR sampler over the whole prefix
    full = RecentNeighborSampler(src, dst, eid, t, DEV, num_nodes=N)
    qn, qt = loop_queries(rng, src, dst, t, N, 2 * B, 3 * B)
    assert_same(s.get_historical_neighbors(qn, qt, 20),
                full.get_historical_neighbors(qn, qt, 20))


def test_self_loops_unseen_nodes_pending_times_and_after_everything():
    N, C = 30, 6
    src = np.array([3, 3, 4, 5, 3, 7, 7, 3], dtype=np.int64)
    dst = np.array([3, 4, 4, 3, 3, 8, 7, 9], dtype=np.int64)
    t = np.array([1.0, 1.0, 2.0, 2.0, 3.0, 3.0, 3.0, 4.0])
    eid = np.arange(100, 108)
    s = StreamingRecentSampler(N, C, DEV, max_batch=4)
    for lo, hi in ((0, 3), (3, 7), (7, 8)):
        s.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        qn = np.array([3, 3, 3, 4, 7, 7, 0, 29, 12, 3, 9], dtype=np.int64)      # 0, 29, 12: never seen
        qt = np.array([t[lo], t[hi - 1], t[hi - 1] + 0.5, t[lo], t[hi - 1], 1e18, 5.0, 1e18, t[lo], np.inf, 1e9])
        for K in (1, 4, 6):
            got = s.get_historical_neighbors(qn, qt, K)
            assert_same(got, o.get_historical_neighbors(qn, qt, K), (hi, K))
            assert not got[0][6:9].any()


def test_tpnet_loop_equals_csr_sampler_on_the_full_stream():
    shape = synth.SHAPES['reddit']
    parts = list(synth.edge_stream(shape, 600, 20, seed=5))
    src = np.concatenate([p[0] for p in parts])
    dst = np.concatenate([p[1] for p in parts])
    t = np.concatenate([p[2] for p in parts])
    eid = np.arange(1, len(src) + 1)
    full = RecentNeighborSampler(src, dst, eid, t, DEV, num_nodes=shape.node_num)
    s = StreamingRecentSampler(shape.node_num, 20, DEV, max_batch=600)
    rng = np.random.default_rng(0)
    for i in range(20):
        lo, hi = 600 * i, 600 * (i + 1)
        s.push(src[lo:hi], dst[lo:hi], eid[lo:hi], t[lo:hi])
        qn, qt = loop_queries(rng, src, dst, t, shape.node_num, lo, hi, extra=0)
        if hi < len(t):
            qt = np.minimum(qt, t[hi])                         # queries at times <= the next batch's first time
        for K in (1, 20):
            a = s.get_historical_neighbors(qn, qt, K)
            b = full.get_historical_neighbors(qn, qt, K)
            for x, y in zip(a, b):
                assert np.array_equal(x, y), (i, K)


def test_device_resident_inputs_and_outputs():
    rng = np.random.default_rng(3)
    N, E, B = 700, 6000, 500
    src = (rng.zipf(1.3, E) - 1) % N
    dst = (rng.zipf(1.3, E) - 1) % N
    t = np.sort(np.floor(rng.random(E) * 40.0))
    eid = rng.integers(1, 1 << 40, E)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    s = StreamingRecentSampler(N, 20, DEV, max_batch=B)
    for lo in range(0, E, B):
        hi = lo + B
        s.push(d(src[lo:hi]), d(dst[lo:hi]), d(eid[lo:hi]), d(t[lo:hi]))
        o = RecentNeighborOracle(src[:hi], dst[:hi], eid[:hi], t[:hi], N)
        qn, qt = loop_queries(rng, src, dst, t, N, lo, hi)
        got = s.get_historical_neighbors(d(qn), d(qt), 20, as_tensors=True)
        assert all(x.is_cuda for x in got) and got[0].dtype == torch.int64 and got[2].dtype == torch.float64
        assert_same(got, o.get_historical_neighbors(qn, qt, 20), hi)
    s.check_errors()


def test_error_paths():
    d = lambda a: torch.as_tensor(a).to(DEV)
    s = StreamingRecentSampler(10, 4, DEV, max_batch=4)
    s.push(np.array([1, 2]), np.array([3, 4]), np.array([1, 2]), np.array([5.0, 6.0]))
    with pytest.raises(ValueError):                                      # host: decreasing within a batch
        s.push(np.array([1, 2]), np.array([3, 4]), np.array([3, 4]), np.array([8.0, 7.0]))
    with pytest.raises(ValueError):                                      # host: before the previous batch
        s.push(np.array([1]), np.array([3]), np.array([3]), np.array([5.5]))
    with pytest.raises(IndexError):
        s.push(np.array([1]), np.array([10]), np.array([3]), np.array([7.0]))
    with pytest.raises(IndexError):
        s.get_historical_neighbors(np.array([-1]), np.array([7.0]), 2)
    with pytest.raises(ValueError):
        s.get_historical_neighbors(np.array([1]), np.array([7.0]), 5)     # num_neighbors > max_neighbors
    s.check_errors()                                                     # nothing launched so far was flagged
    # device-resident: flagged on the device, raised by check_errors
    s.push(d([1, 2]), d([3, 11]), d([5, 6]), d([7.0, 7.0]))
    with pytest.raises(IndexError):
        s.check_errors()
    s.check_errors()                                                     # the flag was cleared
    s.push(d([1, 2]), d([3, 4]), d([7, 8]), d([8.0, 7.5]))
    with pytest.raises(ValueError, match='decreased'):
        s.check_errors()
    s.reset()
    s.push(d([1]), d([3]), d([1]), d([5.0]))
    s.push(d([1]), d([3]), d([2]), d([4.0]))                             # starts before the previous batch
    with pytest.raises(ValueError, match='decreased'):
        s.check_errors()
    s.reset()
    s.push(np.array([1]), np.array([3]), np.array([1]), np.array([5.0]))
    s.push(np.array([1]), np.array([3]), np.array([2]), np.array([6.0]))  # node 1's newest folded time is now 5
    got = s.get_historical_neighbors(d([1, 1]), d([4.0, 6.0]), 2, as_tensors=True)
    with pytest.raises(ValueError, match='before the newest time'):
        s.check_errors()
    assert not got[0][0].any() and got[0][1].tolist() == [0, 3]
    with pytest.raises(ValueError, match='before the newest time'):      # numpy results check the flag themselves
        s.get_historical_neighbors(np.array([1]), np.array([4.0]), 2)
    with pytest.raises(IndexError):
        s.get_historical_neighbors(d([12]), d([9.0]), 2)


def test_reset_matches_a_fresh_sampler():
    rng = np.random.default_rng(9)
    N, E, B = 300, 3000, 250
    src = (rng.zipf(1.3, E) - 1) % N
    dst = (rng.zipf(1.3, E) - 1) % N
    t = np.sort(np.floor(rng.random(E) * 30.0))
    eid = np.arange(E)
    used = StreamingRecentSampler(N, 8, DEV, max_batch=B)
    for lo in range(0, E, B):
        used.push(src[lo:lo + B], dst[lo:lo + B], eid[lo:lo + B], t[lo:lo + B])
    used.reset()
    fresh = StreamingRecentSampler(N, 8, DEV, max_batch=B)
    q = np.arange(N)
    for lo in range(0, 1000, B):
        for s in (used, fresh):
            s.push(src[lo:lo + B], dst[lo:lo + B], eid[lo:lo + B], t[lo:lo + B])
        qt = np.full(N, t[lo + B - 1])
        for x, y in zip(used.get_historical_neighbors(q, qt, 8), fresh.get_historical_neighbors(q, qt, 8)):
            assert np.array_equal(x, y)


def test_graph_capture_of_push_query_encoder_update_equals_eager():
    rng = np.random.default_rng(1)
    N, E, B, K = 2000, 4096, 512, 20
    src = 1 + (rng.zipf(1.3, E) - 1) % (N - 1)
    dst = 1 + (rng.zipf(1.3, E) - 1) % (N - 1)
    t = np.sort(np.floor(rng.random(E) * 64.0))
    eid = np.arange(1, E + 1)
    batches = EpochBatches(src, dst, t, B, DEV, extra={'eid': eid})

    def make():
        torch.manual_seed(0)
        m = RandomProjectionModule(node_num=N, edge_num=E + 1, dim_factor=10, num_layer=3, time_decay_weight=1e-6,
                                   device=DEV, use_matrix=False, beginning_time=np.float64(0.0), not_scale=False,
                                   enforce_dim=-1).to(DEV)
        return m, StreamingRecentSampler(N, K, DEV, max_batch=B)

    def step_for(sampler):
        def step(module, b, out):
            sampler.push(b.src, b.dst, b.extra['eid'], b.t)
            rows = torch.cat([b.src, b.dst])
            nbr, e_, t_ = sampler.get_historical_neighbors(rows, torch.cat([b.t, b.t]), K, as_tensors=True)
            out['nbr'].copy_(nbr)
            out['eid'].copy_(e_)
            out['t'].copy_(t_)
            module.get_neighbor_pair_wise_feature(nbr, torch.cat([b.src, b.src]), torch.cat([b.dst, b.dst]),
                                                  out=out['enc'])
            module.update(b.src, b.dst, b.t, next_time=b.t_last)
        return step

    def outs(module):
        return {'nbr': torch.zeros(2 * B, K, dtype=torch.int64, device=DEV),
                'eid': torch.zeros(2 * B, K, dtype=torch.int64, device=DEV),
                't': torch.zeros(2 * B, K, dtype=torch.float64, device=DEV),
                'enc': torch.zeros(2 * B, K, 2 * module.pair_wise_feature_dim, device=DEV)}

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
    # and the sampled neighbours are the reference's
    o = RecentNeighborOracle(src, dst, eid, t, N)
    lo = E - B
    ref = o.get_historical_neighbors(np.concatenate([src[lo:], dst[lo:]]), np.tile(t[lo:], 2), K)
    assert_same((replayed[-1]['nbr'], replayed[-1]['eid'], replayed[-1]['t']), ref)
    s1.check_errors()
    s2.check_errors()
    m1.check_errors()
    for a, b in zip(m1.random_projections, m2.random_projections):
        assert torch.equal(a, b)
