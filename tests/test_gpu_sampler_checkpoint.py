"""GPU suite of the streaming-sampler checkpoint (tpnet_b200/checkpoint.py: save_sampler / load_sampler).

A sampler saved at any point of a stream and loaded into a fresh sampler of any world size continues the stream with
answers bit-equal to the sampler that never stopped.  In-process ranks (LocalPeerGroup), each on its own stream, one
phase at a time, as in tests/test_gpu_sharded_sampler.py; the real multi-process run is
tests/dist_gpu_resume_check.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.neighbor_sampler import RecentNeighborOracle
from tpnet_b200 import _lib
from tpnet_b200 import checkpoint as ck
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
    """One phase on every rank (each on its own stream), then a device-wide sync (LocalPeerGroup.host_barriers)."""
    out = []
    for s, st in zip(ranks, streams):
        with torch.cuda.stream(st):
            out.append(fn(s))
    torch.cuda.synchronize()
    return out


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
            o[keep] = a.cpu().numpy()
    assert np.all(seen == 1)
    return tuple(out)


def assert_same(got, ref, where=''):
    for g, r, name in zip(got, ref, ('nbr', 'eid', 't')):
        assert g.shape == r.shape and g.dtype == r.dtype, (where, name)
        assert np.array_equal(g, r), (where, name, int((g != r).sum()))


def tied_stream(rng, N, sizes, span):
    """Power-law ids with a hub (node 7) in every batch, ~3 % self-loops, the top 40 ids never pushed, times on an
    integer grid of `span` steps (ties inside and across batches).  Returns src, dst, eid, t and the batch ends."""
    E = int(sum(sizes))
    src = (rng.zipf(1.3, E) - 1) % (N - 40)
    dst = (rng.zipf(1.3, E) - 1) % (N - 40)
    src[rng.random(E) < 0.2] = 7
    loops = rng.random(E) < 0.03
    dst[loops] = src[loops]
    t = np.sort(np.floor(rng.random(E) * span))
    return src.astype(np.int64), dst.astype(np.int64), np.arange(1, E + 1), t, np.cumsum(sizes)


def loop_queries(rng, src, dst, t, N, lo, hi, extra=64):
    """TPNet's queries after pushing edges [lo, hi) (src, dst, negatives at the batch's times, so most lie inside the
    pending batch, before its last time), plus random nodes, unseen ones included, at and after its last time."""
    bt = t[lo:hi]
    qn = np.concatenate([src[lo:hi], dst[lo:hi], rng.integers(0, N, hi - lo), rng.integers(0, N, extra)])
    qt = np.concatenate([bt, bt, bt, bt[-1] + np.floor(rng.random(extra) * 3.0)])
    return qn.astype(np.int64), qt


def batch(stream, i):
    src, dst, eid, t, cuts = stream
    lo = cuts[i - 1] if i else 0
    return src[lo:cuts[i]], dst[lo:cuts[i]], eid[lo:cuts[i]], t[lo:cuts[i]]


def uninterrupted(stream, N, C, Ks, max_batch, seed):
    """One StreamingRecentSampler fed the whole stream: the queries of every batch and their answers per K."""
    src, dst, eid, t, cuts = stream
    rng = np.random.default_rng(seed)
    plain = StreamingRecentSampler(N, C, DEV, max_batch=max_batch)
    queries, answers = [], {}
    for i in range(len(cuts)):
        plain.push(*batch(stream, i))
        queries.append(loop_queries(rng, src, dst, t, N, cuts[i - 1] if i else 0, cuts[i]))
        for K in Ks:
            answers[i, K] = plain.get_historical_neighbors(*queries[-1], K)
    plain.check_errors()
    return queries, answers


# ---------------------------------------------------------------- 1. world 1: save at two points, continue
@pytest.mark.parametrize('C', [1, 20, 40])
def test_resume_at_world_one(tmp_path, C):
    """Saved after batch j's queries ('after') and between push j+1 and its queries ('between', the pending batch is
    then the one being queried, at times before its last one).  A fresh sampler, used on another stream first, loads
    either and answers every later query exactly as the uninterrupted sampler and the oracle over the pushed prefix.
    Loading 'after' grows the loader's pending buffers (batch j has 1,500 edges, max_batch is 300)."""
    N, j = 3000, 3
    stream = tied_stream(np.random.default_rng(C), N, [1, 700, 3, 1500, 64, 900, 5, 1200], span=150.0)
    src, dst, eid, t, cuts = stream
    Ks = sorted({1, C})
    assert len(np.unique(batch(stream, j + 1)[3])) > 1                 # the 'between' batch spans several times
    rng = np.random.default_rng(5)
    a = StreamingRecentSampler(N, C, DEV, max_batch=512)
    answers, queries = {}, []
    for i in range(len(cuts)):
        a.push(*batch(stream, i))
        if i == j + 1:
            ck.save_sampler(a, str(tmp_path), 'between')
        queries.append(loop_queries(rng, src, dst, t, N, cuts[i - 1] if i else 0, cuts[i]))
        for K in Ks:
            answers[i, K] = a.get_historical_neighbors(*queries[-1], K)
        if i == j:
            ck.save_sampler(a, str(tmp_path), 'after', chunk_bytes=1000 * ck.sampler_row_bytes(C))
    a.check_errors()
    for tag, first_push in (('after', j + 1), ('between', j + 2)):
        b = StreamingRecentSampler(N, C, DEV, max_batch=300)
        b.push(np.array([1, 2]), np.array([3, 3]), np.array([9, 9]), np.array([1e6, 1e6]))   # overwritten by the load
        b.push(np.array([1]), np.array([2]), np.array([9]), np.array([2e6]))
        ck.load_sampler(b, str(tmp_path), tag)
        assert b.max_batch == (1500 if tag == 'after' else 300)
        for i in range(j + 1, len(cuts)):
            if i >= first_push:
                b.push(*batch(stream, i))
            o = RecentNeighborOracle(src[:cuts[i]], dst[:cuts[i]], eid[:cuts[i]], t[:cuts[i]], N)
            for K in Ks:
                got = b.get_historical_neighbors(*queries[i], K)          # numpy results: the error flag is checked
                assert_same(got, answers[i, K], (tag, i, K))
                assert_same(got, o.get_historical_neighbors(*queries[i], K), (tag, i, K, 'oracle'))


# ---------------------------------------------------------------- 2. + 3. re-sharding, chunks, a rank without rows
def resume_sharded(tmp_path, stream, N, C, Ks, j, saved_world, load_world, cache_rows, save_chunk=None,
                   load_chunk=None, seed=3):
    """Ranks of `saved_world` push batches 0..j and are saved between push j and its queries; a fresh job of
    `load_world` ranks loads them and answers batch j's queries, then pushes and queries the rest.  The assembled
    slices equal the uninterrupted plain sampler's answers."""
    queries, answers = uninterrupted(stream, N, C, Ks, 256, seed)
    rb = ck.sampler_row_bytes(C)
    kw = lambda chunk: {} if chunk is None else {'chunk_bytes': chunk * rb}     # noqa: E731
    tag = f'w{saved_world}'
    saved, ss = make_ranks(saved_world, N, C, 256, N)
    for i in range(j + 1):
        each(saved, ss, lambda s: s.push(*batch(stream, i)))
        if i < j:
            assert_same(query_all(saved, ss, *queries[i], Ks[-1]), answers[i, Ks[-1]])
    each(saved, ss, lambda s: ck.save_sampler(s, str(tmp_path), tag, **kw(save_chunk)))
    loaded, ls = make_ranks(load_world, N, C, 256, cache_rows)
    each(loaded, ls, lambda s: ck.load_sampler(s, str(tmp_path), tag, **kw(load_chunk)))
    for i in range(j, len(stream[4])):
        if i > j:
            each(loaded, ls, lambda s: s.push(*batch(stream, i)))
        for K in Ks:
            assert_same(query_all(loaded, ls, *queries[i], K), answers[i, K], (saved_world, load_world, i, K))
        if i == j and load_world > 1 and N > load_world:       # the first answers after the load read remote lists
            assert sum(int(s._counters[_lib.SHARD_CTR_NEED].item()) for s in loaded) > 0
    for s in saved + loaded:
        s.check_errors()


@pytest.mark.parametrize('saved_world', [1, 2, 3])
@pytest.mark.parametrize('load_world', [1, 2, 3, 4])
def test_resharding(tmp_path, saved_world, load_world):
    N = 2000
    stream = tied_stream(np.random.default_rng(saved_world * 10 + load_world), N, [400, 1, 900, 250, 600, 333], 80.0)
    resume_sharded(tmp_path, stream, N, 20, [1, 20], 2, saved_world, load_world, cache_rows=N // 2)


def test_small_chunks_and_a_rank_without_rows(tmp_path):
    """Chunks of 7 rows on save and 5 on load (ragged tails); N = 3 < world 4, so one saved shard owns no rows."""
    N = 2503
    stream = tied_stream(np.random.default_rng(1), N, [300, 2000, 40, 700], 60.0)
    resume_sharded(tmp_path / 'a', stream, N, 6, [4, 6], 2, 3, 2, cache_rows=N, save_chunk=7, load_chunk=5)
    rng = np.random.default_rng(2)
    E = 40
    tiny = (rng.integers(0, 3, E), rng.integers(0, 3, E), np.arange(E), np.sort(np.floor(rng.random(E) * 8.0)),
            np.array([3, 4, 17, 30, 40]))
    for load_world in (1, 2, 4):
        resume_sharded(tmp_path / f'tiny{load_world}', tiny, 3, 4, [2, 4], 2, 4, load_world, cache_rows=3,
                       save_chunk=1, load_chunk=2)


# ---------------------------------------------------------------- 4. a graph captured before the load
def test_graph_captured_before_the_load_stays_valid(tmp_path):
    """A push + query step captured on a sampler, then a load into it: replaying the graph continues the saved stream
    exactly as eager calls on the saved sampler do, and no table moved."""
    N, C, K, B, j = 1500, 20, 20, 256, 3
    rng = np.random.default_rng(4)
    stream = tied_stream(rng, N, [B] * 8, 40.0)
    src, dst, eid, t, cuts = stream
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)      # noqa: E731
    a = StreamingRecentSampler(N, C, DEV, max_batch=B)
    for i in range(j + 1):
        a.push(*batch(stream, i))
        a.get_historical_neighbors(*loop_queries(rng, src, dst, t, N, cuts[i] - B, cuts[i]), K)
    ck.save_sampler(a, str(tmp_path), 'g')
    s = StreamingRecentSampler(N, C, DEV, max_batch=B)
    static = [d(x) for x in batch(stream, 7)]
    qn, qt = (d(x) for x in loop_queries(rng, src, dst, t, N, cuts[6], cuts[7], extra=0))
    s.push(*static)                                                     # warm-up, then the capture
    s.get_historical_neighbors(qn, qt, K, as_tensors=True)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        s.push(*static)
        out = s.get_historical_neighbors(qn, qt, K, as_tensors=True)
    tables = list(s._lists.values()) + [s._all_cnt, s._old_cnt, s._newest, s._pend_count, s._last_time, s._err,
                                        s._ws] + list(s._pend.values())
    ptrs = [x.data_ptr() for x in tables]
    ck.load_sampler(s, str(tmp_path), 'g')
    assert [x.data_ptr() for x in tables] == ptrs
    for i in range(j + 1, 8):
        b = [d(x) for x in batch(stream, i)]
        q = [d(x) for x in loop_queries(rng, src, dst, t, N, cuts[i] - B, cuts[i], extra=0)]
        for x, y in zip(static + [qn, qt], b + q):
            x.copy_(y)
        graph.replay()
        a.push(*b)
        want = a.get_historical_neighbors(*q, K, as_tensors=True)
        torch.cuda.synchronize()
        for g_, w in zip(out, want):
            assert torch.equal(g_, w), i
    s.check_errors()
    a.check_errors()


# ---------------------------------------------------------------- 5. refusals
def test_refusals_leave_the_sampler_as_it_was(tmp_path):
    N, C, K = 500, 8, 8
    d = str(tmp_path)
    stream = tied_stream(np.random.default_rng(6), N, [300, 200], 20.0)
    saved, ss = make_ranks(2, N, C, 256, N)
    for i in range(2):
        each(saved, ss, lambda s: s.push(*batch(stream, i)))
    each(saved, ss, lambda s: ck.save_sampler(s, d, 'two'))
    probe = (np.arange(N), np.full(N, 1e9))
    victim = StreamingRecentSampler(N, C, DEV, max_batch=256)
    victim.push(*batch(stream, 0))
    before = victim.get_historical_neighbors(*probe, K)

    def refused(exc, match, sampler=victim, tag='two'):
        with pytest.raises(exc, match=match):
            ck.load_sampler(sampler, d, tag)

    refused(ValueError, 'checkpoint is for', StreamingRecentSampler(N + 1, C, DEV))
    refused(ValueError, 'checkpoint is for', StreamingRecentSampler(N, C + 1, DEV))
    os.rename(ck.shard_path(d, 'two', 1, 2), os.path.join(d, 'moved'))
    refused(FileNotFoundError, 'ranks \\[1\\]')
    os.rename(os.path.join(d, 'moved'), ck.shard_path(d, 'two', 1, 2))
    ck.save_sampler(victim, d, 'two')                                   # a world-1 shard beside the world-2 ones
    refused(ValueError, 'mixes world sizes')
    os.remove(ck.shard_path(d, 'two', 0, 1))
    with open(ck.lists_path(ck.shard_path(d, 'two', 0, 2)), 'r+b') as fh:
        fh.truncate(100)
    refused(ValueError, 'bytes, expected')
    assert_same(victim.get_historical_neighbors(*probe, K), before)    # nothing was written
    # a flagged sampler (device-resident times out of order) is refused before any file is written
    victim.push(torch.tensor([1, 2], device=DEV), torch.tensor([3, 4], device=DEV), torch.tensor([7, 8], device=DEV),
                torch.tensor([2e9, 1e9], dtype=torch.float64, device=DEV))
    with pytest.raises(ValueError, match='decreased'):
        ck.save_sampler(victim, os.path.join(d, 'flagged'))
    assert not os.path.exists(os.path.join(d, 'flagged'))
    for s in saved:
        s.check_errors()


# ---------------------------------------------------------------- 6. the whole TPNet job, state and sampler
def _job(world, N, K, B, mode):
    """`world` ranks of ShardedRandomProjection + ShardedStreamingSampler (in-process peers at world > 1)."""
    from tpnet_b200.peer import LocalPeerGroup
    from tpnet_b200.sharded import ShardedRandomProjection
    kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=3, time_decay_weight=1e-4, device=DEV,
              use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=140, decay_mode=mode,
              state_device=DEV)
    if world == 1:
        torch.manual_seed(11)
        states = [ShardedRandomProjection(ext_rows=64, **kw).to(DEV)]
        samplers = [ShardedStreamingSampler(N, K, DEV, max_batch=B)]
    else:
        groups = LocalPeerGroup.create(world)
        states = []
        for r in range(world):
            torch.manual_seed(11)                  # p0='global': every rank draws the same global P_0, keeps its rows
            states.append(ShardedRandomProjection(ext_rows=2 * N + 64, peers=groups[r], exchange='peer', **kw).to(DEV))
        for m in states:
            m.connect()
        samplers, _ = make_ranks(world, N, K, B, N)
    return list(zip(samplers, states)), [torch.cuda.Stream() for _ in range(world)]


def _step(job, s, d_, n_, e, ts, K):
    """push -> sliced query -> sliced encoder call -> both decoder calls -> update; every output assembled."""
    pairs, streams = job
    rows, times = np.concatenate([s, d_]), np.concatenate([ts, ts])
    each(pairs, streams, lambda p: p[0].push(s, d_, e, ts))
    sliced = each(pairs, streams, lambda p: p[0].get_historical_neighbors(rows, times, K, as_tensors=True))
    enc = each(pairs, streams, lambda p: p[1].get_neighbor_pair_wise_feature(
        sliced[p[0].rank][1], np.concatenate([s, s]), np.concatenate([d_, d_]), sliced_neighbors=True))
    pos = each(pairs, streams, lambda p: p[1].get_pair_wise_feature(s, d_))
    neg = each(pairs, streams, lambda p: p[1].get_pair_wise_feature(s, n_))
    out = {}
    for name, parts, n in (('nbr', [(x[0], x[1]) for x in sliced], 2 * len(s)),
                           ('eid', [(x[0], x[2]) for x in sliced], 2 * len(s)),
                           ('t', [(x[0], x[3]) for x in sliced], 2 * len(s)),
                           ('enc', enc, 2 * len(s)), ('pos', pos, len(s)), ('neg', neg, len(s))):
        full = torch.zeros((n,) + tuple(parts[0][1].shape[1:]), dtype=parts[0][1].dtype, device=DEV)
        for keep, f in parts:
            full[torch.as_tensor(keep, device=DEV)] = f
        out[name] = full
    if len(pairs) == 1:
        pairs[0][1].update(s, d_, ts)
    else:
        pending = each(pairs, streams, lambda p: p[1].update_begin(s, d_, ts))
        for (_, m), st, pd in zip(pairs, streams, pending):
            with torch.cuda.stream(st):
                m.update_end(pd)
        torch.cuda.synchronize()
    return out


def _state_rows(job, N):
    pairs, streams = job
    ids = np.arange(N, dtype=np.int64)
    parts = each(pairs, streams, lambda p: p[1].get_random_projections(ids))
    if len(pairs) == 1:
        return torch.stack(parts[0])
    full = torch.zeros((len(parts[0][1]), N, parts[0][1][0].shape[1]), device=DEV)
    for keep, layers in parts:
        full[:, keep] = torch.stack(layers)
    return full


def _check_job(job):
    for sm, st in job[0]:
        sm.check_errors()
        st.check_errors()


@pytest.mark.parametrize('mode', ['eager', 'lazy'])
@pytest.mark.parametrize('load_world', [3, 1])
def test_whole_job_saved_at_world_two_resumes_at_another_size(tmp_path, mode, load_world):
    """The TPNet batch loop on the sharded state + sharded sampler at world 2 is saved (save_checkpoint + save_sampler)
    at a batch boundary and loaded into a fresh job of `load_world` ranks, which runs 3 more batches.  Against the
    same job run without a stop at that world size: sampler answers bit-equal; features and state rows bit-equal in
    eager mode, and within tests/test_gpu_checkpoint.py's bound in lazy mode (the reloaded state restarts its decay
    log: one more rounding per row)."""
    N, K, B, j = 997, 20, 600, 1
    nb = j + 4
    rng = np.random.default_rng(load_world)
    E = B * nb
    src = (1 + (rng.zipf(1.3, E) - 1) % (N - 1)).astype(np.int64)
    dst = (1 + (rng.zipf(1.3, E) - 1) % (N - 1)).astype(np.int64)
    neg = rng.integers(1, N, E).astype(np.int64)
    t = np.sort(np.floor(rng.random(E) * 40.0) * 10.0)
    eid = np.arange(1, E + 1)
    b = lambda i: tuple(x[i * B:(i + 1) * B] for x in (src, dst, neg, eid, t))     # noqa: E731
    d = str(tmp_path)
    with torch.no_grad():
        saving = _job(2, N, K, B, mode)
        for i in range(j + 1):
            _step(saving, *b(i), K)
        each(*saving, lambda p: (ck.save_checkpoint(p[1], d, 'state'), ck.save_sampler(p[0], d, 'sampler')))
        _check_job(saving)
        ref = _job(load_world, N, K, B, mode)
        for _, m in ref[0]:                        # the head the checkpoint carries
            m.mlp.load_state_dict(saving[0][0][1].mlp.state_dict())
        want = [_step(ref, *b(i), K) for i in range(nb)][j + 1:]
        want_rows = _state_rows(ref, N)
        resumed = _job(load_world, N, K, B, mode)
        each(*resumed, lambda p: (ck.load_checkpoint(p[1], d, 'state'), ck.load_sampler(p[0], d, 'sampler')))
        got = [_step(resumed, *b(i), K) for i in range(j + 1, nb)]
        got_rows = _state_rows(resumed, N)
    for i, (g, w) in enumerate(zip(got, want)):
        for name in g:
            if mode == 'eager' or name in ('nbr', 'eid', 't'):
                assert torch.equal(g[name], w[name]), (i, name)
            else:
                scale = max(float(w[name].abs().max()), 1.0)
                assert torch.allclose(g[name], w[name], rtol=1e-5, atol=1e-6 * scale), (i, name)
    if mode == 'eager':
        assert torch.equal(got_rows, want_rows)
    else:
        scale = max(float(want_rows.abs().max()), 1.0)
        assert torch.allclose(got_rows, want_rows, rtol=1e-5, atol=1e-6 * scale)
    _check_job(ref)
    _check_job(resumed)


# ---------------------------------------------------------------- real ranks
def test_resume_real_ranks(tmp_path):
    """One process per GPU (torchrun): saved at world 2, resumed at world 1 and back (tests/dist_gpu_resume_check.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    script = os.path.join(ROOT, 'tests', 'dist_gpu_resume_check.py')
    for save_world, load_world in ((2, 1), (1, 2)):
        d = str(tmp_path / f'{save_world}to{load_world}')
        for phase, world in (('save', save_world), ('resume', load_world)):
            cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world),
                   '--master-addr', '127.0.0.1', '--master-port', '29547', script, '--phase', phase, '--dir', d]
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
            assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        assert 'PASS' in r.stdout
