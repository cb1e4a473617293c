"""GPU suite: the persistent, column-half pipelined kernel of large tpn_pairwise calls (pairwise_pipe_kernel).

Every large call is run twice on the same state: with the default kernel and with the one-shot TMA kernel it
replaced (TPN_DEBUG_LEGACY_PAIRWISE).  Both walk each lane's columns in the same order, so the features must be
bit-identical; they are also checked against the oracle within the bound of test_gpu_parity.test_pairwise_large_call.
"""
import numpy as np
import pytest
import torch

from oracle.walk_projection import WalkProjectionOracle
from tpnet_b200 import RandomProjectionModule, _lib

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
LEGACY = 128                                     # TPN_DEBUG_LEGACY_PAIRWISE (include/tpnet_b200.h)
N = 3000


def legacy_and_new(fn):
    """fn() under the legacy kernel, then under the default one: (legacy, new), each synchronised and copied."""
    lib = _lib.load()
    out = []
    for flags in (LEGACY, 0):
        old = lib.tpn_set_debug_flags(flags)
        try:
            r = fn()
            torch.cuda.synchronize()
            out.append(r.clone() if isinstance(r, torch.Tensor) else r)
        finally:
            lib.tpn_set_debug_flags(old)
    return out


def resident_tiles():
    """Tiles the resident warps of the pipelined kernel take at once at the bench shape (2 CTAs x 4 warps per SM)."""
    return torch.cuda.get_device_properties(0).multi_processor_count * 8


def pairs(rng, n, n_nodes):
    """Random pairs with runs of repeated b ids (the per-warp dedup), self pairs and the padding id 0."""
    a = rng.integers(0, n_nodes, n).astype(np.int64)
    b = rng.integers(0, n_nodes, n).astype(np.int64)
    runs = np.repeat(rng.integers(0, n_nodes, n // 8 + 1), 8)[:n]
    sel = rng.random(n) < 0.4
    b[sel] = runs[sel]
    b[:64] = a[:64]
    a[rng.random(n) < 0.05] = 0
    b[rng.random(n) < 0.05] = 0
    return a, b


def trained(L, dim, mode, seed=5):
    kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=2e-5, use_matrix=False,
              beginning_time=0.0, not_scale=False, enforce_dim=dim)
    o = WalkProjectionOracle(**kw)
    torch.manual_seed(0)                         # the head's weights: equal across modules of one test
    m = RandomProjectionModule(device=DEV, decay_mode=mode, **{k: v for k, v in kw.items() if k != 'beginning_time'},
                               beginning_time=np.float64(0.0))
    m.random_projections[0].data.copy_(torch.from_numpy(o.P[0]))
    m = m.to(DEV)
    rng = np.random.default_rng(seed)
    t = 0.0
    for _ in range(4):
        s = rng.integers(1, N, 1500).astype(np.int64)
        d = rng.integers(1, N, 1500).astype(np.int64)
        ts = np.sort(t + rng.random(1500) * 2000.0)
        t = ts[-1]
        o.update(s, d, ts)
        m.update(s, d, ts)
    return o, m


def check_oracle(o, got, a, b):
    ref = o.pair_wise_gram(a, b)
    o.not_scale = True
    raw = o.pair_wise_gram(a, b, exact=True)
    o.not_scale = False
    tol = 1e-5 * np.abs(ref) + 2e-6 * o.pair_norm_bound(a, b) / (1.0 + np.maximum(raw, 0)) + 1e-7
    assert np.all(np.abs(got - ref) <= tol), float(np.max(np.abs(got - ref) - tol))


def kernel_names(fn):
    """Names of the CUDA kernels fn() launches."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return ' '.join(e.name for e in prof.events())


@pytest.mark.parametrize('mode', ['eager', 'lazy'])
@pytest.mark.parametrize('L,dim', [(L, d) for L in (1, 2, 3, 4) for d in (64, 72, 120, 140, 210)
                                   if (L, d) != (4, 210)])      # 138 KB per CTA: neither staging kernel fits
def test_pipelined_equals_legacy(L, dim, mode):
    """Rows of 16, 18, 30, 36 and 54 float4 columns (chunks of odd and even widths), one tile past the small-call
    path, a few hundred tiles more than the resident warps, and a ragged tail."""
    o, m = trained(L, dim, mode)
    rng = np.random.default_rng(L * 1000 + dim)
    for n in (4097, 4 * (resident_tiles() + 300) + 3, 100_003):
        a, b = pairs(rng, n, N)
        if n == 4097:
            assert 'pairwise_pipe_kernel' in kernel_names(lambda: m.pair_wise_gram(a, b))
        old, new = legacy_and_new(lambda: m.pair_wise_gram(a, b))
        assert np.array_equal(old.cpu().numpy(), new.cpu().numpy()), n
        if n == 4097:
            check_oracle(o, new.cpu().numpy(), a, b)
        dev = [torch.from_numpy(x).to(DEV) for x in (a, b)]
        assert torch.equal(m.pair_wise_gram(*dev), new)
    m.check_errors()


def test_bench_shape_runs_the_pipelined_kernel():
    """At d = 210, L = 3 the default is pairwise_pipe_kernel and the debug flag selects pairwise_tma_kernel."""
    _, m = trained(3, 210, 'lazy')
    a, b = pairs(np.random.default_rng(1), 20_000, N)
    m.pair_wise_gram(a, b)
    torch.cuda.synchronize()
    names = []
    for flags in (0, LEGACY):
        old = _lib.load().tpn_set_debug_flags(flags)
        try:
            names.append(kernel_names(lambda: m.pair_wise_gram(a, b)))
        finally:
            _lib.load().tpn_set_debug_flags(old)
    assert 'pairwise_pipe_kernel' in names[0] and 'pairwise_tma_kernel' not in names[0]
    assert 'pairwise_tma_kernel' in names[1] and 'pairwise_pipe_kernel' not in names[1]


@pytest.mark.parametrize('mode', ['eager', 'lazy'])
def test_bad_device_id_sets_the_flag(mode):
    """An out-of-range device-resident id is clamped and flagged by both kernels, with the same features."""
    _, m = trained(3, 210, mode)
    a, b = pairs(np.random.default_rng(2), 50_001, N)
    b[30_007] = N + 5
    a[40_000] = -N - 9
    dev = [torch.from_numpy(x).to(DEV) for x in (a, b)]
    old, new = legacy_and_new(lambda: m.pair_wise_gram(*dev))
    assert torch.equal(old, new)
    with pytest.raises(IndexError):
        m.check_errors()
    m.check_errors()                             # the flag was cleared


@pytest.mark.parametrize('mode', ['eager', 'lazy'])
def test_device_count_below_capacity(mode):
    """Raw ABI call with a device-resident count n_dev < n: rows [0, n_dev) are the first n_dev pairs' features,
    later rows are not written; n_dev > n is flagged (code 4) and only n pairs are written."""
    _, m = trained(3, 210, mode)
    lib = _lib.load()
    n, k = 60_000, 37_771
    a, b = (torch.from_numpy(x).to(DEV) for x in pairs(np.random.default_rng(3), n, N))
    full = m.pair_wise_gram(a, b)
    st = m._c_state()
    stream = torch.cuda.current_stream().cuda_stream

    def call(count, cap):
        out = torch.full((cap, m.pair_wise_feature_dim), -7.0, device=DEV)
        nd = torch.tensor([count], dtype=torch.int32, device=DEV)
        assert lib.tpn_pairwise(st, a.data_ptr(), b.data_ptr(), cap, nd.data_ptr(), 1, out.data_ptr(), stream) == 0
        return out

    for got in legacy_and_new(lambda: call(k, n)):
        assert torch.equal(got[:k], full[:k])
        assert torch.all(got[k:] == -7.0)
    m.check_errors()
    for flags in (LEGACY, 0):
        old = lib.tpn_set_debug_flags(flags)
        try:
            got = call(n + 500, 50_000)
        finally:
            lib.tpn_set_debug_flags(old)
        assert torch.equal(got, full[:50_000])
        with pytest.raises(RuntimeError, match='more items'):
            m.check_errors()


@pytest.mark.parametrize('world', [1, 2])
def test_routed_calls(world):
    """Routed decoder pairs of the sharded state (device count <= launch capacity), in-process ranks."""
    from test_gpu_sharded_encoder import _each, _setup, _update_all
    ranks, streams, ref = _setup(world, 'lazy', N, 210, 3, False)
    rng = np.random.default_rng(world)
    s = rng.integers(1, N, 2000).astype(np.int64)
    d = rng.integers(1, N, 2000).astype(np.int64)
    ts = np.sort(rng.random(2000) * 500.0)
    _update_all(ranks, streams, s, d, ts)
    ref.update(s, d, ts)
    n = 30_001
    a, b = pairs(rng, n, N)

    def routed():
        parts = [r.trimmed() for r in _each(ranks, streams, lambda m: m.routed_pair_wise_gram(a, b))]
        got = torch.zeros(n, ref.pair_wise_feature_dim, device=DEV)
        for keep, feat in parts:
            got[keep] = feat
        return got

    old, new = legacy_and_new(routed)
    assert torch.equal(old, new)
    assert torch.allclose(new, ref.pair_wise_gram(a, b), rtol=1e-5, atol=2e-5)
    for m in ranks:
        m.check_errors()


def test_step_graph_capture_equals_eager():
    """StepGraphs (one CUDA graph per batch: both decoder calls of 6,000 pairs, then the update) replays the eager
    run's features and state."""
    from tpnet_b200.pipeline import EpochBatches, StepGraphs, tpnet_step

    rng = np.random.default_rng(4)
    src, dst = (1 + (rng.zipf(1.3, 24_000) - 1) % (N - 1) for _ in range(2))
    t = np.sort(rng.random(24_000) * 5000.0) + 1e4
    neg = rng.integers(1, N, len(src)).astype(np.int64)
    batches = EpochBatches(src, dst, t, 6_000, DEV, extra={'neg': neg})

    def make():
        _, m = trained(3, 210, 'lazy')
        return m

    m1 = make()
    with torch.no_grad():
        graphs = StepGraphs(m1, batches)
        replayed = [{k: v.clone() for k, v in graphs.replay(i).items()} for i in range(len(graphs))]
    m2 = make()
    out = {k: torch.empty_like(v) for k, v in graphs.out.items()}
    with torch.no_grad():
        for i, bt in enumerate(batches):
            tpnet_step(m2, bt, out)
            torch.cuda.synchronize()
            for k in out:
                assert torch.equal(out[k][:len(bt)], replayed[i][k][:len(bt)]), (i, k)
    m1.materialize()
    m2.materialize()
    for x, y in zip(m1.random_projections, m2.random_projections):
        assert torch.equal(x, y)
    m1.check_errors()
    m2.check_errors()
