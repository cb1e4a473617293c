"""GPU suite: P_0 from the counter-based generator (tpn_init_projection, ``p0_seed``) and the sharded reset of P_0.

- the kernel against the numpy restatement (oracle/p0_counter.py) through the raw C ABI, on hand-built layouts;
- the same bits at every placement: in-process sharded ranks (LocalPeerGroup) at worlds 1-4 against the plain module,
  at construction, after resets, and through updates and feature calls;
- the reset bookkeeping, a checkpoint re-sharded across world sizes, and the reset of the torch-RNG modes of the
  sharded class.
The real multi-process run is tests/dist_gpu_p0_check.py."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.p0_counter import p0_rows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = 'cuda:0'
SEED = 0xC0FFEE_1234_5678_9A          # above 2^63: the seed travels as a full uint64
TPN_ERR_INVALID_ARGUMENT = -1


# ---------------------------------------------------------------- in-process ranks (as in tests/test_gpu_sharded.py)
@pytest.fixture
def local_ranks():
    """Factory of in-process ranks on cuda:0: every rank connected; each rank has a stream.
    World 1 is the sharded class without peers (its whole graph is local)."""
    from tpnet_b200.peer import LocalPeerGroup
    from tpnet_b200.sharded import ShardedRandomProjection

    def make(world, kw, mode, ext_rows, torch_seed=11, **extra):
        groups = LocalPeerGroup.create(world)
        ranks = []
        for r in range(world):
            torch.manual_seed(torch_seed)          # as torchrun ranks are seeded: alike
            ranks.append(ShardedRandomProjection(decay_mode=mode, ext_rows=ext_rows, peers=groups[r],
                                                 exchange='peer' if world > 1 else 'auto', state_device=DEV,
                                                 **extra, **kw).to(DEV))
        for m in ranks:
            m.connect()
        return ranks, [torch.cuda.Stream() for _ in range(world)]
    return make


def _each(ranks, streams, fn):
    """One phase on every rank (each on its own stream), then a device-wide sync (LocalPeerGroup.host_barriers)."""
    out = []
    for m, s in zip(ranks, streams):
        with torch.cuda.stream(s):
            out.append(fn(m))
    torch.cuda.synchronize()
    return out


def _update_all(ranks, streams, s, d, ts):
    if len(ranks) == 1:
        ranks[0].update(s, d, ts)
        torch.cuda.synchronize()
        return
    pending = _each(ranks, streams, lambda m: m.update_begin(s, d, ts, None))
    for m, st, p in zip(ranks, streams, pending):
        with torch.cuda.stream(st):
            m.update_end(p)
    torch.cuda.synchronize()


def _global(ranks, layer, N):
    world = len(ranks)
    g = torch.full((N, ranks[0].dim), float('nan'), device=DEV)
    for r, m in enumerate(ranks):
        g[r::world] = m.random_projections[layer].data[:m.n_local]
    return g


def _kw(N, dim, L=3):
    return dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=1e-4, device=DEV,
                use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=dim)


def _plain(N, dim, mode, seed=SEED, L=3):
    from tpnet_b200 import RandomProjectionModule
    return RandomProjectionModule(decay_mode=mode, state_device=DEV, p0_seed=seed, **_kw(N, dim, L)).to(DEV)


def _assert_oracle(got, seed, draw, nodes, dim):
    want, amb = p0_rows(seed, draw, nodes, dim)
    got = np.asarray(got)
    bad = (got.view(np.uint32) != want.view(np.uint32)) & ~amb
    assert not bad.any(), (np.argwhere(bad)[:5], got[bad][:5], want[bad][:5])
    np.testing.assert_allclose(got[amb], want[amb], rtol=2e-7, atol=0)


# ---------------------------------------------------------------- the kernel against the oracle, raw C ABI
def _init(raw, rows, first, step, seed, draw):
    from tpnet_b200 import _lib
    rc = _lib.load().tpn_init_projection(ctypes.byref(raw.st), rows, first, step, seed, draw,
                                 torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize('d', [1, 3, 4, 5, 120, 210, 1000])
def test_kernel_matches_oracle(d):
    """row_stride = 4 mod 8, a padded node_stride with NaN in the gap, random layers 1..L: only columns [0, d) of
    layer 0 of rows < `rows` change, to the oracle's bits (the pad columns of the last block of 4 stay zero)."""
    from raw_state import RawState
    rng = np.random.default_rng(d)
    N, L = 41, 2
    rs = (d + 3) // 4 * 4 + (4 if ((d + 3) // 4 * 4) % 8 == 0 else 0)
    assert rs % 8 == 4 and rs >= d
    ns = (L + 1) * rs + 8
    cases = [(N, 0, 1, 0, 0), (N - 3, 2, 3, SEED, 1), (17, 10 ** 12 + 5, 7, 2 ** 64 - 1, 2 ** 40 + 3),
             (N, 1, 4, 12345, 2)]
    for rows, first, step, seed, draw in cases:
        raw = RawState(rng.standard_normal((N, L + 1, d)).astype(np.float32), rs, ns)
        assert _init(raw, rows, first, step, seed, draw) == 0
        host = raw.host()[0]
        before = raw.host0
        nodes = first + step * np.arange(rows, dtype=np.uint64)
        _assert_oracle(host[:rows, :d], seed, draw, nodes, d)
        assert np.all(host[:rows, d:rs] == 0)
        rest_now, rest_before = host.copy(), before.copy()
        rest_now[:rows, :d] = rest_before[:rows, :d] = 0          # everything but the written block: same bits
        assert np.array_equal(rest_now.view(np.uint32), rest_before.view(np.uint32)), (d, rows, first, step)


def test_kernel_invalid_arguments():
    """rows > num_nodes, node_step < 1, first_node < 0, rows < 0, a last node id past INT64_MAX: nothing written."""
    from raw_state import RawState
    raw = RawState(np.ones((9, 3, 5), np.float32), 12, 40)
    for rows, first, step in ((10, 0, 1), (9, 0, 0), (9, -1, 1), (-1, 0, 1), (9, 2 ** 62, 2 ** 60)):
        assert _init(raw, rows, first, step, 1, 0) == TPN_ERR_INVALID_ARGUMENT, (rows, first, step)
    assert np.array_equal(raw.host()[0].view(np.uint32), raw.host0.view(np.uint32))
    assert _init(raw, 0, 0, 1, 1, 0) == 0                              # nothing to write


# ---------------------------------------------------------------- the same bits at every placement
@pytest.mark.parametrize('mode', ['eager', 'lazy'])
def test_same_bits_at_every_world(local_ranks, mode):
    """P_0 gathered from worlds 1-4 == the plain module's (== the oracle) at construction and after one and two resets;
    then routed updates, encoder calls and row gathers stay bit-equal to the plain module."""
    N, dim, L = 997, 140, 3
    rng = np.random.default_rng(3)
    for world in (1, 2, 3, 4):
        ref = _plain(N, dim, mode)
        _assert_oracle(ref.random_projections[0].data.cpu().numpy(), SEED, 0, np.arange(N), dim)
        ranks, streams = local_ranks(world, _kw(N, dim, L), mode, 2 * N + 64, p0_seed=SEED)
        assert torch.equal(_global(ranks, 0, N), ref.random_projections[0].data), (world, 'construction')
        for k in (1, 2):
            _each(ranks, streams, lambda m: m.reset_random_projections())
            ref.reset_random_projections()
            torch.cuda.synchronize()
            assert all(m.p0_draw == k for m in ranks) and ref.p0_draw == k
            assert torch.equal(_global(ranks, 0, N), ref.random_projections[0].data), (world, 'reset', k)
        t = 0.0
        for B in (300, 4000):
            s = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
            d = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
            ts = np.sort(t + rng.random(B) * 500.0)
            t = ts[-1]
            _update_all(ranks, streams, s, d, ts)
            ref.update(s, d, ts)
            nbr = rng.integers(0, N, (101, 20)).astype(np.int64)
            src, dst = rng.integers(1, N, 101).astype(np.int64), rng.integers(1, N, 101).astype(np.int64)
            got = _assemble(_each(ranks, streams, lambda m: m.neighbor_pair_wise_gram(nbr, src, dst)), 101)
            want = ref.neighbor_pair_wise_gram(nbr, src, dst)
            torch.cuda.synchronize()
            assert torch.equal(got, want), (world, (got - want).abs().max().item())
            a, b = rng.integers(0, N, 501).astype(np.int64), rng.integers(0, N, 501).astype(np.int64)
            if world > 1:
                routed = _each(ranks, streams, lambda m: m.routed_pair_wise_gram(a, b))
                got = torch.zeros(501, ref.pair_wise_feature_dim, device=DEV)
                for r in routed:
                    keep, feat = r.trimmed()
                    got[keep] = feat
            else:
                got = ranks[0].pair_wise_gram(a, b)[1]
            assert torch.allclose(got, ref.pair_wise_gram(a, b), rtol=1e-5, atol=2e-5)
        _each(ranks, streams, lambda m: m.materialize())
        ref.materialize()
        for i in range(L + 1):
            assert torch.equal(_global(ranks, i, N), ref.random_projections[i].data), (world, mode, i)
        for m in ranks:
            m.check_errors()


def _assemble(parts, m):
    keep0, feat0 = parts[0]
    got = torch.zeros((m,) + tuple(feat0.shape[1:]), dtype=feat0.dtype, device=DEV)
    seen = torch.zeros(m, dtype=torch.int64, device=DEV)
    for keep, feat in parts:
        got[keep] = feat
        seen[keep] += 1
    assert torch.all(seen == 1)
    return got


# ---------------------------------------------------------------- reset bookkeeping
def test_reset_advances_draw_and_leaves_torch_rng_alone():
    N, dim = 513, 36
    m = _plain(N, dim, 'lazy', seed=77, L=2)
    rng = np.random.default_rng(0)
    s, d = rng.integers(1, N, 3000).astype(np.int64), rng.integers(1, N, 3000).astype(np.int64)
    m.update(s, d, np.sort(rng.random(3000) * 10.0))
    m.materialize()
    assert m.random_projections[1].data.abs().sum() > 0
    cpu, cuda = torch.get_rng_state(), torch.cuda.get_rng_state()
    for k in (1, 2, 3):
        m.reset_random_projections()
        assert m.p0_draw == k and m.p0_seed == 77
        torch.cuda.synchronize()
        _assert_oracle(m.random_projections[0].data.cpu().numpy(), 77, k, np.arange(N), dim)
        m.materialize()
        for i in (1, 2):
            assert torch.count_nonzero(m.random_projections[i].data) == 0
        assert float(m.now_time.item()) == 0.0
    assert torch.equal(torch.get_rng_state(), cpu) and torch.equal(torch.cuda.get_rng_state(), cuda)
    assert set(m.state_dict().keys()) == set(_plain_torch_keys(N, dim))       # no new state_dict entries


def _plain_torch_keys(N, dim):
    from tpnet_b200 import RandomProjectionModule
    return RandomProjectionModule(state_device=DEV, **_kw(N, dim, 2)).state_dict().keys()


# ---------------------------------------------------------------- checkpoint across world sizes
@pytest.mark.parametrize('mode', ['eager', 'lazy'])
def test_checkpoint_resumes_the_generator(local_ranks, tmp_path, mode):
    """Saved at world 2 after one reset, loaded at worlds 3 and 1 (modules built with another seed adopt the saved
    one), then reset: the uninterrupted job's P_0 of draw 2."""
    from tpnet_b200 import checkpoint as ck
    N, dim = 601, 36
    rng = np.random.default_rng(4)
    s, d = rng.integers(1, N, 2000).astype(np.int64), rng.integers(1, N, 2000).astype(np.int64)
    ts = np.sort(rng.random(2000) * 50.0)
    ranks, streams = local_ranks(2, _kw(N, dim), mode, 2 * N + 64, p0_seed=SEED)
    _each(ranks, streams, lambda m: m.reset_random_projections())
    _update_all(ranks, streams, s, d, ts)
    _each(ranks, streams, lambda m: ck.save_checkpoint(m, str(tmp_path), 'walk'))
    ref = _plain(N, dim, mode)
    for _ in range(2):
        ref.reset_random_projections()
    torch.cuda.synchronize()
    for world in (3, 1):
        if world == 1:
            new = [_plain(N, dim, mode, seed=5)]
            streams2 = [torch.cuda.Stream()]
        else:
            new, streams2 = local_ranks(world, _kw(N, dim), mode, 2 * N + 64, p0_seed=5)
        _each(new, streams2, lambda m: ck.load_checkpoint(m, str(tmp_path), 'walk'))
        assert all(m.p0_seed == SEED and m.p0_draw == 1 for m in new)
        _each(new, streams2, lambda m: m.reset_random_projections())
        got = new[0].random_projections[0].data if world == 1 else _global(new, 0, N)
        assert torch.equal(got, ref.random_projections[0].data), world
        assert all(m.p0_draw == 2 for m in new)


def test_checkpoint_header_records_the_generator(tmp_path):
    from tpnet_b200 import RandomProjectionModule
    from tpnet_b200 import checkpoint as ck
    m = _plain(101, 12, 'eager', seed=3)
    m.reset_random_projections()
    hdr = torch.load(ck.save_checkpoint(m, str(tmp_path), 'a'), weights_only=True)
    assert hdr['p0'] == {'seed': 3, 'draw': 1}
    plain = RandomProjectionModule(state_device=DEV, **_kw(101, 12)).to(DEV)
    hdr = torch.load(ck.save_checkpoint(plain, str(tmp_path), 'b'), weights_only=True)
    assert hdr['p0'] is None
    ck.load_checkpoint(plain, str(tmp_path), 'a')                       # a torch-RNG module keeps its mode
    assert plain.p0_seed is None and plain.p0_draw == 0


# ---------------------------------------------------------------- the sharded reset of the torch-RNG modes
@pytest.mark.parametrize('world', [2, 3])
def test_sharded_reset_global_equals_single_gpu(local_ranks, world):
    """p0='global', every rank re-seeded alike before its reset (as torchrun ranks are seeded): the gathered P_0 is
    the plain module's reset under the same seed, and the cache rows are not redrawn."""
    from tpnet_b200 import RandomProjectionModule
    N, dim = 403, 20
    ranks, streams = local_ranks(world, _kw(N, dim), 'eager', 64)
    torch.manual_seed(11)
    ref = RandomProjectionModule(decay_mode='eager', **_kw(N, dim)).to(DEV)
    assert torch.equal(_global(ranks, 0, N), ref.random_projections[0].data)
    ext = [m.random_projections[0].data[m.n_local:].clone() for m in ranks]

    def reset(m):
        torch.manual_seed(11)
        m.reset_random_projections()
    _each(ranks, streams, reset)
    torch.manual_seed(11)
    ref.reset_random_projections()
    torch.cuda.synchronize()
    assert torch.equal(_global(ranks, 0, N), ref.random_projections[0].data)
    for m, e in zip(ranks, ext):
        assert torch.equal(m.random_projections[0].data[m.n_local:], e)


@pytest.mark.parametrize('world', [2, 3])
def test_sharded_reset_device_draws_distinct_rows(local_ranks, world):
    """p0='device' (per-rank seeds), every rank re-seeded alike before its reset: no two nodes share a P_0 row, and
    the cache rows are not redrawn."""
    N, dim = 403, 20
    ranks, streams = local_ranks(world, _kw(N, dim), 'eager', 64, p0='device')
    _each(ranks, streams, lambda m: m.init_p0_on_device(5))
    ext = [m.random_projections[0].data[m.n_local:].clone() for m in ranks]

    def reset(m):
        torch.manual_seed(11)
        m.reset_random_projections()
    _each(ranks, streams, reset)
    full = _global(ranks, 0, N).cpu().numpy()
    assert np.isfinite(full).all()
    assert len(np.unique(full, axis=0)) == N
    for m, e in zip(ranks, ext):
        assert torch.equal(m.random_projections[0].data[m.n_local:], e)


# ---------------------------------------------------------------- real ranks
@pytest.mark.parametrize('world', [2, 8])
def test_p0_equal_across_worlds_real_ranks(world):
    """One process per GPU (torchrun): tests/dist_gpu_p0_check.py."""
    if torch.cuda.device_count() < world:
        pytest.skip(f'needs >= {world} GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world),
           '--master-addr', '127.0.0.1', '--master-port', str(29567 + world),
           os.path.join(ROOT, 'tests', 'dist_gpu_p0_check.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'PASS' in r.stdout
