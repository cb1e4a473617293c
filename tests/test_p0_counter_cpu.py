"""CPU suite: the numpy restatement of the counter-based P_0 (oracle/p0_counter.py, tpn_init_projection in
include/tpnet_b200.h).  Its Philox equals numpy's own np.random.Philox, and the values it defines are N(0, 1/sqrt(d)),
with no correlation between neighbouring nodes, columns or draws and no repeated rows."""
import math

import numpy as np
import pytest
from scipy import stats

from oracle.p0_counter import normals, p0_rows, philox4x64_10


def _numpy_philox(ctr, key):
    """numpy's Philox increments its 256-bit counter before each block: start it one below the wanted counter (for
    c0 = 0 the borrow runs into the higher words)."""
    c = sum(int(ctr[i]) << (64 * i) for i in range(4))
    k = int(key[0]) | (int(key[1]) << 64)
    return np.random.Philox(counter=(c - 1) % (1 << 256), key=k).random_raw(4)


def _u64(rng, shape):
    return rng.integers(0, 1 << 63, shape, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, shape, dtype=np.uint64)


def test_philox_equals_numpy():
    rng = np.random.default_rng(1)
    ctr = _u64(rng, (400, 4))
    key = _u64(rng, (400, 2))
    ctr[:100, 0] = 0                      # borrow into word 1
    ctr[:50, 1] = 0                       # ... and on into word 2
    ctr[100:130, :2] = [0, 7]             # the counters tpn_init_projection uses: (block, node, 0, 0)
    ctr[100:130, 2:] = 0
    key[:20] = 0
    ctr[200:210] = np.uint64((1 << 64) - 1)
    got = philox4x64_10(ctr, key)
    for i in range(len(ctr)):
        assert np.array_equal(got[i], _numpy_philox(ctr[i], key[i])), i


@pytest.mark.parametrize('dim', [210, 5])
def test_values_are_normal(dim):
    nodes = np.arange(3, 3 + (1_050_000 // dim) + 1) * 7
    x = p0_rows(20261022, 2, nodes, dim)[0].astype(np.float64).reshape(-1)
    n = x.size
    assert n >= 1_000_000
    std = 1 / math.sqrt(dim)
    assert abs(x.mean()) < 5 * std / math.sqrt(n)
    assert abs(x.var() / std ** 2 - 1) < 5 * math.sqrt(2 / n)
    assert stats.kstest(x, stats.norm(loc=0, scale=std).cdf).pvalue > 1e-3
    z = normals(20261022, 2, nodes[:2000], dim).reshape(-1)
    assert stats.kstest(z, stats.norm().cdf).pvalue > 1e-3


def _corr(a, b):
    return float(np.corrcoef(a.reshape(-1), b.reshape(-1))[0, 1])


def test_neighbours_uncorrelated():
    d = 64
    n = 20_000
    z = normals(5, 0, np.arange(n + 1), d)
    bound = 5 / math.sqrt(n * (d - 4))
    assert abs(_corr(z[:-1], z[1:])) < 5 / math.sqrt(n * d)                 # node u vs u + 1
    for lag in (1, 2, 3, 4):                                               # inside and across a block of 4
        assert abs(_corr(z[:, :-lag], z[:, lag:])) < bound, lag
    z1 = normals(5, 1, np.arange(n + 1), d)
    assert abs(_corr(z, z1)) < 5 / math.sqrt((n + 1) * d)                   # draw k vs k + 1
    s1 = normals(6, 0, np.arange(n + 1), d)
    assert abs(_corr(z, s1)) < 5 / math.sqrt((n + 1) * d)                   # seed s vs s + 1
    # the squares too: Box-Muller pairs share r
    sq = z ** 2
    assert abs(_corr(sq[:, 0::4], sq[:, 1::4])) < 5 / math.sqrt(n * d / 4)


def test_no_equal_rows():
    f = p0_rows(0, 0, np.arange(100_000), 4)[0]
    assert len(np.unique(f, axis=0)) == len(f)


def test_midpoint_mask_is_rare():
    """The entries the GPU suite exempts from bit equality: about 1e-7 of them."""
    amb = p0_rows(9, 3, np.arange(50_000), 21)[1]
    assert amb.sum() < 10


def _kw(**over):
    kw = dict(node_num=50, edge_num=500, dim_factor=1, num_layer=2, time_decay_weight=1e-4, device='cuda:0',
              use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=8)
    kw.update(over)
    return kw


@pytest.mark.parametrize('case', ['use_matrix', 'init_p0_false', 'no_state_device', 'cpu_state', 'seed_range',
                                  'negative_seed', 'sharded_p0_device'])
def test_p0_seed_refusals(case):
    """p0_seed is refused where there is nothing to draw, where the caller fills P_0, off the GPU (there is no CPU
    path), outside [0, 2^64), and with the sharded class's other P_0 modes.  All before any CUDA call."""
    from tpnet_b200 import RandomProjectionModule
    from tpnet_b200.sharded import ShardedRandomProjection
    args = {'use_matrix': dict(use_matrix=True, state_device='cuda:0'),
            'init_p0_false': dict(init_p0=False, state_device='cuda:0'),
            'no_state_device': dict(),
            'cpu_state': dict(state_device='cpu'),
            'seed_range': dict(state_device='cuda:0'),
            'negative_seed': dict(state_device='cuda:0')}
    seed = {'seed_range': 1 << 64, 'negative_seed': -1}.get(case, 3)
    with pytest.raises(ValueError):
        if case == 'sharded_p0_device':
            ShardedRandomProjection(p0='device', state_device='cuda:0', p0_seed=3, **_kw())
        else:
            RandomProjectionModule(p0_seed=seed, **_kw(**args[case]))
