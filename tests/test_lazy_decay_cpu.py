"""CPU checks of oracle/lazy_decay.py, the restatement of the library's lazy decay that the GPU suite holds the kernels
to bit for bit (tests/test_gpu_update_lazy.py): it must be the eager chain whenever at most one update was skipped,
stay within the float64 anchor's error bound on long gaps, and keep the log rules.
"""
import numpy as np
import pytest

from oracle.lazy_decay import LOG_FULL, LazyDecayModel, anchor_bound
from oracle.walk_projection import WalkProjectionOracle, decay_factors

FACTOR_SET = np.float32([0.5, 0.37, 0.81, 0.62, 0.9])


def make_state(rng, N, L, d, rs, ns, epoch, stamps, scale=1.0):
    rows = (rng.standard_normal((N, L + 1, d)) * scale / np.sqrt(d)).astype(np.float32)
    data = np.full((N + 1, ns), np.nan, np.float32)
    blk = data[:N, :(L + 1) * rs].reshape(N, L + 1, rs)
    blk[:] = 0
    blk[:, :, :d] = rows
    for l in range(1, L + 1):
        blk[stamps[:, l - 1] < 0, l, :] = 0
    factors = rng.choice(FACTOR_SET, size=(epoch, L))
    return LazyDecayModel(data, N, L, d, rs, ns, stamps=stamps, factors=factors, log_capacity=epoch + 40)


def edges(rng, N, B, hub=None):
    src = rng.integers(0, N, B)
    dst = rng.integers(0, N, B)
    if hub is not None:
        dst[rng.random(B) < 0.6] = hub
    t = np.sort(rng.random(B) * 2000.0) + 10_000.0
    return src.astype(np.int64), dst.astype(np.int64), t


def eager_oracle(model, lam, now):
    """WalkProjectionOracle over the model's CURRENT rows (full row_stride, pad columns included)."""
    o = WalkProjectionOracle.__new__(WalkProjectionOracle)
    o.node_num, o.num_layer, o.time_decay_weight = model.N, model.L, lam
    o.now_time = np.float64(now)
    o.P = [model.current_layer(l) for l in range(model.L + 1)]
    return o


@pytest.mark.parametrize('L', [1, 2, 3, 4])
@pytest.mark.parametrize('B,chunk', [(300, 0), (3000, 0), (3000, 256)])
def test_one_skipped_epoch_is_the_eager_chain(L, B, chunk):
    """Every stamp at the epoch before the call (or -1 on a zero row): the update and a materialize afterwards give
    the eager chain's state bit for bit — the header's "identical for epoch - s <= 1"."""
    rng = np.random.default_rng(L * 100 + B + chunk)
    N, d, rs = 120, 13, 16
    e = 9
    stamps = np.full((N, L), e, np.int32)
    stamps[rng.random((N, L)) < 0.1] = -1
    m = make_state(rng, N, L, d, rs, (L + 1) * rs + 4, e, stamps)
    m.giant_chunk = chunk
    src, dst, t = edges(rng, N, B, hub=5)
    lam = 4e-4
    now = t[-1] - 1500.0                                    # lambda * dt = 0.6
    o = eager_oracle(m, lam, now)
    decay = decay_factors(lam, t[-1], now, L)
    assert decay.min() < 0.6
    assert m.update(src, dst, t, lam, decay) == 0
    o.update(src, dst, t, giant_chunk=chunk if 2 * B > 4096 else 0)
    m.materialize()
    for l in range(L + 1):
        assert np.array_equal(m.rows()[:, l, :].view(np.int32), o.P[l].view(np.int32)), l


@pytest.mark.parametrize('L', [1, 3])
def test_frozen_clock_is_the_eager_chain(L):
    """decay == NULL: no epoch is logged, lagging stamps keep their pending factor, and a sequence of updates equals
    the eager chain run on the current rows with a clock that does not move."""
    rng = np.random.default_rng(L)
    N, d, rs, e = 90, 20, 20, 30
    stamps = rng.integers(-1, e + 1, (N, L)).astype(np.int32)
    m = make_state(rng, N, L, d, rs, (L + 1) * rs, e, stamps)
    lam = 1e-3
    src, dst, t = edges(rng, N, 400)
    o = eager_oracle(m, lam, t[-1])
    for _ in range(4):
        src, dst, t = edges(rng, N, 400)
        t = t - t[-1] + o.now_time                           # same t_last: every factor is 1
        assert m.update(src, dst, t, lam, None) == 0
        o.update(src, dst, t)
        assert m.epoch == e
    for l in range(L + 1):
        assert np.array_equal(m.current_layer(l).view(np.int32), o.P[l].view(np.int32))


def test_log_quotient_gives_back_the_factor():
    """fl32(f64(Q * c) / Q) == c for fp32 c in (0, 1] (subnormal c included) and Q in [1e-200, 1]: the factor a row
    stamped one epoch back reads is exactly this call's c."""
    rng = np.random.default_rng(3)
    n = 4_000_000
    c = rng.integers(1, 0x3f800001, n, dtype=np.int64).astype(np.uint32).view(np.float32)
    c[:20_000] = rng.integers(1, 0x800000, 20_000, dtype=np.int64).astype(np.uint32).view(np.float32)   # subnormal
    q = 10.0 ** -rng.uniform(0, 200, n)
    q[:1000] = 1e-200
    got = ((q * c.astype(np.float64)) / q).astype(np.float32)
    assert np.array_equal(got.view(np.uint32), c.view(np.uint32))


@pytest.mark.parametrize('L', [2, 4])
def test_long_gaps_within_the_anchor_bound(L):
    """Hundreds of skipped epochs (factors 0.37..0.9, rows that decay into the subnormal range and to zero), then
    updates with c far from 1: every target row stays within the derived bound of the float64 anchor."""
    rng = np.random.default_rng(L + 40)
    N, d, rs, e = 200, 30, 32, 300
    stamps = rng.integers(-1, e + 1, (N, L)).astype(np.int32)
    stamps[rng.random((N, L)) < 0.3] = e
    stamps[:20] = rng.integers(0, 5, (20, L))
    m = make_state(rng, N, L, d, rs, (L + 1) * rs, e, stamps, scale=4.0)
    lam = 5e-4
    now = 0.0
    for B in (200, 2500, 3000):
        src, dst, t = edges(rng, N, B, hub=7)
        t = t - t[-1] + now + 1400.0
        decay = decay_factors(lam, t[-1], now, L)
        gap = m.epoch + 1 - int(m.stamps[m.stamps >= 0].min())
        X = float(np.nanmax(np.abs(m.rows())))
        rc, (R, A, cnt) = m.update(src, dst, t, lam, decay, anchor=True)
        assert rc == 0
        now = t[-1]
        tg = np.unique(np.concatenate([src, dst]))
        for l in range(1, L + 1):
            got = m.rows()[tg, l, :].astype(np.float64)
            tol = anchor_bound(A[l - 1][tg], cnt[tg][:, None], gap, X)
            assert np.all(np.abs(got - R[l - 1][tg]) <= tol), l
        assert np.abs(R).max() > 0


def test_log_full_rules_change_nothing():
    rng = np.random.default_rng(5)
    N, L, d, rs, e = 40, 3, 8, 8, 6
    m = make_state(rng, N, L, d, rs, (L + 1) * rs, e, rng.integers(-1, e + 1, (N, L)).astype(np.int32))
    m.Q = m.Q[:e + 1].copy()                                # capacity exhausted
    src, dst, t = edges(rng, N, 50)
    decay = np.float32([0.5, 0.25, 0.125])
    before = (m.data.copy(), m.stamps.copy(), m.Q.copy(), m.epoch, m.cum_floor)
    assert m.update(src, dst, t, 1e-3, decay) == LOG_FULL
    after = (m.data, m.stamps, m.Q, m.epoch, m.cum_floor)
    assert all(np.array_equal(np.atleast_1d(x).view(np.uint8), np.atleast_1d(y).view(np.uint8))
               for x, y in zip(before, after))
    assert m.update(src, dst, t, 1e-3, None) == 0 and m.epoch == e          # no clock move: no epoch needed
    m2 = make_state(rng, N, L, d, rs, (L + 1) * rs, e, rng.integers(-1, e + 1, (N, L)).astype(np.int32))
    m2.cum_floor = 5e-200
    assert m2.update(src, dst, t, 1e-3, decay) == LOG_FULL                 # floor * 0.125 < 1e-200
    assert m2.update(src, dst, t, 1e-3, np.float32([0.5, 0.5, 0.5])) == 0  # floor * 0.5 >= 1e-200
    m2.materialize()
    m2.reset_epoch()
    assert m2.epoch == 0 and m2.cum_floor == 1.0
    assert m2.update(src, dst, t, 1e-3, np.float32([1e-30, 1e-30, 1e-30])) == 0   # epoch 0: the floor restarts


def test_restart_keeps_current_values():
    """materialize, then reset_epoch: the same current values (gather) and the same blocks; stamp -1 rows stay -1."""
    rng = np.random.default_rng(6)
    N, L, d, rs, e = 80, 3, 11, 12, 5
    m = make_state(rng, N, L, d, rs, (L + 1) * rs + 8, e, rng.integers(-1, e + 1, (N, L)).astype(np.int32))
    lam, now = 3e-4, 0.0
    for B in (100, 2100):
        src, dst, t = edges(rng, N, B)
        t = t - t[-1] + now + 1000.0
        assert m.update(src, dst, t, lam, decay_factors(lam, t[-1], now, L)) == 0
        now = t[-1]
    ids = np.arange(-N, N)
    want, blocks = m.gather(ids), m.gather_blocks(ids)
    dead = m.stamps < 0
    m.materialize()
    assert np.all(m.stamps[~dead] == m.epoch) and np.all(m.stamps[dead] == -1)
    m.reset_epoch()
    assert np.all(m.stamps[~dead] == 0) and np.all(m.stamps[dead] == -1) and m.epoch == 0
    assert np.array_equal(m.gather(ids).view(np.int32), want.view(np.int32))
    assert np.array_equal(m.gather_blocks(ids).view(np.int32), blocks.view(np.int32))
