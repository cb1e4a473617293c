"""GPU suite: the lazy-decay update and its readers, bit for bit, on hand-built raw-ABI states and on every walk path.

The kernels are held to oracle/lazy_decay.py (the restatement of the one-multiply rule: a row of layer l last written
at epoch s is read at epoch e as fl32(x * fl32(Q[e][l-1] / Q[s][l-1])), division in f64) bit for bit: the whole data
buffer (every node's rows 0..L, the pad columns, the NaN node_stride gap and the NaN node past num_nodes), the stamps,
the log, epoch and cum_floor after every call.  States have stamps drawn per node AND per layer (many one epoch back,
some current, some more than 100 epochs back, some -1 on zero rows), per-epoch factors from {0.5, 0.37, 0.81, 0.62,
0.9}, this call's factors far from 1 (lambda * dt in 0.3..1) and weights over [e^-2, 1].

Independently of the restatement, every target row is held to the float64 anchor (LazyDecayModel.chain64), which
keeps the list of fp32 factors per epoch instead of Q: the true value of a row of m messages is
    R = T + sum_j S_j w_j,   T = x_t * prod_{k=s_t+1..e} c_k,   S_j = x_j * prod_{k=s_j+1..e} c_k
(T: the target brought current, S_j: the current source rows, w_j the fp32 weights).  The kernel computes
fl(fl(x_t * f_t) + sum_j fl(fl(x_j * f_j) * w_j)) with f = fl32(Q[e] / Q[s]): every source term goes through at most
three roundings before the sum (the factor, the rescale, the product with w) and the target through two, and the
m adds of a sequential or chunked sum add at most m more to any term, so in any summation order
    |got - R| <= (gamma_{m+3} + eta) * (|T| + sum_j |S_j w_j|) + (m + 1) (X + 2) 2^-149,   gamma_k = k u / (1 - k u)
with u = 2^-24.  eta = (2 K + m + 4) 2^-52 covers the f64 roundings of the log's products and quotient and of the
anchor itself (K: the longest gap); the last term covers gradual underflow — a rounding into the subnormal range
errs by at most 2^-150 absolutely, once in the factor (scaled by |x| <= X, the largest stored value) and once in
each product, on each of the m + 1 terms.
"""
import contextlib
import zlib

import numpy as np
import pytest
import torch

import tpnet_b200.random_projection as rpmod
from oracle.lazy_decay import LazyDecayModel, anchor_bound
from oracle.walk_projection import decay_factors
from raw_state import DEV, RawState
from tpnet_b200 import RandomProjectionModule, _lib

pytestmark = pytest.mark.gpu

PER_LAYER, SERIAL, SNAP_P0, LEGACY_FRONT, NO_STREAM, STREAM_ALL = 1, 2, 4, 16, 32, 64
LOG_FULL = _lib.TPN_ERR_LOG_FULL
EPOCH = 150                                      # epochs already logged in a hand-built lazy state


@contextlib.contextmanager
def debug_flags(flags):
    lib = _lib.load()
    old = lib.tpn_set_debug_flags(int(flags))
    try:
        yield
    finally:
        lib.tpn_set_debug_flags(old)


# --------------------------------------------------------------------------- states and batches
def draw_stamps(rng, N, L, e):
    """Per node and per layer: 30 % current (e), 25 % one back, 10 % more than 100 back, 10 % never written (-1),
    the rest anywhere in [0, e]."""
    u = rng.random((N, L))
    s = rng.integers(0, e + 1, (N, L))
    s[u < 0.30] = e
    s[(u >= 0.30) & (u < 0.55)] = e - 1
    lag = (u >= 0.55) & (u < 0.65)
    s[lag] = rng.integers(0, e - 100, int(lag.sum()))
    s[(u >= 0.65) & (u < 0.75)] = -1
    return s.astype(np.int32)


def make_state(seed, N, L, d, rs, ns, lazy, chunk=0, capacity=None):
    rng = np.random.default_rng(seed)
    rows = (rng.standard_normal((N, L + 1, d)) / np.sqrt(d)).astype(np.float32)
    if not lazy:
        st = RawState(rows, rs, ns, giant_chunk=chunk)
    else:
        factors = rng.choice(np.float32([0.5, 0.37, 0.81, 0.62, 0.9]), size=(EPOCH, L))
        st = RawState(rows, rs, ns, stamps=draw_stamps(rng, N, L, EPOCH), factors=factors,
                      log_capacity=EPOCH + 8 if capacity is None else capacity, giant_chunk=chunk)
    return st, LazyDecayModel(**st.model_args()), rng


def times_for(rng, B, lam, t_last):
    """Sorted timestamps ending at t_last with lambda * (t_last - t) in [0, 2]: weights over [e^-2, 1]."""
    t = np.sort(t_last - rng.random(B) * 2.0 / lam)
    t[-1] = t_last
    return t


def clock(rng, lam, L, t_last, frozen=False):
    """This call's factors: lambda * dt in [0.3, 1] (c_L down to ~0.02), or None for a clock that did not move."""
    if frozen:
        return None
    return decay_factors(lam, t_last, t_last - rng.uniform(0.3, 1.0) / lam, L)


def designed_batch(rng, N, hubs):
    """Edges whose targets have the given message counts: hubs = [(node, count)], each as the dst of `count` edges
    from random sources, then one random edge per 4 nodes; shuffled."""
    src, dst = [], []
    for node, cnt in hubs:
        src.append(rng.integers(0, N, cnt))
        dst.append(np.full(cnt, node))
    src.append(rng.integers(0, N, N // 4 + 1))
    dst.append(rng.integers(0, N, N // 4 + 1))
    src, dst = np.concatenate(src).astype(np.int64), np.concatenate(dst).astype(np.int64)
    p = rng.permutation(len(src))
    return src[p], dst[p]


def walker_hubs(rng):
    """Segments for every large-batch walker: 1..63 (walk_small_kernel), 64..2047 (hub2 regular), >= 2048 (hub2
    giants) and one target with more than a quarter of the messages (walk_stream_kernel)."""
    hubs = [(1, 24_000), (2, 2100), (3, 2600), (4, 3000)]
    hubs += [(n, int(c)) for n, c in zip(range(5, 15), rng.integers(64, 600, 10))] + [(15, 2047)]
    hubs += [(n, int(c)) for n, c in zip(range(40, 200), rng.integers(5, 63, 160))]
    return hubs


# --------------------------------------------------------------------------- assertions
def same_bits(got, want, what):
    g, w = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    gb, wb = g.view(np.uint8).reshape(g.shape[0], -1), w.view(np.uint8).reshape(w.shape[0], -1)
    bad = np.nonzero(np.any(gb != wb, axis=1))[0]
    assert bad.size == 0, f'{what}: {bad.size} rows differ, first {bad[:8].tolist()}'


def check_state(st, model, anchor=None):
    data, stamps, log, epoch, floor, err = st.host()
    assert err == 0, err
    same_bits(data, model.data, 'data')
    if model.lazy:
        same_bits(stamps, model.stamps, 'stamps')
        same_bits(log, model.Q, 'decay log')
        assert epoch == model.epoch and floor == model.cum_floor, (epoch, model.epoch, floor, model.cum_floor)
    if anchor is not None:
        (R, A, cnt), gap, X = anchor
        tg = np.nonzero(cnt)[0]
        got = data[:st.N, :(st.L + 1) * st.rs].reshape(st.N, st.L + 1, st.rs)
        for l in range(1, st.L + 1):
            err = np.abs(got[tg, l, :].astype(np.float64) - R[l - 1][tg])
            tol = anchor_bound(A[l - 1][tg], cnt[tg][:, None], gap, X)
            assert np.all(err <= tol), (l, float(np.max(err - tol)))


def anchor_inputs(model):
    live = model.stamps[model.stamps >= 0]
    gap = model.epoch + 1 - (int(live.min()) if live.size else model.epoch)
    return gap, float(np.nanmax(np.abs(model.rows())))


def run_update(st, model, src, dst, t, lam, decay, flags=0):
    """One tpn_update against the model; returns the code."""
    anchor = model.lazy and decay is not None
    gap, X = anchor_inputs(model) if anchor else (0, 0.0)
    with debug_flags(flags):
        rc = st.update(src, dst, t, lam, decay)
    out = model.update(src, dst, t, lam, decay, flags=flags, anchor=anchor)
    want, res = out if anchor else (out, None)
    assert rc == want, (rc, want)
    check_state(st, model, (res, gap, X) if res is not None else None)
    return rc


# --------------------------------------------------------------------------- the paths
# (id, N, L, d, rs, ns, batch, flags, giant_chunk).  batch: 'small-rank' / 'small-bitonic' (single-CTA sort), 'walkers'
# (every large-batch walker), 'uniform' (short segments only), 'giants' (more than 2,048 giant rows in one call).
CASES = [
    ('small-rank-L1', 300, 1, 210, 212, 2 * 212 + 8, 'small-rank', 0, 0),
    ('small-rank-L4', 200, 4, 30, 32, 5 * 32, 'small-rank', 0, 0),
    ('small-bitonic-L2', 500, 2, 37, 40, 3 * 40 + 4, 'small-bitonic', 0, 0),
    ('small-bitonic-L3', 400, 3, 210, 212, 4 * 212 + 8, 'small-bitonic', 0, 0),
    ('walkers-1pass', 250, 2, 20, 20, 3 * 20 + 4, 'walkers', 0, 0),
    ('walkers-2pass', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', 0, 0),
    ('walkers-3pass', 70_000, 4, 12, 12, 5 * 12 + 4, 'walkers', 0, 0),
    ('no-stream', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', NO_STREAM, 0),
    ('stream-all', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', STREAM_ALL, 0),
    ('serial-walk', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', SERIAL, 0),
    ('snapshot-p0', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', SNAP_P0, 0),
    ('legacy-front', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', LEGACY_FRONT, 0),
    ('per-layer', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', PER_LAYER, 0),
    ('per-layer-tiles', 3000, 2, 1000, 1000, 3 * 1000 + 4, 'uniform', PER_LAYER, 0),
    ('chunk-256', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', 0, 256),
    ('chunk-2048', 5000, 2, 64, 64, 3 * 64, 'walkers', 0, 2048),
    ('chunk-per-layer', 5000, 3, 210, 212, 4 * 212 + 8, 'walkers', PER_LAYER, 256),
    ('giants-2100', 2100, 2, 16, 16, 3 * 16 + 4, 'giants', 0, 0),
    ('giants-2100-chunk', 2100, 2, 16, 16, 3 * 16 + 4, 'giants', 0, 256),
]


def batch_for(kind, rng, N):
    if kind == 'small-rank':
        s, d = designed_batch(rng, N, [(3, 100), (4, 40)])                          # 2B <= 1,024
        assert 2 * len(s) <= 1024
        return s, d
    if kind == 'small-bitonic':
        s, d = designed_batch(rng, N, [(3, 900), (4, 300), (5, 64)])                # 1,024 < 2B <= 4,096
        assert 1024 < 2 * len(s) <= 4096
        return s, d
    if kind == 'walkers':
        return designed_batch(rng, N, walker_hubs(rng))
    if kind == 'uniform':
        s = rng.integers(0, N, 6000)
        return s.astype(np.int64), rng.integers(0, N, 6000).astype(np.int64)
    if kind == 'giants':
        B = 2_200_000                  # every node receives ~2,095 >= 2,048 messages: 2,100 giants in one call
        j = np.arange(B, dtype=np.int64)
        return j % N, (j * 11 + 3) % N
    raise ValueError(kind)


def edge_arrays(kind, rng, N):
    return batch_for(kind, rng, N)


# the frozen clock adds nothing to the giant-list fallback that the lazy and eager modes run
PATH_PARAMS = [pytest.param(*c, mode, id=f'{c[0]}-{mode}') for c in CASES for mode in ('lazy', 'frozen', 'eager')
               if not (c[6] == 'giants' and mode == 'frozen')]


@pytest.mark.parametrize('name,N,L,d,rs,ns,kind,flags,chunk,mode', PATH_PARAMS)
def test_update_paths(name, N, L, d, rs, ns, kind, flags, chunk, mode):
    """Two updates per path (the second reads the rows the first wrote), bit for bit against the model, every
    target row within the anchor's bound; 'frozen': decay == NULL while stamps lag; 'eager': stamps == NULL."""
    lazy = mode != 'eager'
    st, model, rng = make_state(zlib.crc32(name.encode()), N, L, d, rs, ns, lazy, chunk)
    lam = 1e-3
    t_last = 5.0e4
    for _ in range(2):
        src, dst = edge_arrays(kind, rng, N)
        t = times_for(rng, len(src), lam, t_last)
        decay = clock(rng, lam, L, t_last, frozen=mode == 'frozen')
        assert run_update(st, model, src, dst, t, lam, decay, flags) == 0
        t_last += 700.0


def test_stream_and_giant_paths_are_reached():
    """The designed batches really have what the cases above are named for."""
    rng = np.random.default_rng(0)
    src, dst = edge_arrays('walkers', rng, 5000)
    cnt = np.bincount(np.concatenate([src, dst]))
    E = 2 * len(src)
    assert cnt.max() * 4 > E
    assert ((cnt >= 2048) & (cnt * 4 <= E)).sum() >= 3
    assert ((cnt >= 64) & (cnt < 2048)).sum() >= 10 and ((cnt > 0) & (cnt < 64)).sum() >= 1000
    src, dst = edge_arrays('giants', rng, 2100)
    cnt = np.bincount(np.concatenate([src, dst]))
    assert (cnt >= 2048).sum() > 2048 and (2 * len(src)) // 2048 + 2 > 2048


# --------------------------------------------------------------------------- split call
@pytest.mark.parametrize('mode', ['lazy', 'eager'])
def test_split_call(mode):
    """tpn_update_phase PREPARE on a second stream, then APPLY: the bits of the whole call; after PREPARE alone the
    data and stamps are unchanged and the epoch has not moved."""
    lazy = mode == 'lazy'
    st, model, rng = make_state(11, 5000, 3, 210, 212, 4 * 212 + 8, lazy)
    lam, t_last = 1e-3, 9.0e4
    side = torch.cuda.Stream()
    for _ in range(2):
        src, dst = edge_arrays('walkers', rng, st.N)
        t = times_for(rng, len(src), lam, t_last)
        decay = clock(rng, lam, st.L, t_last)
        before = st.host()
        keep = []
        torch.cuda.synchronize()
        assert st.update(src, dst, t, lam, decay, phase=_lib.UPDATE_PREPARE, stream=side.cuda_stream, keep=keep) == 0
        mid = st.host()
        same_bits(mid[0], before[0], 'data after PREPARE')
        if lazy:
            same_bits(mid[1], before[1], 'stamps after PREPARE')
        assert mid[3] == before[3] and mid[4] == before[4]
        gap, X = anchor_inputs(model) if lazy else (0, 0.0)
        assert st.update(src, dst, t, lam, decay, phase=_lib.UPDATE_APPLY) == 0
        out = model.update(src, dst, t, lam, decay, anchor=lazy)
        rc, res = out if lazy else (out, None)
        assert rc == 0
        check_state(st, model, (res, gap, X) if lazy else None)
        t_last += 500.0


# --------------------------------------------------------------------------- message mode
def message_batch(rng, n_local, n_ext, kind):
    """Messages of a shard: both directions of edges among local rows, plus messages from received rows
    (rows >= n_local) to local targets, shuffled.  'large': one target holds > 1/4 of the messages, giants, regular
    hubs and short segments all read received rows."""
    B = 1200 if kind == 'small' else 15_000
    a, b = rng.integers(0, n_local, B), rng.integers(0, n_local, B)
    tgt, src = [np.concatenate([a, b])], [np.concatenate([b, a])]
    counts = [(7, 300), (8, 60)] if kind == 'small' else [(7, 35_000), (8, 2500), (9, 3000)] + \
        [(n, int(c)) for n, c in zip(range(10, 40), rng.integers(64, 2048, 30))]
    for node, c in counts:
        tgt.append(np.full(c, node))
        src.append(rng.integers(n_local, n_local + n_ext, c))
    few = rng.integers(0, n_local, 400)
    tgt.append(few)
    src.append(rng.integers(n_local, n_local + n_ext, 400))
    tgt, src = np.concatenate(tgt).astype(np.int64), np.concatenate(src).astype(np.int64)
    p = rng.permutation(len(tgt))
    return tgt[p], src[p]


# the debug flags select large-batch paths only
MESSAGE_PARAMS = [pytest.param(kind, flags, mode, id=f'{mode}-{kind}-{flags}') for mode in ('lazy', 'eager')
                  for kind, flags in (('small', 0), ('large', 0), ('large', STREAM_ALL), ('large', PER_LAYER))]


@pytest.mark.parametrize('kind,flags,mode', MESSAGE_PARAMS)
def test_update_messages(kind, flags, mode):
    """tpn_update_messages with received rows whose stamps lag, in a shuffled order; the large calls pass the count
    on the device, below the capacity (the messages past it must not be applied)."""
    lazy = mode == 'lazy'
    n_local, n_ext = 3000, 700
    N = n_local + n_ext
    st, model, rng = make_state(31 + flags + (kind == 'large'), N, 3, 210, 212, 4 * 212 + 8, lazy)
    lam, t_last = 1e-3, 3.0e4
    for _ in range(2):
        tgt, src = message_batch(rng, n_local, n_ext, kind)
        t = t_last - rng.random(len(tgt)) * 2.0 / lam
        count = None
        if kind == 'large':
            count = len(tgt)
            tgt = np.concatenate([tgt, np.zeros(999, np.int64)])
            src = np.concatenate([src, np.ones(999, np.int64)])
            t = np.concatenate([t, np.full(999, t_last)])
        decay = clock(rng, lam, st.L, t_last)
        gap, X = anchor_inputs(model) if lazy else (0, 0.0)
        with debug_flags(flags):
            assert st.update_messages(tgt, src, t, t_last, lam, decay, n_local, count) == 0
        out = model.update_messages(tgt, src, t, t_last, lam, decay, n_local, count, device_count=count is not None,
                                    flags=flags, anchor=lazy)
        rc, res = out if lazy else (out, None)
        assert rc == 0
        check_state(st, model, (res, gap, X) if lazy else None)
        t_last += 600.0


@pytest.mark.parametrize('kind', ['small', 'large'])
def test_update_messages_precondition_flag(kind):
    """Lazy mode: a local source that is not a target of the same call sets the error flag to 2."""
    st, model, rng = make_state(41, 3000, 2, 20, 20, 3 * 20, True)
    n = 1000 if kind == 'small' else 20_000
    tgt = rng.integers(0, 1000, n).astype(np.int64)
    src = rng.integers(0, 1000, n).astype(np.int64)
    src[5] = 2500                                          # local (num_local_rows = 3000), never a target
    t = np.full(n, 100.0)
    st.update_messages(tgt, src, t, 100.0, 1e-3, None, 3000, None if kind == 'small' else n)
    assert int(st.err.item()) == 2


# --------------------------------------------------------------------------- refusals
@pytest.mark.parametrize('batch', [500, 20_000])
@pytest.mark.parametrize('why', ['capacity', 'floor'])
def test_log_full_changes_nothing(why, batch):
    """TPN_ERR_LOG_FULL: the log is full, or cum_floor * min(c) < 1e-200 — data, stamps, log, epoch and cum_floor
    unchanged bit for bit.  The same call without a clock move goes through."""
    st, model, rng = make_state(51, 3000, 3, 30, 32, 4 * 32 + 4, True, capacity=EPOCH + 1 if why == 'capacity' else None)
    if why == 'floor':
        st.st.cum_floor = model.cum_floor = 5e-200
    src, dst = rng.integers(0, 3000, batch).astype(np.int64), rng.integers(0, 3000, batch).astype(np.int64)
    lam, t_last = 1e-3, 1.0e4
    t = times_for(rng, batch, lam, t_last)
    decay = decay_factors(lam, t_last, t_last - 2.0 / lam, 3)
    before = st.host()
    assert st.update(src, dst, t, lam, decay) == LOG_FULL
    assert model.update(src, dst, t, lam, decay) == LOG_FULL
    after = st.host()
    for i, what in enumerate(('data', 'stamps', 'decay log')):
        same_bits(after[i], before[i], what)
    assert after[3:] == before[3:]
    assert run_update(st, model, src, dst, t, lam, None) == 0


# --------------------------------------------------------------------------- readers
READ_LAYOUTS = [(1, 210, 212, 2 * 212 + 8), (2, 13, 16, 3 * 16), (3, 997, 1004, 4 * 1004 + 12), (4, 5, 8, 5 * 8 + 4)]


@pytest.mark.parametrize('L,d,rs,ns', READ_LAYOUTS, ids=[f'L{x[0]}-rs{x[2]}' for x in READ_LAYOUTS])
def test_readers(L, d, rs, ns):
    """tpn_gather, tpn_gather_blocks (the whole node block, NaN gap included), then tpn_materialize (stamp -1 rows
    untouched, the others set to the epoch) and tpn_reset_epoch, on hand-built states."""
    st, model, rng = make_state(61 + L, 700, L, d, rs, ns, True)
    ids = np.concatenate([rng.integers(-700, 700, 900), [0, 699, -1, -700]]).astype(np.int64)
    same_bits(st.gather(ids), model.gather(ids), 'gather')
    same_bits(st.gather_blocks(ids), model.gather_blocks(ids), 'gather_blocks')
    dead = model.stamps < 0
    assert st.materialize() == 0
    model.materialize()
    check_state(st, model)
    assert np.all(model.stamps[dead] == -1) and np.all(model.stamps[~dead] == EPOCH)
    same_bits(st.gather(ids), model.gather(ids), 'gather after materialize')
    assert st.reset_epoch() == 0
    model.reset_epoch()
    check_state(st, model)
    same_bits(st.gather_blocks(ids), model.gather_blocks(ids), 'gather_blocks after the restart')
    src, dst = rng.integers(0, 700, 300).astype(np.int64), rng.integers(0, 700, 300).astype(np.int64)
    lam, t_last = 1e-3, 2.0e3
    assert run_update(st, model, src, dst, times_for(rng, 300, lam, t_last), lam, clock(rng, lam, L, t_last)) == 0


# --------------------------------------------------------------------------- the module
def module_model(m):
    st = m._state.detach().cpu().numpy().reshape(m.node_num, -1)
    return LazyDecayModel(st, m.node_num, m.num_layer, m.dim, m.row_stride, m.node_stride,
                          stamps=m._stamps.cpu().numpy(), log_capacity=m._decay_log.shape[0])


def test_module_bits_and_log_restart(monkeypatch):
    """A lazy RandomProjectionModule with a 5-row log (restarted every 4 updates) and lambda * dt ~ 0.3 per update,
    fed small and large batches through update_prepare + update, get_random_projections, backup / reload and
    state_dict: after every call its state and stamps are the model's bit for bit, the model restarting its log
    exactly where the module does."""
    monkeypatch.setattr(rpmod, '_DEFAULT_LOG_EPOCHS', 5)
    rng = np.random.default_rng(71)
    N, L, dim = 6000, 3, 44
    lam = 3e-4
    kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=lam, use_matrix=False,
              beginning_time=0.0, not_scale=False, enforce_dim=dim)
    torch.manual_seed(3)
    m = RandomProjectionModule(device=DEV, decay_mode='lazy', **kw).to(DEV)
    m.get_random_projections(np.arange(4))                   # creates the stamps (-1: nothing written) and the log
    model = module_model(m)
    now = 0.0
    restarts = 0

    def compare(what):
        torch.cuda.synchronize()
        same_bits(m._state.detach().cpu().numpy().reshape(N, -1), model.data, f'state after {what}')
        same_bits(m._stamps.cpu().numpy(), model.stamps, f'stamps after {what}')
        assert m._h.epoch == model.epoch, what

    def update(src, dst, t, prepare):
        nonlocal now, restarts
        decay = decay_factors(lam, t[-1], now, L)
        if prepare:
            m.update_prepare(src, dst, t)
            compare('update_prepare')
        m.update(src, dst, t)
        rc = model.update(src, dst, t, lam, decay)
        if rc == LOG_FULL:
            model.materialize()
            model.reset_epoch()
            restarts += 1
            rc = model.update(src, dst, t, lam, decay)
        assert rc == 0
        now = float(t[-1])
        compare('update')

    saved = None
    for k in range(14):
        B = int(rng.choice([300, 1800, 9000]))
        src, dst = designed_batch(rng, N, [(1, B // 3)] if B > 2048 else [])
        src, dst = src[:B], dst[:B]
        t = times_for(rng, len(src), lam, now + 0.3 / lam)
        update(src, dst, t, prepare=k % 2 == 1)
        if k % 3 == 2:
            ids = rng.integers(0, N, 500)
            got = [x.cpu().numpy() for x in m.get_random_projections(ids)]
            same_bits(np.stack(got), model.gather(ids), 'get_random_projections')
        if k == 5:
            saved = m.backup_random_projections()
            model.materialize()
            compare('backup')
            saved_rows = model.rows()[:, 1:, :].copy()
            saved_now = now
        if k == 9:
            m.reload_random_projections(saved)
            model.rows()[:, 1:, :] = saved_rows
            model.stamps[:] = 0
            model.epoch = 0
            now = saved_now
            compare('reload')
        if k == 11:
            sd = m.state_dict()
            model.materialize()
            compare('state_dict')
            for i in range(L + 1):
                same_bits(sd[f'random_projections.{i}'].cpu().numpy(), model.rows()[:, i, :dim], 'state_dict')
    assert restarts >= 2
