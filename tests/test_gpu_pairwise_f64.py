"""GPU suite: every pair-wise kernel and both heads against a float64 reference, on hand-built raw-ABI states.

The pair-wise features are held to a bound from error analysis, not a fitted one.  A Gram entry G = sum_i x_i y_i
over n = row_stride + 8 or fewer fp32 operations (FFMA or not, any order) satisfies
    |got - G| <= gamma_n * sum_i |x_i y_i| + n * 2^-149,    gamma_n = n u / (1 - n u),  u = 2^-24
(the additive term covers subnormal products).  The log features add the propagation of that bound through
log(max(G, 0) + 1), 2^-24 for rounding g + 1, and 1 ulp for the log itself.

States are laid out by hand (tpn_state_t): any row_stride that is a multiple of 4, a padded node_stride, and in lazy
mode hand-made stamps and a decay log with factors far from 1.  The node_stride gap and one node past num_nodes are
NaN, so a read outside a node's L+1 rows shows up as NaN in the raw features.
"""
import ctypes
import re

import numpy as np
import pytest
import torch

from raw_state import RawState
from tpnet_b200 import RandomProjectionModule, _lib

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
U = 2.0 ** -24
TINY = 2.0 ** -149
UNSUPPORTED = -5
HEAD_FFMA = 8                                    # TPN_DEBUG_HEAD_FFMA (include/tpnet_b200.h)


# --------------------------------------------------------------------------- the reference bound
def raw_bound(s, rs):
    n = rs + 8
    return n * U / (1 - n * U) * s + n * TINY


def check_raw(got, g, s, rs):
    assert np.isfinite(g).all() and np.isfinite(got).all()
    err = np.abs(got.astype(np.float64) - g)
    tol = raw_bound(s, rs)
    assert np.all(err <= tol), (float(np.max(err - tol)), int(np.argmax(err - tol)))


def log_expect(g, s, rs):
    """Reference log feature and its bound."""
    e = raw_bound(s, rs)
    ref = np.log1p(np.maximum(g, 0.0))
    tol = e / (1.0 + np.maximum(g - e, 0.0)) + U
    tol = tol + np.spacing(np.float32(ref + tol)).astype(np.float64)
    return ref, tol


def check_log(got, g, s, rs):
    assert np.isfinite(g).all() and np.isfinite(got).all()
    ref, tol = log_expect(g, s, rs)
    err = np.abs(got.astype(np.float64) - ref)
    assert np.all(err <= tol), (float(np.max(err - tol)), int(np.argmax(err - tol)))


def check(got, g, s, rs, log):
    (check_log if log else check_raw)(got, g, s, rs)


def random_rows(rng, N, H, d):
    return (rng.standard_normal((N, H, d)) / np.sqrt(d)).astype(np.float32)


def nbr_reference(state, nbr, src, dst, exact_nonfinite=False):
    """Reference of tpn_pairwise_neighbors as two tpn_pairwise references: [m, K, 2, F] for G and sum |xy|."""
    m, K = nbr.shape
    a = np.concatenate([nbr.reshape(-1), nbr.reshape(-1)])
    b = np.concatenate([np.repeat(src, K), np.repeat(dst, K)])
    g, s = state.reference(a, b, exact_nonfinite)
    F = g.shape[1]
    shape = lambda x: x.reshape(2, m, K, F).transpose(1, 2, 0, 3)
    return shape(g), shape(s)


# --------------------------------------------------------------------------- which kernel a call takes
def _slot4(H, w):
    return (H * w + 7) & ~7


def pipe_fits(H, rs):
    """launch_pipe's test (tpn_pairwise.cu): two column chunks of the node blocks fit the per-warp staging."""
    ds4 = rs // 4
    if ds4 < 2:
        return False
    w = (ds4 + 1) // 2
    best = w
    for x in range(w, min(w + 3, ds4 - 1) + 1):
        if _slot4(H, x) - H * x < _slot4(H, best) - H * best:
            best = x
    w0, w1 = best, ds4 - best
    R = 2 * H
    per_warp = 16 * 8 * (_slot4(H, w0) + _slot4(H, w1))
    return (per_warp <= 110 * 1024 // 4 and 16 * R * R <= 128 * _slot4(H, w1) and 1 <= w0 <= 64 and 1 <= w1 <= 64)


def tma_fits(H, rs):
    bb = H * rs * 4
    R = 2 * H
    return 32 * bb <= 110 * 1024 and 16 * R * R <= 8 * bb


def pairwise_kernel_for(L, rs, n):
    H = L + 1
    if n <= 4096:
        return f'pairwise_kernel<{L}, 32>'
    if pipe_fits(H, rs):
        return f'pairwise_pipe_kernel<{L}>'
    if tma_fits(H, rs):
        return f'pairwise_tma_kernel<{L}>'
    return f'pairwise_kernel<{L}, 8>'


def nbr_warps(L, rs, K):
    """Warps per CTA of pairwise_nbr_kernel (launch_nbr), 0: TPN_ERR_UNSUPPORTED."""
    H = L + 1
    bb = H * rs * 4
    F = 4 * H * H
    wb = (max(4 * bb, 32 * F) + 127) // 128 * 128
    if 2 * bb + wb > 200 * 1024:
        return 0
    nw = min((K + 3) // 4, 5)
    budget = (72 if L <= 3 else 100) * 1024
    while nw > 1 and 2 * bb + nw * wb > budget:
        nw -= 1
    return nw


def launched(fn):
    """Pair-wise kernels fn() launches, as 'name<L[, G]>' strings, and its result."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r'(pairwise_(?:pipe_|tma_|nbr_)?kernel)<(\d+), (?:(\d+), )?(?:true|false)>', e.name)
        if m:
            names.add(f'{m.group(1)}<{m.group(2)}' + (f', {m.group(3)}>' if m.group(3) else '>'))
    return names, r


def _first_rs(L, want, lo=8, hi=1200, odd=None):
    """Smallest row_stride in [lo, hi) whose large call takes kernel `want` (odd: row_stride % 8 == 4 only)."""
    for rs in range(lo, hi, 4):
        if odd is not None and (rs % 8 == 4) != odd:
            continue
        if pairwise_kernel_for(L, rs, 5000) == want:
            return rs
    return None


def dispatch_cases():
    """(L, rs, n, kernel) for every tpn_pairwise path: small calls, the pipelined kernel at its narrowest rows and
    at a row_stride of 4 mod 8, the TMA kernel chosen by size and the register kernel for wide rows."""
    cases = []
    for L in (1, 2, 3, 4):
        cases.append((L, 20, 1003, f'pairwise_kernel<{L}, 32>'))
        pipe = [_first_rs(L, f'pairwise_pipe_kernel<{L}>'), _first_rs(L, f'pairwise_pipe_kernel<{L}>', lo=52, odd=True)]
        tma = _first_rs(L, f'pairwise_tma_kernel<{L}>')
        wide = _first_rs(L, f'pairwise_kernel<{L}, 8>', lo=160)
        for rs in sorted({x for x in pipe + [tma, wide] if x is not None}):
            cases.append((L, rs, 4099 + 4 * L, pairwise_kernel_for(L, rs, 4099)))
    return cases


def nbr_cases():
    """(L, rs, K, warps) with 5, 4, 3, 2 and 1 warps of pairwise_nbr_kernel, and the widest rows it refuses."""
    cases = []
    for L in (1, 2, 3, 4):
        seen = set()
        for rs in range(8, 6000, 4):
            w = nbr_warps(L, rs, 20)
            if w not in seen:
                seen.add(w)
                cases.append((L, rs, 20, w))
            if w == 0:
                break
    return cases


DISPATCH = dispatch_cases()
NBR = nbr_cases()
KERNELS = {f'pairwise_kernel<{L}, 32>' for L in (1, 2, 3, 4)} | {f'pairwise_kernel<{L}, 8>' for L in (1, 2, 3, 4)} | \
    {f'pairwise_{k}_kernel<{L}>' for k in ('pipe', 'tma') for L in (1, 2, 3, 4)}


def test_dispatch_table_covers_every_kernel():
    """Each kernel at each L is among the cases, the pipelined kernel runs 1-float4 column chunks (row_stride 8 or 12)
    and a row_stride of 4 mod 8, and pairwise_nbr_kernel runs 5..1 warps and refuses the next width."""
    assert {k for _, _, _, k in DISPATCH} == KERNELS
    assert any(rs in (8, 12) and k.startswith('pairwise_pipe') for _, rs, _, k in DISPATCH)
    for L in (1, 2, 3, 4):
        assert any(rs % 8 == 4 and k == f'pairwise_pipe_kernel<{L}>' for l, rs, _, k in DISPATCH if l == L)
        assert {w for l, _, _, w in NBR if l == L} == {0, 1, 2, 3, 4, 5}


def _state(rng, L, rs, lazy, N=257, d=None, pad=12):
    d = d if d is not None else rs - 3 if rs > 8 else rs - 1         # d not a multiple of 4
    return RawState(random_rows(rng, N, L + 1, d), rs, (L + 1) * rs + pad, lazy=lazy, rng=rng)


def _pairs(rng, N, n):
    """Random pairs with runs of repeated b ids, self pairs and valid negative ids."""
    a = rng.integers(-N, N, n)
    b = np.repeat(rng.integers(-N, N, n // 4 + 1), 4)[:n]
    sel = rng.random(n) < 0.5
    b[sel] = rng.integers(-N, N, int(sel.sum()))
    b[:16] = a[:16]
    a[:3] = -1
    return a.astype(np.int64), b.astype(np.int64)


@pytest.mark.parametrize('lazy', [False, True], ids=['eager', 'lazy'])
@pytest.mark.parametrize('L,rs,n,kernel', DISPATCH, ids=[f'{k}-rs{rs}' for _, rs, _, k in DISPATCH])
def test_dispatch_paths(L, rs, n, kernel, lazy):
    rng = np.random.default_rng(L * 7919 + rs + lazy)
    st = _state(rng, L, rs, lazy)
    a, b = _pairs(rng, st.N, n)
    g, s = st.reference(a, b)
    for log in (False, True):
        names, got = launched(lambda: st.pairwise(a, b, log))
        assert names == {kernel}, names
        check(got, g, s, rs, log)


@pytest.mark.parametrize('lazy', [False, True], ids=['eager', 'lazy'])
@pytest.mark.parametrize('L,rs,K,warps', NBR, ids=[f'L{L}-rs{rs}-w{w}' for L, rs, _, w in NBR])
def test_neighbor_paths(L, rs, K, warps, lazy):
    """tpn_pairwise_neighbors at each warp count (ragged K: 19 and K = 20), and TPN_ERR_UNSUPPORTED past them,
    where the tpn_pairwise call of the same pairs gives the same features."""
    rng = np.random.default_rng(L * 31 + rs + lazy)
    st = _state(rng, L, rs, lazy, N=97)
    for k in (K - 1, K):
        m = 7
        nbr = rng.integers(-st.N, st.N, (m, k)).astype(np.int64)
        src = rng.integers(-st.N, st.N, m).astype(np.int64)
        dst = src.copy()
        dst[::2] = rng.integers(0, st.N, (m + 1) // 2)
        g, s = nbr_reference(st, nbr, src, dst)
        for log in (False, True):
            names, (rc, got) = launched(lambda: st.neighbors(nbr, src, dst, log))
            if warps == 0:
                assert rc == UNSUPPORTED and not names
                a = np.concatenate([nbr.reshape(-1), nbr.reshape(-1)])
                b = np.concatenate([np.repeat(src, k), np.repeat(dst, k)])
                gf, sf = st.reference(a, b)
                check(st.pairwise(a, b, log), gf, sf, rs, log)
                continue
            assert rc == 0 and names == {f'pairwise_nbr_kernel<{L}>'}, (rc, names)
            check(got.reshape(-1, g.shape[-1]), g.reshape(-1, g.shape[-1]), s.reshape(-1, g.shape[-1]), rs, log)


# --------------------------------------------------------------------------- magnitudes
@pytest.mark.parametrize('lazy', [False, True], ids=['eager', 'lazy'])
@pytest.mark.parametrize('rs,n', [(60, 1500), (60, 6000), (220, 6000), (300, 6000)])
def test_magnitudes(rs, n, lazy):
    """Rows scaled by 2^k, k in [-75, 60]: G from subnormal to ~2^120, near-cancelling pairs (clamped), zero rows."""
    rng = np.random.default_rng(rs + n + lazy)
    L, N, d = 3, 300, rs - 2
    rows = random_rows(rng, N, L + 1, d)
    k = rng.integers(-75, 61, N)
    rows *= np.exp2(k).astype(np.float32)[:, None, None]
    rows[N // 2:N // 2 + 40] = -rows[N // 2 - 40:N // 2] * np.float32(1 + 2 ** -20)     # G(a, b) ~ -|a|^2
    rows[7] = 0
    st = RawState(rows, rs, (L + 1) * rs + 4, lazy=lazy, rng=rng)
    a, b = _pairs(rng, N, n)
    b[:200] = (a[:200] % N + N // 2) % N
    g, s = st.reference(a, b)
    assert np.max(s) < 2.0 ** 126 and np.min(np.abs(g[g != 0])) < 2.0 ** -126
    for log in (False, True):
        check(st.pairwise(a, b, log), g, s, rs, log)
    nbr = rng.integers(0, N, (40, 20)).astype(np.int64)
    src, dst = rng.integers(0, N, 40).astype(np.int64), rng.integers(0, N, 40).astype(np.int64)
    if nbr_warps(L, rs, 20):
        gn, sn = nbr_reference(st, nbr, src, dst)
        for log in (False, True):
            rc, got = st.neighbors(nbr, src, dst, log)
            assert rc == 0
            F = gn.shape[-1]
            check(got.reshape(-1, F), gn.reshape(-1, F), sn.reshape(-1, F), rs, log)


@pytest.mark.parametrize('n', [64, 6000])
def test_overflow_is_inf(n):
    """An entry whose exact G is >= 2^129 is +inf, raw and log, in every kernel."""
    L, N, rs, d = 2, 50, 24, 20
    rows = np.full((N, L + 1, d), 2.0 ** 63, np.float32)          # G = 20 * 2^126 > 2^130 between big nodes
    rows[:25] *= np.float32(2.0 ** -61)
    st = RawState(rows, rs, (L + 1) * rs, lazy=False)
    rng = np.random.default_rng(n)
    a, b = rng.integers(0, N, n).astype(np.int64), rng.integers(0, N, n).astype(np.int64)
    g, _ = st.reference(a, b)
    big = g >= 2.0 ** 129
    assert big.any() and (~big).any()
    for log in (False, True):
        got = st.pairwise(a, b, log)
        assert np.all(np.isposinf(got[big]))
        assert np.all(np.isfinite(got[g < 2.0 ** 127]))
    rc, got = st.neighbors(rng.integers(0, N, (4, 20)), np.arange(4), np.arange(40, 44), True)
    assert rc == 0 and np.isposinf(got).any()


# --------------------------------------------------------------------------- epilogue sweep
def sweep_values(rng):
    """Inputs of the epilogue: power-of-two boundaries +-4 ulps, the mantissa split of log_ge1 (4/3 2^k),
    random bit patterns over [0, FLT_MAX], negatives, +-0, subnormals, +-inf and NaN."""
    pos = []
    for e in range(-149, 128):
        p = np.float32(2.0 ** e).view(np.int32)
        pos.append(p + np.arange(-4, 5))
    for k in range(0, 127):
        pos.append(0x3f2aaaab + (k << 23) + np.arange(-4, 5))      # a = x + 1 at the split; x = a - 1 below
    bits = np.concatenate(pos).astype(np.int64)
    bits = bits[(bits > 0) & (bits < 0x7f800000)].astype(np.int32)
    v = bits.view(np.float32)
    split = v[-127 * 9:][v[-127 * 9:] >= 1] - np.float32(1)
    rnd = rng.integers(0, 0x7f7fffff, 2_000_000, dtype=np.int64).astype(np.int32).view(np.float32)
    sub = rng.integers(1, 0x7fffff, 20_000, dtype=np.int64).astype(np.int32).view(np.float32)
    special = np.float32([0.0, -0.0, np.inf, -np.inf, np.nan, -1.0, -3e38, -1e-45, 1e-45])
    x = np.concatenate([v, split, rnd, -rnd[:200_000], sub, -sub, special]).astype(np.float32)
    return x


def epilogue_expect(x):
    """log(fl32(max(x, 0) + 1)) in float64, NaN -> NaN, +inf -> +inf, -inf -> 0."""
    with np.errstate(invalid='ignore'):
        a = np.where(x < 0, np.float32(0), x).astype(np.float32) + np.float32(1)
        return np.log(a.astype(np.float64))


def check_epilogue(got, x):
    ref = epilogue_expect(x)
    nan = np.isnan(x)
    assert np.array_equal(np.isnan(got), nan)
    assert np.all(np.isposinf(got[np.isposinf(x)]))
    assert np.all(got[np.isneginf(x)] == 0)
    fin = np.isfinite(ref)
    err = np.abs(got[fin].astype(np.float64) - ref[fin])
    ulp = np.spacing(np.abs(ref[fin]).astype(np.float32)).astype(np.float64)
    assert np.all(err <= ulp), (float(np.max(err / ulp)), float(x[fin][np.argmax(err / ulp)]))


def test_epilogue_sweep():
    """Node a has P_l = [x_l, 0, ...], node `one` has P_0 = [1, 0, ...]: the entry (a_l, one_0) is x_l exactly, so the
    log features are the epilogue of each x, through tpn_pairwise (pipelined kernel) and tpn_pairwise_neighbors."""
    rng = np.random.default_rng(11)
    x = sweep_values(rng)
    L, H, rs = 3, 4, 8
    N = (len(x) + H - 1) // H + 1
    vals = np.zeros(N * H, np.float32)
    vals[:len(x)] = x
    rows = np.zeros((N, H, 5), np.float32)
    rows[:, :, 0] = vals.reshape(N, H)
    one = N - 1
    rows[one] = 0
    rows[one, 0, 0] = 1
    st = RawState(rows, rs, H * rs, lazy=False)
    a = np.arange(N - 1, dtype=np.int64)
    b = np.full(N - 1, one, np.int64)
    names, got = launched(lambda: st.pairwise(a, b, True))
    assert names == {pairwise_kernel_for(L, rs, N - 1)}
    R = 2 * H
    ent = got.reshape(N - 1, R, R)[:, :H, H].reshape(-1)[:len(x)]      # rows a_l, column one_0
    check_epilogue(ent, x)
    K = 16
    m = (N - 1) // K
    rc, out = st.neighbors(a[:m * K].reshape(m, K), np.full(m, one, np.int64), np.full(m, one, np.int64), True)
    assert rc == 0
    for side in (0, 1):                                   # W.S and W.D blocks
        ent = out[:, :, side].reshape(m * K, R, R)[:, :H, H].reshape(-1)
        check_epilogue(ent, x[:m * K * H])
    small = st.pairwise(a[:1000], b[:1000], True).reshape(1000, R, R)[:, :H, H].reshape(-1)
    check_epilogue(small, x[:4000])


# --------------------------------------------------------------------------- non-finite rows
@pytest.mark.parametrize('lazy', [False, True], ids=['eager', 'lazy'])
@pytest.mark.parametrize('rs,n', [(24, 900), (24, 5000), (140, 5000), (300, 5000)])
def test_nonfinite_rows(rs, n, lazy):
    """NaN, +inf and -inf in a few nodes' rows: raw features have the reference's non-finite pattern entry by entry,
    log features map NaN -> NaN, +inf -> +inf, -inf -> 0; pairs that touch no poisoned node are bit-identical to a
    run on the state without the poison."""
    L, N = 2, 64
    rng = np.random.default_rng(rs + n + lazy)
    d = rs - 3
    rows = random_rows(rng, N, L + 1, d)
    bad = {3: (1, 5, np.nan), 4: (0, 0, np.inf), 5: (2, d - 1, -np.inf), 6: (0, 2, np.inf)}
    poisoned = rows.copy()
    for node, (l, c, v) in bad.items():
        poisoned[node, l, c] = v
    poisoned[6, 1, 2] = -np.inf                            # +inf and -inf in one node: NaN in its self entries
    sts = [RawState(r, rs, (L + 1) * rs + 8, lazy=lazy, rng=np.random.default_rng(7)) for r in (rows, poisoned)]
    a, b = _pairs(rng, N, n)
    a[:40] = np.repeat(np.arange(3, 7), 10)
    g, s = sts[1].reference(a, b, exact_nonfinite=True)
    touch = np.isin(a % N, list(bad)) | np.isin(b % N, list(bad))
    assert touch.any() and (~touch).any()
    for log in (False, True):
        clean = sts[0].pairwise(a, b, log)
        got = sts[1].pairwise(a, b, log)
        assert np.array_equal(got[~touch].view(np.int32), clean[~touch].view(np.int32))
        if log:
            assert np.array_equal(np.isnan(got), np.isnan(g))
            assert np.array_equal(np.isposinf(got), np.isposinf(g))
            assert np.all(got[np.isneginf(g)] == 0)
        else:
            for f in (np.isnan, np.isposinf, np.isneginf):
                assert np.array_equal(f(got), f(g)), f.__name__
        fin = np.isfinite(g)
        tol_ref = log_expect(g[fin], s[fin], rs) if log else (g[fin], raw_bound(s[fin], rs))
        assert np.all(np.abs(got[fin] - tol_ref[0]) <= tol_ref[1])
    nbr = np.tile(np.arange(0, 20), (6, 1)).astype(np.int64)
    src, dst = np.array([3, 4, 5, 6, 1, 2]), np.array([2, 6, 1, 9, 5, 4])
    if nbr_warps(L, rs, 20):
        gn, _ = nbr_reference(sts[1], nbr, src, dst, exact_nonfinite=True)
        rc, got = sts[1].neighbors(nbr, src, dst, True)
        assert rc == 0
        assert np.array_equal(np.isnan(got), np.isnan(gn))
        assert np.array_equal(np.isposinf(got), np.isposinf(gn))
        assert np.all(got[np.isneginf(gn)] == 0)


# --------------------------------------------------------------------------- the heads
@pytest.fixture(params=['ffma', 'tensor'])
def head_kernel(request):
    lib = _lib.load()
    old = lib.tpn_set_debug_flags(HEAD_FFMA if request.param == 'ffma' else 0)
    yield request.param
    lib.tpn_set_debug_flags(old)


def head(mlp, x):
    y = torch.full_like(x, -7.0)
    l1, l2 = mlp[0], mlp[2]
    rc = _lib.load().tpn_head_forward(x.data_ptr(), x.shape[0], None, 64, 256, l1.weight.data_ptr(),
                                      l1.bias.data_ptr(), l2.weight.data_ptr(), l2.bias.data_ptr(), y.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    return y


def make_mlp(seed):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(64, 256), torch.nn.ReLU(), torch.nn.Linear(256, 64)).to(DEV)


@pytest.mark.parametrize('bias', ['init', 'zero'])
def test_head_full_range(head_kernel, bias):
    """Row magnitudes 2^-126 .. 2^120 (the hidden and output layers stay finite in fp32 up to there), within the
    row-relative bound of test_gpu_parity.test_tensor_core_head_dynamic_range_and_counts."""
    mlp = make_mlp(7)
    if bias == 'zero':
        with torch.no_grad():
            mlp[0].bias.zero_()
            mlp[2].bias.zero_()
    n = 1000
    x = torch.rand(n, 64, device=DEV)
    x[::5, ::3] *= -1.0
    x *= torch.exp2(torch.linspace(-126, 120, n, device=DEV).round())[:, None]
    x[17] = 0
    got = head(mlp, x).double()
    with torch.no_grad():
        ref32 = mlp(x).double()
    want = mlp.double()(x.double())
    mlp.float()
    assert torch.isfinite(want).all() and torch.isfinite(ref32).all()
    row = want.abs().max(dim=1, keepdim=True).values + torch.finfo(torch.float64).tiny
    err = ((got - want).abs() / row).max(dim=1).values
    err32 = ((ref32 - want).abs() / row).max().item()
    assert torch.all(err <= 4 * err32 + 2e-6), (head_kernel, float(err.max()), int(err.argmax()), err32)


def test_head_nonfinite_inputs(head_kernel):
    """NaN in a row of x: that row is all NaN, every other row bit-identical to the call without it.  +-inf in x:
    the row is non-finite wherever torch's is."""
    mlp = make_mlp(8)
    n = 300
    x = torch.rand(n, 64, device=DEV) * 12.0
    clean = head(mlp, x)
    xp = x.clone()
    nan_rows, inf_rows = [3, 130, 299], [5, 200]
    xp[3, 0] = float('nan')
    xp[130, 63] = float('nan')
    xp[299] = float('nan')
    xp[5, 7] = float('inf')
    xp[200, 9] = -float('inf')
    got = head(mlp, xp)
    with torch.no_grad():
        ref = mlp(xp)
    assert torch.isnan(got[nan_rows]).all()
    assert (~torch.isfinite(got[~torch.isfinite(ref)])).all()
    assert not torch.isfinite(ref[inf_rows]).all(dim=1).any()
    keep = torch.ones(n, dtype=torch.bool, device=DEV)
    keep[nan_rows + inf_rows] = False
    assert torch.equal(got[keep].view(torch.int32), clean[keep].view(torch.int32))


@pytest.mark.parametrize('where', ['w1', 'b1'])
def test_head_nan_weights(head_kernel, where):
    """A NaN in W1 or b1 (a diverged training run): every output is NaN, as torch gives."""
    mlp = make_mlp(9)
    with torch.no_grad():
        (mlp[0].weight if where == 'w1' else mlp[0].bias).view(-1)[37] = float('nan')
    x = torch.rand(200, 64, device=DEV) * 12.0
    with torch.no_grad():
        assert torch.isnan(mlp(x)).all()
    assert torch.isnan(head(mlp, x)).all()


def test_get_pair_wise_feature_nonfinite_matches_autograd(head_kernel):
    """The no-grad kernel path of get_pair_wise_feature against the autograd (PyTorch) path: a NaN in a node's
    projection and then a NaN in mlp[0].weight give NaN exactly where the reference does."""
    kw = dict(node_num=60, edge_num=600, dim_factor=10, num_layer=3, time_decay_weight=1e-6, use_matrix=False,
              beginning_time=0.0, not_scale=False, enforce_dim=-1)
    torch.manual_seed(4)
    m = RandomProjectionModule(device=DEV, decay_mode='eager', **kw).to(DEV)
    ids = np.arange(1, 50, dtype=np.int64)
    other = ids[::-1].copy()
    with torch.no_grad():
        m.random_projections[0].data[9, 3] = float('nan')
        m.random_projections[0].data[12, 0] = float('inf')

    def both():
        with torch.no_grad():
            fused = m.get_pair_wise_feature(ids, other).clone()
        ref = m.get_pair_wise_feature(ids, other).detach()
        return fused, ref

    fused, ref = both()
    assert torch.equal(torch.isfinite(fused), torch.isfinite(ref))
    touch = torch.from_numpy(np.isin(ids, [9, 12]) | np.isin(other, [9, 12])).to(DEV)
    assert not torch.isfinite(ref[touch]).any() and torch.isfinite(ref[~touch]).all()
    scale = float(ref[~touch].abs().max()) + 1.0
    assert float((fused[~touch] - ref[~touch]).abs().max()) <= 2e-5 * scale
    with torch.no_grad():
        m.mlp[0].weight[5, 5] = float('nan')
    fused, ref = both()
    assert torch.isnan(ref).all() and torch.isnan(fused).all()
