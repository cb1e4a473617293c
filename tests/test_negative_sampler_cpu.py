"""CPU suite of the negative edge sampler: the device algorithm's numpy restatement (oracle/negative_sampler.py)
against the literal set semantics of the reference's NegativeEdgeSampler, the Feistel permutation, draw statistics,
host refusals and the C struct layout."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy import stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.negative_sampler import (TAG_FILL, TAG_HIST, DeviceRestatement, LiteralNegativeSampler,  # noqa: E402
                                     feistel_bits, permute)
from oracle.p0_counter import philox4x64_10  # noqa: E402
from tpnet_b200 import _lib  # noqa: E402
from tpnet_b200.negative_sampler import NegativeEdgeSampler  # noqa: E402

REF = os.path.join(ROOT, 'oracle', '_ref', 'TPNet')


def graph(seed, E=300, n_src=12, n_dst=9, bipartite=True, ties=4, shuffle=True):
    """A small graph with heavy time ties, in a shuffled (unsorted) order unless asked otherwise."""
    rng = np.random.default_rng(seed)
    src = rng.integers(1, n_src + 1, E)
    dst = rng.integers(n_src + 1, n_src + n_dst + 1, E) if bipartite else rng.integers(1, n_src + 1, E)
    t = np.floor(np.sort(rng.random(E)) * E / ties).astype(np.float64)
    if shuffle:
        p = rng.permutation(E)
        src, dst, t = src[p], dst[p], t[p]
    return src.astype(np.int64), dst.astype(np.int64), t


def batches(t, B):
    """(start, end, edge indices) of the time-ordered batches of B edges, as the evaluation loop slices them."""
    order = np.argsort(t, kind='stable')
    for i in range(0, len(t), B):
        idx = order[i:i + B]
        yield t[idx[0]], t[idx[-1]], idx


def domain_pairs(dev, strategy, s, e):
    a, b, marked = dev.params(strategy, s, e)
    keep = np.setdiff1d(np.arange(a, b), marked)
    return set(zip(dev.f_src[keep].tolist(), dev.f_dst[keep].tolist()))


LOTS = ('before', 'inside', 'after')


@pytest.mark.parametrize('bipartite', [True, False])
@pytest.mark.parametrize('lot', LOTS)
@pytest.mark.parametrize('seed', [0, 1, 2])
def test_domains_equal_the_literal_sets(bipartite, lot, seed):
    src, dst, t = graph(seed, bipartite=bipartite)
    lot_v = {'before': t.min() - 1.0, 'inside': float(np.median(t)), 'after': t.max() + 1.0}[lot]
    lit_h = LiteralNegativeSampler(src, dst, t, lot_v, 'historical', seed=1)
    lit_i = LiteralNegativeSampler(src, dst, t, lot_v, 'inductive', seed=1)
    dev = DeviceRestatement(src, dst, t, lot_v, seed=5)
    assert np.array_equal(dev.S, lit_h.unique_src_node_ids) and np.array_equal(dev.D, lit_h.unique_dst_node_ids)
    for s, e, idx in batches(t, 17):
        assert domain_pairs(dev, 'historical', s, e) == lit_h.historical_domain(s, e)
        assert domain_pairs(dev, 'inductive', s, e) == lit_i.inductive_domain(s, e)
        keys = dev.batch_keys(src[idx], dst[idx])
        nsd = len(dev.S) * len(dev.D)
        fill = set((int(dev.S[q // len(dev.D)]), int(dev.D[q % len(dev.D)])) for q in range(nsd) if q not in set(keys))
        assert fill == lit_h.fill_domain(src[idx], dst[idx])


def test_window_covers_ties_spilling_into_the_next_batch():
    src, dst, t = graph(3, ties=25)
    dev = DeviceRestatement(src, dst, t, seed=1)
    lit = LiteralNegativeSampler(src, dst, t, None, 'historical', seed=1)
    spilled = 0
    for s, e, idx in batches(t, 10):
        w = lit.window(s, e)
        spilled += len(w - set(zip(src[idx].tolist(), dst[idx].tolist())))
        a, b, marked = dev.params('historical', s, e)
        assert len(marked) == len(w & lit.window(lit.earliest_time, s))
    assert spilled > 0                                   # the graph does put equal end times into the next batch


@pytest.mark.parametrize('strategy', ['historical', 'inductive'])
@pytest.mark.parametrize('size', [1, 5, 40, 500])
def test_outputs_follow_the_reference_rule(strategy, size):
    src, dst, t = graph(4, bipartite=False)
    lot = float(np.quantile(t, 0.3))
    lit = LiteralNegativeSampler(src, dst, t, lot, strategy, seed=1)
    dev = DeviceRestatement(src, dst, t, lot, seed=9)
    cases = {'fill': 0, 'plain': 0, 'replace': 0, 'empty': 0}
    for call, (s, e, idx) in enumerate(batches(t, 23)):
        dom = lit.historical_domain(s, e) if strategy == 'historical' else lit.inductive_domain(s, e)
        os_, od = dev.sample(strategy, call, size, src[idx], dst[idx], s, e)
        assert os_.dtype == np.int64 and len(os_) == size
        pairs = list(zip(os_.tolist(), od.tolist()))
        if size <= len(dom):
            cases['plain'] += 1
            assert len(set(pairs)) == size and set(pairs) <= dom
            continue
        cases['empty' if not dom else 'fill'] += 1
        k = size - len(dom)
        assert set(pairs[k:]) == dom and len(pairs[k:]) == len(dom)       # all of Hc, after the fill
        pool = lit.fill_domain(src[idx], dst[idx])
        assert set(pairs[:k]) <= pool
        if len(pool) >= k:
            assert len(set(pairs[:k])) == k
        else:
            cases['replace'] += 1
    assert cases['plain'] + cases['fill'] > 0
    if size == 500:
        assert cases['replace'] > 0 and cases['fill'] > 0


def test_empty_fill_domain_writes_minus_one():
    src = np.array([1, 1, 2, 2], dtype=np.int64)
    dst = np.array([3, 4, 3, 4], dtype=np.int64)
    t = np.array([0.0, 1.0, 2.0, 3.0])
    dev = DeviceRestatement(src, dst, t, seed=1)
    os_, od = dev.sample('historical', 0, 3, src, dst, 0.0, 3.0)
    assert (os_ == -1).all() and (od == -1).all()


def inverse_permute(y, n, tag, seed, call):
    half = feistel_bits(n) // 2
    mask = np.uint64((1 << half) - 1)
    key = np.array([seed, call], dtype=np.uint64)
    y = np.asarray(y, dtype=np.uint64).copy()
    todo = np.ones(len(y), dtype=bool)
    while todo.any():
        cur = y[todo]
        L, R = cur >> np.uint64(half), cur & mask
        for r in (3, 2, 1, 0):
            ctr = np.stack([L, np.full_like(L, r), np.full_like(L, tag), np.zeros_like(L)], axis=1)
            f = philox4x64_10(ctr, key)[:, 0]
            L, R = R ^ (f & mask), L
        cur = (L << np.uint64(half)) | R
        y[todo] = cur
        todo[todo] = cur >= np.uint64(n)
    return y


@pytest.mark.parametrize('n', [1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 255, 256, 257, 1023, 1024, 1025, 4097])
def test_feistel_is_a_bijection(n):
    for call in (0, 1, 77):
        y = permute(np.arange(n, dtype=np.uint64), n, TAG_HIST, 12345, call)
        assert np.array_equal(np.sort(y), np.arange(n, dtype=np.uint64))


def test_feistel_near_1e14_inverts():
    n = 10 ** 14 + 12345
    assert feistel_bits(n) == 48
    pos = np.random.default_rng(0).integers(0, n, 2000, dtype=np.uint64)
    y = permute(pos, n, TAG_FILL, 99, 3)
    assert (y < np.uint64(n)).all()
    assert np.array_equal(inverse_permute(y, n, TAG_FILL, 99, 3), pos)
    assert len(np.unique(y)) == len(pos)


def test_draws_are_uniform_over_elements_and_positions():
    src, dst, t = graph(5, E=400, n_src=10, n_dst=6)
    dev = DeviceRestatement(src, dst, t, seed=2024)
    s, e = float(t.max()) + 1, float(t.max()) + 2         # empty window: the domain is every distinct key
    n = len(dev.f_src)
    k = 8
    hits = np.zeros(n)
    first = np.zeros(n)
    for call in range(3000):
        os_, od = dev.sample('historical', call, k, src[:0], dst[:0], s, e)
        idx = {p: i for i, p in enumerate(zip(dev.f_src.tolist(), dev.f_dst.tolist()))}
        got = [idx[p] for p in zip(os_.tolist(), od.tolist())]
        hits[got] += 1
        first[got[0]] += 1
    assert stats.chisquare(hits).pvalue > 1e-4
    assert stats.chisquare(first).pvalue > 1e-4
    r_s, r_d = dev.sample('random', 0, 200_000)
    cs = np.unique(r_s, return_counts=True)[1]
    cd = np.unique(r_d, return_counts=True)[1]
    assert len(cs) == len(dev.S) and len(cd) == len(dev.D)
    assert stats.chisquare(cs).pvalue > 1e-4 and stats.chisquare(cd).pvalue > 1e-4


def test_draws_depend_on_seed_and_call_only():
    src, dst, t = graph(6)
    a = DeviceRestatement(src, dst, t, seed=7)
    b = DeviceRestatement(src[::-1], dst[::-1], t[::-1], seed=7)          # the same edges, another input order
    s, e, idx = next(batches(t, 30))
    for call in range(3):
        x = a.sample('historical', call, 6, src[idx], dst[idx], s, e)
        y = b.sample('historical', call, 6, src[idx], dst[idx], s, e)
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])
    assert not np.array_equal(a.sample('historical', 0, 6, src[idx], dst[idx], s, e)[0],
                              a.sample('historical', 1, 6, src[idx], dst[idx], s, e)[0])


@pytest.mark.parametrize('kwargs, exc', [
    (dict(negative_sample_strategy='uniform'), ValueError),
    (dict(src_node_ids=[1, -2]), IndexError),
    (dict(src_node_ids=[1, 2 ** 32]), IndexError),
    (dict(src_node_ids=[1, 2, 3]), ValueError),
    (dict(src_node_ids=[], dst_node_ids=[]), ValueError),
    (dict(negative_sample_strategy='historical', interact_times=None), ValueError),
    (dict(negative_sample_strategy='inductive', last_observed_time=None), ValueError),
    (dict(interact_times=[0.0, np.nan]), ValueError),
    (dict(interact_times=[0.0]), ValueError),
    (dict(seed=-1), ValueError),
    (dict(device='cpu'), RuntimeError),
])
def test_constructor_refusals_before_any_device_work(kwargs, exc):
    args = dict(src_node_ids=[1, 2], dst_node_ids=[3, 4], interact_times=[0.0, 1.0], last_observed_time=0.5,
                negative_sample_strategy='inductive', seed=0, device='cuda:0')
    args.update(kwargs)
    with pytest.raises(exc):
        NegativeEdgeSampler(**args)


def test_struct_layout_matches_header(tmp_path):
    fields = [f[0] for f in _lib.TpnNegSampler._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tpnet_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(tpn_neg_sampler_t));']
    lines += [f'  printf("{f} %zu\\n", offsetof(tpn_neg_sampler_t, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'layout'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(_lib.TpnNegSampler)
    for f in fields:
        assert int(out[f]) == getattr(_lib.TpnNegSampler, f).offset, f


def test_c_entry_points_refuse_bad_arguments_without_a_gpu():
    lib = _lib.load()
    s = _lib.TpnNegSampler()
    assert lib.tpn_neg_sampler_build(ctypes.byref(s), None, None, None, None, 0, None) < 0
    assert lib.tpn_neg_sampler_sample(ctypes.byref(s), 1, 0, 10, None, None, 0, 0.0, 0.0, None, None, None, None,
                                      None, 0, None) < 0
    assert lib.tpn_neg_sampler_workspace_bytes(1000, 0, 0) > lib.tpn_neg_sampler_workspace_bytes(10, 0, 0)
    assert lib.tpn_neg_sampler_workspace_bytes(0, 200, 200) > 0


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, 'utils', 'utils.py')),
                    reason='oracle/_ref/TPNet is not installed (oracle/make_ref.py copies it from a TPNet checkout)')
@pytest.mark.parametrize('strategy', ['historical', 'inductive'])
def test_against_the_reference_class(strategy):
    sys.path.insert(0, REF)
    try:
        from utils.utils import NegativeEdgeSampler as Ref
    finally:
        sys.path.remove(REF)
    src, dst, t = graph(8, bipartite=False)
    lot = float(np.quantile(t, 0.4))
    ref = Ref(src, dst, t, lot, strategy, seed=0)
    lit = LiteralNegativeSampler(src, dst, t, lot, strategy, seed=0)
    dev = DeviceRestatement(src, dst, t, lot, seed=0)
    for call, (s, e, idx) in enumerate(batches(t, 23)):
        for size in (5, 200):
            rs, rd = ref.sample(size, src[idx], dst[idx], s, e)
            ds, dd = dev.sample(strategy, call, size, src[idx], dst[idx], s, e)
            dom = lit.historical_domain(s, e) if strategy == 'historical' else lit.inductive_domain(s, e)
            if size > len(dom):
                k = size - len(dom)
                assert set(zip(rs[k:].tolist(), rd[k:].tolist())) == set(zip(ds[k:].tolist(), dd[k:].tolist()))
            else:
                assert set(zip(rs.tolist(), rd.tolist())) <= dom and set(zip(ds.tolist(), dd.tolist())) <= dom
                assert len(set(zip(ds.tolist(), dd.tolist()))) == size
