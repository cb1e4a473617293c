"""TEST / BASELINE INFRASTRUCTURE ONLY — two restatements of the negative edge sampler.

1. ``LiteralNegativeSampler``: the reference's ``NegativeEdgeSampler`` (DyGLib, the reference's utils/utils.py:315-505)
   written out with Python sets, as the reference computes it: ``W(a, b)`` = the distinct (src, dst) of the edges with
   a <= t <= b, ``Hc = W(earliest, s) - W(s, e)``, ``Ic = W(earliest, s) - observed - W(s, e)``,
   ``U = (S x D) - set(batch)``, the sizes and the ordering rule (random fill first, then all of Hc).  Its draws use
   ``np.random.RandomState`` like the reference; its set iteration order is Python's.

2. ``DeviceRestatement``: an integer-exact numpy restatement of ``tpn_neg_sampler_*`` (include/tpnet_b200.h): the
   tables T and F, the keyed Feistel permutation on top of Philox4x64-10 (``oracle.p0_counter``), the exclusion and
   the compaction.  The device must be bit-equal to it.
"""
from __future__ import annotations

from typing import Optional, Set, Tuple

import numpy as np

from oracle.p0_counter import mulhilo64, philox4x64_10

TAG_HIST, TAG_FILL, TAG_REPLACE, TAG_RANDOM = 1, 2, 3, 4
STRATEGIES = ('random', 'historical', 'inductive')


# ---------------------------------------------------------------------------------------------- 1. the literal sets
class LiteralNegativeSampler:
    def __init__(self, src_node_ids, dst_node_ids, interact_times=None, last_observed_time=None,
                 negative_sample_strategy: str = 'random', seed: Optional[int] = None):
        assert negative_sample_strategy in STRATEGIES
        self.seed = seed
        self.negative_sample_strategy = negative_sample_strategy
        self.src_node_ids = np.asarray(src_node_ids)
        self.dst_node_ids = np.asarray(dst_node_ids)
        self.interact_times = None if interact_times is None else np.asarray(interact_times)
        self.unique_src_node_ids = np.unique(self.src_node_ids)
        self.unique_dst_node_ids = np.unique(self.dst_node_ids)
        self.earliest_time = None if interact_times is None else self.interact_times.min()
        self.last_observed_time = last_observed_time
        if negative_sample_strategy != 'random':
            self.possible_edges = set((int(s), int(d)) for s in self.unique_src_node_ids
                                      for d in self.unique_dst_node_ids)
        if negative_sample_strategy == 'inductive':
            self.observed_edges = self.window(self.earliest_time, self.last_observed_time)
        if seed is not None:
            self.random_state = np.random.RandomState(seed)

    def window(self, start, end) -> Set[Tuple[int, int]]:
        """W(start, end): both bounds inclusive, every edge of the constructor's data."""
        sel = np.logical_and(self.interact_times >= start, self.interact_times <= end)
        return set((int(s), int(d)) for s, d in zip(self.src_node_ids[sel], self.dst_node_ids[sel]))

    def historical_domain(self, start, end) -> Set[Tuple[int, int]]:
        return self.window(self.earliest_time, start) - self.window(start, end)

    def inductive_domain(self, start, end) -> Set[Tuple[int, int]]:
        return self.window(self.earliest_time, start) - self.observed_edges - self.window(start, end)

    def fill_domain(self, batch_src, batch_dst) -> Set[Tuple[int, int]]:
        return self.possible_edges - set((int(s), int(d)) for s, d in zip(batch_src, batch_dst))

    def reset_random_state(self):
        self.random_state = np.random.RandomState(self.seed)

    def sample(self, size, batch_src_node_ids=None, batch_dst_node_ids=None, current_batch_start_time=0.0,
               current_batch_end_time=0.0):
        if self.negative_sample_strategy == 'random':
            rs = np.random if self.seed is None else self.random_state
            i = rs.randint(0, len(self.unique_src_node_ids), size)
            j = rs.randint(0, len(self.unique_dst_node_ids), size)
            return self.unique_src_node_ids[i], self.unique_dst_node_ids[j]
        assert self.seed is not None, 'Random state is not initialized!'
        if self.negative_sample_strategy == 'historical':
            dom = self.historical_domain(current_batch_start_time, current_batch_end_time)
        else:
            dom = self.inductive_domain(current_batch_start_time, current_batch_end_time)
        src = np.array([e[0] for e in dom], dtype=np.int64)
        dst = np.array([e[1] for e in dom], dtype=np.int64)
        if size > len(dom):
            assert batch_src_node_ids is not None and batch_dst_node_ids is not None
            pool = list(self.fill_domain(batch_src_node_ids, batch_dst_node_ids))
            assert len(pool) > 0
            idx = self.random_state.choice(len(pool), size=size - len(dom), replace=len(pool) < size - len(dom))
            fs = np.array([pool[i][0] for i in idx], dtype=np.int64)
            fd = np.array([pool[i][1] for i in idx], dtype=np.int64)
            return np.concatenate([fs, src]).astype(np.int64), np.concatenate([fd, dst]).astype(np.int64)
        idx = self.random_state.choice(len(dom), size=size, replace=False)
        return src[idx].astype(np.int64), dst[idx].astype(np.int64)


# ---------------------------------------------------------------------------------------------- 2. the device algorithm
def time_key(t: np.ndarray) -> np.ndarray:
    """The order-preserving uint64 of an f64 (no NaN)."""
    u = np.asarray(t, dtype=np.float64).view(np.uint64)
    neg = (u >> np.uint64(63)) != 0
    return np.where(neg, ~u, u | np.uint64(1 << 63))


def feistel_bits(n: int) -> int:
    m = 2
    while m < 62 and (1 << m) < n:
        m += 2
    return m


def permute(pos: np.ndarray, n: int, tag: int, seed: int, call: int) -> np.ndarray:
    """Positions -> elements of the keyed permutation of [0, n): 4-round balanced Feistel, cycle-walking."""
    half = feistel_bits(n) // 2
    mask = np.uint64((1 << half) - 1)
    key = np.array([seed, call], dtype=np.uint64)
    y = np.asarray(pos, dtype=np.uint64).copy()
    todo = np.ones(len(y), dtype=bool)
    while todo.any():
        cur = y[todo]
        L, R = cur >> np.uint64(half), cur & mask
        for r in range(4):
            ctr = np.stack([R, np.full_like(R, r), np.full_like(R, tag), np.zeros_like(R)], axis=1)
            f = philox4x64_10(ctr, key)[:, 0] if len(R) else R
            L, R = R, L ^ (f & mask)
        cur = (L << np.uint64(half)) | R
        y[todo] = cur
        todo[todo] = cur >= np.uint64(n)
    return y


def draw_first(n: int, k: int, P: int, excluded, tag: int, seed: int, call: int, identity: bool = False) -> np.ndarray:
    """The first k elements of positions [0, P) of the order (keyed permutation, or identity) of [0, n) for which
    ``excluded`` is False, in position order."""
    if k == 0 or P == 0:
        return np.zeros(0, dtype=np.uint64)
    pos = np.arange(P, dtype=np.uint64)
    val = pos if identity else permute(pos, n, tag, seed, call)
    keep = val[~excluded(val)]
    assert len(keep) >= k
    return keep[:k]


def uniform_index(x: np.ndarray, n: int) -> np.ndarray:
    """hi64(x * n): an index in [0, n)."""
    return mulhilo64(np.asarray(x, dtype=np.uint64), np.full(len(x), n, dtype=np.uint64))[0]


class DeviceRestatement:
    """The tables and the draw rule of ``tpn_neg_sampler_*``, in numpy, integer-exact."""

    def __init__(self, src, dst, times=None, last_observed_time=None, seed: int = 0):
        src = np.asarray(src, dtype=np.int64)
        dst = np.asarray(dst, dtype=np.int64)
        self.seed = int(seed) & ((1 << 64) - 1)
        self.lot = -np.inf if last_observed_time is None else float(last_observed_time)
        self.S = np.unique(src)
        self.D = np.unique(dst)
        if times is None:
            return
        t = np.asarray(times, dtype=np.float64)
        order = np.argsort(time_key(t), kind='stable')                       # T
        self.t_src, self.t_dst, self.t_time = src[order], dst[order], t[order]
        k = np.lexsort((np.arange(len(t)), self.t_dst, self.t_src))         # (src, dst, T position)
        head = np.ones(len(k), dtype=bool)
        head[1:] = (self.t_src[k][1:] != self.t_src[k][:-1]) | (self.t_dst[k][1:] != self.t_dst[k][:-1])
        first = k[head]                                                      # K: the first edge of each key
        kid_of_t = np.empty(len(t), dtype=np.int64)
        kid_of_t[k] = np.cumsum(head) - 1
        ksrc, kdst, kf = self.t_src[first], self.t_dst[first], self.t_time[first]
        perm_f = np.argsort(time_key(kf), kind='stable')                     # F: (f, src, dst)
        self.f_src, self.f_dst, self.f_time = ksrc[perm_f], kdst[perm_f], kf[perm_f]
        fpos_of_k = np.empty(len(perm_f), dtype=np.int64)
        fpos_of_k[perm_f] = np.arange(len(perm_f))
        self.t_fpos = fpos_of_k[kid_of_t]

    # the parts of one call
    def params(self, strategy: str, start: float, end: float):
        lo = int(np.searchsorted(self.t_time, start, side='left'))
        hi = max(int(np.searchsorted(self.t_time, end, side='right')), lo)
        h = int(np.searchsorted(self.f_time, start, side='right'))
        o = int(np.searchsorted(self.f_time, self.lot, side='right')) if strategy == 'inductive' else 0
        a, b = o, max(o, h)
        win = np.unique(self.t_fpos[lo:hi])
        marked = win[(win >= a) & (win < b)]
        return a, b, marked

    def batch_keys(self, bsrc, bdst) -> np.ndarray:
        """Sorted indices i_S * |D| + i_D of the batch pairs inside S x D (|S||D| for the others)."""
        bsrc = np.asarray(bsrc, dtype=np.int64)
        bdst = np.asarray(bdst, dtype=np.int64)
        nS, nD = len(self.S), len(self.D)
        i = np.searchsorted(self.S, bsrc)
        j = np.searchsorted(self.D, bdst)
        ok = (i < nS) & (j < nD)
        ok[ok] &= (self.S[i[ok]] == bsrc[ok]) & (self.D[j[ok]] == bdst[ok])
        q = np.where(ok, i.astype(np.uint64) * np.uint64(nD) + j.astype(np.uint64), np.uint64(nS * nD))
        return np.sort(q)

    def sample(self, strategy: str, call: int, size: int, bsrc=None, bdst=None, start: float = 0.0,
               end: float = 0.0) -> Tuple[np.ndarray, np.ndarray]:
        seed, call = self.seed, int(call)
        if size == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.int64)
        if strategy == 'random':
            ctr = np.zeros((size, 4), dtype=np.uint64)
            ctr[:, 0] = np.arange(size, dtype=np.uint64)
            ctr[:, 2] = TAG_RANDOM
            x = philox4x64_10(ctr, np.array([seed, call], dtype=np.uint64))
            return (self.S[uniform_index(x[:, 0], len(self.S)).astype(np.int64)].astype(np.int64),
                    self.D[uniform_index(x[:, 1], len(self.D)).astype(np.int64)].astype(np.int64))
        a, b, marked = self.params(strategy, start, end)
        n = b - a
        xh = len(marked)
        hc = n - xh
        k = min(size, hc)
        mset = np.zeros(max(n, 1), dtype=bool)
        mset[marked - a] = True
        hidx = a + draw_first(n, k, k + xh, lambda v: mset[v.astype(np.int64)], TAG_HIST, seed,
                              call).astype(np.int64)
        out_src = np.empty(size, np.int64)
        out_dst = np.empty(size, np.int64)
        kf = size - hc if size > hc else 0
        out_src[kf:] = self.f_src[hidx]
        out_dst[kf:] = self.f_dst[hidx]
        if kf:
            keys = self.batch_keys(bsrc, bdst)
            nD = len(self.D)
            nsd = len(self.S) * nD
            xf = len(np.unique(keys[keys < np.uint64(nsd)]))
            u = nsd - xf
            if u == 0:
                out_src[:kf] = -1
                out_dst[:kf] = -1
                return out_src, out_dst
            excl = lambda v: np.isin(v, keys)                                # noqa: E731
            if u >= kf:
                q = draw_first(nsd, kf, kf + xf, excl, TAG_FILL, seed, call)
            else:                                                            # with replacement over U in index order
                pool = draw_first(nsd, u, nsd, excl, TAG_FILL, seed, call, identity=True)
                ctr = np.zeros((kf, 4), dtype=np.uint64)
                ctr[:, 0] = np.arange(kf, dtype=np.uint64)
                ctr[:, 2] = TAG_REPLACE
                x = philox4x64_10(ctr, np.array([seed, call], dtype=np.uint64))
                q = pool[uniform_index(x[:, 0], u).astype(np.int64)]
            q = q.astype(np.int64)
            out_src[:kf] = self.S[q // nD]
            out_dst[:kf] = self.D[q % nD]
        return out_src, out_dst
