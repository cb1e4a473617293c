"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) — numpy restatement of the
reference's temporal-walk-matrix projection state.

Follows ``/root/reference/models/TPNet.py:9-157`` (class RandomProjectionModule)
operation by operation, in fp32 with the reference's exact rounding points, so
that on identical inputs it reproduces the reference CPU result bit for bit when
given the reference's own edge weights (torch's vectorised ``exp`` is 1-ulp, not
correctly rounded, so the weights are the only quantity that cannot be
re-derived bit-exactly outside torch; see ``edge_weights``).

Parity status: PINNED.  ``tests/golden/make_golden.py`` (run in the build
container, where /root/reference is importable) checks this file bit-for-bit
against the imported reference class and writes the fixtures under
``tests/golden/``; ``tests/test_oracle.py`` re-checks it against those fixtures
and against the brute-force walk enumeration of the reference notebook
(``oracle/walk_bruteforce.py``) without needing /root/reference.

Rounding points restated (reference line in brackets):
  * timestamps are cast f64 -> f32 BEFORE the subtraction            [TPNet.py:77]
  * ``t_last`` is the LAST element of the batch, not the max          [TPNet.py:76]
  * diff  = f32(t_last) - f32(t_j)              (fp32 subtract)        [TPNet.py:78]
  * arg   = f32(-lambda) * diff                 (fp32 multiply)        [TPNet.py:78]
  * w_j   = exp(arg) in fp32                                          [TPNet.py:78]
  * c_i   = f32( pow(exp(-lambda*(t_last-now)), i) ), f64 on the host  [TPNet.py:84-85]
  * P_i  <- fl32(P_i * c_i) for i = 1..L over the WHOLE matrix          [TPNet.py:83-85]
  * layers processed top-down, so layer i consumes the decayed but not yet
    updated layer i-1                                                  [TPNet.py:90]
  * msg   = fl32(P_{i-1}[other] * w_j)          (rounded before add)   [TPNet.py:91-92]
  * P_i[src_j] += msg, all j in batch order; THEN P_i[dst_j] += msg    [TPNet.py:93-96]
  * now  <- t_last (f64)                                              [TPNet.py:99]
  * pair-wise: rows ordered a:P_0..P_L then b:P_0..P_L, Gram in fp32,
    row-major flatten, clamp at 0, log(x + 1.0) (not log1p)            [TPNet.py:119-128]
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np

F32 = np.float32


def projection_dim(node_num: int, edge_num: int, dim_factor: int, enforce_dim: int, use_matrix: bool) -> int:
    """Width rule of the projections — TPNet.py:30-33 and :45."""
    if use_matrix:
        return int(node_num)
    if enforce_dim != -1:
        return int(enforce_dim)
    return min(int(math.log(edge_num * 2)) * dim_factor, node_num)


def edge_weights(times: np.ndarray, t_last: float, lam: float) -> np.ndarray:
    """w_j of TPNet.py:77-78.  exp is evaluated in f64 and rounded once to f32
    (the correctly rounded value; torch's CPU exp agrees with it on ~97-99 % of
    inputs and is within 1 ulp otherwise)."""
    tf = np.asarray(times, dtype=np.float64).astype(F32)
    diff = F32(t_last) - tf                      # fp32 subtract
    arg = F32(-lam) * diff                       # fp32 multiply
    return np.exp(arg.astype(np.float64)).astype(F32)


def decay_factors(lam: float, t_last: float, now: float, num_layer: int) -> np.ndarray:
    """c_1..c_L of TPNet.py:84-85: f64 pow of f64 exp on the host, then one
    rounding to f32 when it meets the fp32 tensor."""
    base = np.exp(-lam * (np.float64(t_last) - np.float64(now)))
    return np.array([F32(np.power(base, i)) for i in range(1, num_layer + 1)], dtype=F32)


class WalkProjectionOracle:
    """State + operations of the reference module, numpy/fp32, CPU only."""

    LOOP_MAX = 512      # batches up to this size use the explicit Python loop

    def __init__(self, node_num: int, edge_num: int, dim_factor: int, num_layer: int,
                 time_decay_weight: float, use_matrix: bool, beginning_time: float,
                 not_scale: bool, enforce_dim: int, p0: Optional[np.ndarray] = None,
                 rng: Optional[np.random.Generator] = None):
        self.node_num = int(node_num)
        self.edge_num = int(edge_num)
        self.num_layer = int(num_layer)
        self.time_decay_weight = float(time_decay_weight)
        self.use_matrix = bool(use_matrix)
        self.not_scale = bool(not_scale)
        self.dim = projection_dim(node_num, edge_num, dim_factor, enforce_dim, use_matrix)
        self.begging_time = np.float64(beginning_time)   # (sic) reference attribute name, TPNet.py:36
        self.now_time = np.float64(beginning_time)
        self.pair_wise_feature_dim = (2 * self.num_layer + 2) ** 2          # TPNet.py:63
        self._rng = rng if rng is not None else np.random.default_rng(0)
        self.P: List[np.ndarray] = []
        self.reset(p0)

    # ---------------------------------------------------------------- state
    def _draw_p0(self) -> np.ndarray:
        # TPNet.py:58 / :139 — N(0, 1/sqrt(d)).  The RNG stream is torch's in the
        # reference; parity tests always copy P_0 across instead of re-drawing.
        return (self._rng.standard_normal((self.node_num, self.dim)) / math.sqrt(self.dim)).astype(F32)

    def reset(self, p0: Optional[np.ndarray] = None) -> None:
        """TPNet.py:131-139 (and the constructor, :44-62)."""
        if self.use_matrix:
            base = np.eye(self.node_num, dtype=F32) if not self.P else self.P[0]
        elif p0 is not None:
            base = np.ascontiguousarray(p0, dtype=F32).copy()
            assert base.shape == (self.node_num, self.dim)
        else:
            base = self._draw_p0()
        self.P = [base] + [np.zeros((self.node_num, self.dim), dtype=F32) for _ in range(self.num_layer)]
        self.now_time = np.float64(self.begging_time)

    def backup(self) -> Tuple[np.float64, List[np.ndarray]]:
        """TPNet.py:141-147 — P_0 is NOT part of the backup."""
        return np.float64(self.now_time), [self.P[i].copy() for i in range(1, self.num_layer + 1)]

    def reload(self, saved: Tuple[np.float64, Sequence[np.ndarray]]) -> None:
        """TPNet.py:149-157."""
        now, layers = saved
        self.now_time = np.float64(now)
        for i in range(1, self.num_layer + 1):
            self.P[i] = np.array(layers[i - 1], dtype=F32, copy=True)

    # --------------------------------------------------------------- update
    GIANT_MIN = 2048    # chunked order: rows with at least this many messages in one update

    def update(self, src: np.ndarray, dst: np.ndarray, times: np.ndarray,
               weights: Optional[np.ndarray] = None, giant_chunk: int = 0) -> None:
        """TPNet.py:67-99.  ``weights`` lets the pinning script inject the
        reference's own torch-computed w_j so that everything else can be
        compared bit-for-bit.

        ``giant_chunk = C > 0`` restates the library's CHUNKED accumulation order
        (include/tpnet_b200.h, ``tpn_state_t::giant_chunk``; not a reference behaviour): a row that
        receives >= GIANT_MIN messages in this update has them cut, in the reference's order, into
        chunks of C; each chunk is summed sequentially; the chunk sums are added to the decayed row in
        chunk order.  Every other row keeps the reference's sequential order."""
        src = np.asarray(src, dtype=np.int64)
        dst = np.asarray(dst, dtype=np.int64)
        times = np.asarray(times, dtype=np.float64)
        if src.size == 0:
            raise IndexError("empty batch: the reference indexes node_interact_times[-1] (TPNet.py:76)")
        if src.min() < 0 or dst.min() < 0 or src.max() >= self.node_num or dst.max() >= self.node_num:
            raise IndexError("node id out of range")
        t_last = np.float64(times[-1])
        w = edge_weights(times, t_last, self.time_decay_weight) if weights is None \
            else np.asarray(weights, dtype=F32)
        c = decay_factors(self.time_decay_weight, t_last, self.now_time, self.num_layer)
        for i in range(1, self.num_layer + 1):
            self.P[i] = self.P[i] * c[i - 1]                     # fp32 * fp32, whole matrix
        for i in range(self.num_layer, 0, -1):
            below = self.P[i - 1]
            msg_to_src = below[dst] * w[:, None]                 # gathered BEFORE either scatter
            msg_to_dst = below[src] * w[:, None]
            tgt = self.P[i]
            if giant_chunk > 0:
                self._chunked_scatter(tgt, np.concatenate([src, dst]), np.concatenate([msg_to_src, msg_to_dst]),
                                      int(giant_chunk))
            elif src.shape[0] <= self.LOOP_MAX:
                for j in range(src.shape[0]):                    # batch order per target row
                    tgt[src[j]] += msg_to_src[j]
                for j in range(dst.shape[0]):
                    tgt[dst[j]] += msg_to_dst[j]
            else:
                # ufunc.at is unbuffered and applies the operands one index at a time in
                # index order — the same sequential fp32 adds as the loop above
                # (tests/test_oracle.py::test_add_at_equals_loop), just not in Python
                np.add.at(tgt, src, msg_to_src)
                np.add.at(tgt, dst, msg_to_dst)
        self.now_time = t_last

    def _chunked_scatter(self, tgt: np.ndarray, rows: np.ndarray, msgs: np.ndarray, chunk: int) -> None:
        """``rows``/``msgs``: the 2B messages of one layer in the reference's order (all src-role messages
        in batch order, then all dst-role messages).  Non-giant rows: sequential adds (== the two add.at of
        the reference order).  Giant rows: chunk sums, then the chunk sums in order."""
        counts = np.bincount(rows, minlength=self.node_num)
        giants = np.nonzero(counts >= self.GIANT_MIN)[0]
        small = ~np.isin(rows, giants)
        np.add.at(tgt, rows[small], msgs[small])
        order = np.argsort(rows, kind='stable')                   # each row's messages, in order
        start = np.searchsorted(rows[order], giants)
        for g, lo in zip(giants, start):
            m = msgs[order[lo:lo + counts[g]]]
            acc = tgt[g].copy()
            for c0 in range(0, m.shape[0], chunk):
                # np.add.accumulate adds one element at a time in the array's dtype (sequential fp32 adds)
                part = np.add.accumulate(m[c0:c0 + chunk], axis=0, dtype=F32)[-1]
                acc = acc + part
            tgt[g] = acc

    # ---------------------------------------------------------------- reads
    def get_random_projections(self, node_ids: np.ndarray) -> List[np.ndarray]:
        """TPNet.py:101-110 — list of L+1 arrays [n, d]."""
        ids = np.asarray(node_ids, dtype=np.int64)
        return [self.P[i][ids] for i in range(self.num_layer + 1)]

    def pair_wise_gram(self, a_ids: np.ndarray, b_ids: np.ndarray, exact: bool = False) -> np.ndarray:
        """The input of ``self.mlp`` in TPNet.py:112-129: [n, (2L+2)^2] fp32.
        ``exact=True`` accumulates the Gram in f64 (used to bound fp32 summation
        -order noise; the reference itself uses an fp32 batched GEMM)."""
        a = np.stack(self.get_random_projections(a_ids), axis=1)   # [n, L+1, d]
        b = np.stack(self.get_random_projections(b_ids), axis=1)
        x = np.concatenate([a, b], axis=1)                          # [n, 2L+2, d]
        if exact:
            g = np.einsum('nrd,ncd->nrc', x.astype(np.float64), x.astype(np.float64)).astype(F32)
        else:
            g = np.matmul(x, x.transpose(0, 2, 1))                  # fp32
        g = g.reshape(len(x), -1)
        if self.not_scale:
            return g
        g = np.where(g < 0, F32(0), g)
        return np.log(g + F32(1.0)).astype(F32)

    def neighbor_pair_lists(self, nbr: np.ndarray, src: np.ndarray, dst: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """The two id lists the encoder builds at TPNet.py:313-316 for m rows with K neighbours:
        ``np.tile(nbr.reshape(-1), 2)`` and ``concat(repeat(src, K), repeat(dst, K))``."""
        k = nbr.shape[1]
        a = np.tile(nbr.reshape(-1), 2)
        b = np.concatenate([np.repeat(src, k), np.repeat(dst, k)])
        return a.astype(np.int64), b.astype(np.int64)

    def neighbor_pair_wise_gram(self, nbr: np.ndarray, src: np.ndarray, dst: np.ndarray, exact: bool = False
                                ) -> np.ndarray:
        """TPNet.py:313-324 without the head: the generic pair encoder over the 2mK pairs of
        ``neighbor_pair_lists``, then ``cat([f[:mK], f[mK:]], dim=1).reshape(m, K, -1)`` -> [m, K, 2F]
        (the head acts on each F-block separately, so it commutes with the re-split)."""
        m, k = nbr.shape
        a, b = self.neighbor_pair_lists(nbr, src, dst)
        f = self.pair_wise_gram(a, b, exact=exact)
        return np.concatenate([f[:m * k], f[m * k:]], axis=1).reshape(m, k, -1)

    def pair_norm_bound(self, a_ids: np.ndarray, b_ids: np.ndarray) -> np.ndarray:
        """sqrt(G_rr * G_cc) per output element — the Cauchy-Schwarz scale that
        fp32 summation-order noise of a dot product is proportional to."""
        a = np.stack(self.get_random_projections(a_ids), axis=1).astype(np.float64)
        b = np.stack(self.get_random_projections(b_ids), axis=1).astype(np.float64)
        x = np.concatenate([a, b], axis=1)
        nrm = np.sqrt(np.einsum('nrd,nrd->nr', x, x))
        return (nrm[:, :, None] * nrm[:, None, :]).reshape(len(x), -1)
