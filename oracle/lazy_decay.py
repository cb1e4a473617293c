"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) — numpy restatement of the library's LAZY decay.

This is not a reference behaviour: it restates what ``tpn_update`` / ``tpn_update_messages`` and the readers do with
``stamps != NULL`` (include/tpnet_b200.h, "Time decay"; DESIGN.md section 3), as ``giant_chunk`` restates the chunked
order in ``walk_projection.py``.  Rules restated:

  * the decay log: row k of ``Q`` holds, per layer, the f64 product of the fp32 factors of epochs 1..k; an update
    whose factors are not all 1.0 appends ``Q[e+1] = Q[e] * f64(c)``; an update with ``decay == NULL`` (or all ones)
    appends nothing and runs at the same epoch
  * a row of layer l >= 1 last written at epoch s is read at epoch e as ``fl32(x * fl32(Q[e][l-1] / Q[s][l-1]))``,
    the division in f64; ``s == e`` reads x unchanged; ``s < 0`` (never written) reads the stored row, which the
    contract says is all zero.  P_0 never decays
  * an update refused with TPN_ERR_LOG_FULL (``epoch + 1 >= capacity``, or ``epoch > 0`` and
    ``cum_floor * min(1, c) < 1e-200``) changes nothing
  * every target and source is read current at the NEW epoch; the messages are the reference's
    (``WalkProjectionOracle``'s scatter, run on the current rows at a clock that does not move), in the chunked order
    only where the kernel uses it: a large batch (> 4,096 messages, or a device-side count) on the snapshot path
  * the targets' rows 1..L are stored and their L stamps set to the new epoch; nothing else is written

``chain64`` is the float64 anchor: it keeps the per-epoch fp32 factors (not Q), so the true current value of a row is
``x * prod_{k=s+1..e} c_k``, and runs the same messages in float64.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np

from oracle.walk_projection import WalkProjectionOracle, edge_weights

F32 = np.float32
SMALL_MAX_MSGS = 4096        # 2B <= this: the single-CTA sort path (reference order always)
GIANT_MIN = WalkProjectionOracle.GIANT_MIN
PER_LAYER_WALK = 1           # TPN_DEBUG_PER_LAYER_WALK
LOG_FULL = -3                # TPN_ERR_LOG_FULL


def effective_chunk(giant_chunk: int) -> int:
    """tpn_state_t::giant_chunk as update_impl clamps it: 0, or a multiple of 32 in 256..2048."""
    c = int(giant_chunk)
    if c <= 0:
        return 0
    c = min(max(c, 256), GIANT_MIN)
    return c & ~31


def _scatter(P: List[np.ndarray], lam: float, src, dst, times, chunk: int) -> None:
    """WalkProjectionOracle.update on rows that are already current: with now_time = t_last every factor is
    exactly 1.0 (fl32(x * 1) == x), so only the weights and the reference's scatter remain."""
    o = WalkProjectionOracle.__new__(WalkProjectionOracle)
    o.node_num, o.num_layer, o.time_decay_weight = P[0].shape[0], len(P) - 1, float(lam)
    o.now_time = np.float64(np.asarray(times, np.float64)[-1])
    o.P = P
    o.update(src, dst, times, giant_chunk=chunk)


class LazyDecayModel:
    """State of a tpn_state_t in host memory: ``data`` [rows, node_stride] fp32 (rows >= num_nodes: whatever lies
    past the state, compared but never touched), ``stamps`` [N, L] int32 (None: eager), ``Q`` [capacity, L] f64,
    ``epoch``, ``cum_floor`` and, for the anchor, ``factors[k]`` = the fp32 factors of epoch k (k >= 1)."""

    def __init__(self, data: np.ndarray, num_nodes: int, num_layer: int, dim: int, row_stride: int,
                 node_stride: int, stamps: Optional[np.ndarray] = None, factors: Optional[np.ndarray] = None,
                 log_capacity: int = 0, cum_floor: Optional[float] = None, giant_chunk: int = 0,
                 log_fill: Optional[np.ndarray] = None):
        self.N, self.L, self.d, self.rs, self.ns = int(num_nodes), int(num_layer), int(dim), int(row_stride), \
            int(node_stride)
        self.data = np.array(data, dtype=F32).reshape(-1, self.ns)
        self.giant_chunk = int(giant_chunk)
        self.lazy = stamps is not None
        self.stamps = None if stamps is None else np.array(stamps, dtype=np.int32).reshape(self.N, self.L)
        fac = np.zeros((0, self.L), F32) if factors is None else np.asarray(factors, F32).reshape(-1, self.L)
        self.factors: List[Optional[np.ndarray]] = [None] + [f.copy() for f in fac]
        self.epoch = len(fac)
        cap = max(int(log_capacity), self.epoch + 1)
        self.Q = np.full((cap, self.L), -7.0) if log_fill is None else np.array(log_fill, np.float64).reshape(cap, self.L)
        self.Q[0] = 1.0
        for k in range(1, self.epoch + 1):
            self.Q[k] = self.Q[k - 1] * self.factors[k].astype(np.float64)
        self.cum_floor = float(self.Q[:self.epoch + 1].min()) if cum_floor is None else float(cum_floor)

    # ------------------------------------------------------------------ rows
    def rows(self) -> np.ndarray:
        """[N, L+1, row_stride] view of the stored rows."""
        H = self.L + 1
        return self.data[:self.N, :H * self.rs].reshape(self.N, H, self.rs)

    def _factor(self, l: int, e: int) -> np.ndarray:
        """fl32(Q[e] / Q[s]) of every node's layer-l row (1.0 where s == e or s < 0)."""
        s = self.stamps[:, l - 1].astype(np.int64)
        live = (s >= 0) & (s != e)
        with np.errstate(divide='ignore', invalid='ignore'):
            f = (self.Q[e, l - 1] / self.Q[np.maximum(s, 0), l - 1]).astype(F32)
        return np.where(live, f, F32(1.0)).astype(F32)

    def current_layer(self, l: int, e: Optional[int] = None) -> np.ndarray:
        """[N, row_stride] values of layer l read at epoch e (default: the current one)."""
        x = self.rows()[:, l, :]
        if not self.lazy or l == 0:
            return x.copy()
        return (x * self._factor(l, self.epoch if e is None else e)[:, None]).astype(F32)

    def current(self, v: int, l: int) -> np.ndarray:
        return self.current_layer(l)[v]

    # ------------------------------------------------------------------ update
    def _advance(self, decay: Optional[np.ndarray]) -> Tuple[int, int, float, bool]:
        """(rc, new epoch, new floor, has_decay) as update_impl decides them before any launch."""
        has = decay is not None and bool(np.any(np.asarray(decay, F32) != F32(1.0)))
        if not (self.lazy and has):
            return 0, self.epoch, self.cum_floor, has
        if self.epoch + 1 >= self.Q.shape[0]:
            return LOG_FULL, self.epoch, self.cum_floor, has
        cmin = 1.0
        for c in np.asarray(decay, F32):
            cmin = float(c) if float(c) < cmin else cmin
        floor = 1.0 if self.epoch == 0 else self.cum_floor
        if self.epoch > 0 and not floor * cmin >= 1e-200:
            return LOG_FULL, self.epoch, self.cum_floor, has
        return 0, self.epoch + 1, floor * cmin, has

    def _chunk_for(self, small: bool, flags: int) -> int:
        if small or (flags & PER_LAYER_WALK):
            return 0
        return effective_chunk(self.giant_chunk)

    def _begin(self, decay):
        rc, e_new, floor, has = self._advance(decay)
        if rc:
            return rc, None
        dec = np.asarray(decay, F32) if decay is not None else np.ones(self.L, F32)
        if self.lazy and e_new != self.epoch:
            self.Q[e_new] = self.Q[self.epoch] * dec.astype(np.float64)
            del self.factors[e_new:]
            self.factors.append(dec.copy())
        if self.lazy:
            P = [self.current_layer(l, e_new) for l in range(self.L + 1)]
        else:
            P = [self.rows()[:, l, :].copy() for l in range(self.L + 1)]
            if has:
                for l in range(1, self.L + 1):
                    P[l] = (P[l] * dec[l - 1]).astype(F32)
        return 0, (P, e_new, floor, has)

    def _finish(self, P, targets, e_new, floor, has) -> None:
        R = self.rows()
        if self.lazy:
            t = np.unique(targets)
            for l in range(1, self.L + 1):
                R[t, l, :] = P[l][t]
            self.stamps[t, :] = e_new
            self.epoch, self.cum_floor = e_new, floor
        else:
            for l in range(1, self.L + 1):
                R[:, l, :] = P[l]

    def update(self, src, dst, times, lam: float, decay: Optional[np.ndarray], flags: int = 0,
               anchor: bool = False):
        """tpn_update (t_last = times[-1], neg_lambda = f32(-lam)).  Returns the return code, and with
        ``anchor=True`` also chain64's (value, magnitude, message count) of every row (or None when refused)."""
        src = np.asarray(src, np.int64)
        dst = np.asarray(dst, np.int64)
        times = np.asarray(times, np.float64)
        pre = self._pre_anchor() if anchor else None
        rc, st = self._begin(decay)
        if rc:
            return (rc, None) if anchor else rc
        P, e_new, floor, has = st
        small = 2 * src.size <= SMALL_MAX_MSGS
        _scatter(P, lam, src, dst, times, self._chunk_for(small, flags))
        tgt = np.concatenate([src, dst])
        oth = np.concatenate([dst, src])
        w = edge_weights(times, times[-1], lam)
        res = self.chain64(pre, tgt, oth, np.concatenate([w, w]), e_new) if anchor else None
        self._finish(P, tgt, e_new, floor, has)
        return (0, res) if anchor else 0

    def update_messages(self, tgt, src, times, t_last: float, lam: float, decay: Optional[np.ndarray],
                        num_local_rows: int, count: Optional[int] = None, device_count: bool = False,
                        flags: int = 0, anchor: bool = False):
        """tpn_update_messages: message m adds source row src[m] into target row tgt[m] with the weight of times[m],
        in the given order; only the first ``count`` messages exist.  Rows >= num_local_rows are read current from
        their own stamps and never written.  ``device_count``: the count is on the device (always the large path)."""
        n = len(tgt) if count is None else int(count)
        tgt = np.asarray(tgt, np.int64)[:n]
        src = np.asarray(src, np.int64)[:n]
        times = np.asarray(times, np.float64)[:n]
        assert np.all(tgt < num_local_rows)
        pre = self._pre_anchor() if anchor else None
        rc, st = self._begin(decay)
        if rc:
            return (rc, None) if anchor else rc
        P, e_new, floor, has = st
        small = not device_count and len(tgt) <= SMALL_MAX_MSGS
        chunk = self._chunk_for(small, flags)
        w = edge_weights(times, t_last, lam)
        o = WalkProjectionOracle.__new__(WalkProjectionOracle)
        o.node_num = self.N
        for l in range(self.L, 0, -1):
            msgs = (P[l - 1][src] * w[:, None]).astype(F32)         # every source read from the pre-batch layer
            if chunk > 0:
                o._chunked_scatter(P[l], tgt, msgs, chunk)
            else:
                np.add.at(P[l], tgt, msgs)                          # sequential, in message order
        res = self.chain64(pre, tgt, src, w, e_new) if anchor else None
        self._finish(P, tgt, e_new, floor, has)
        return (0, res) if anchor else 0

    # ------------------------------------------------------------------ float64 anchor
    def _pre_anchor(self):
        return self.rows().copy(), None if self.stamps is None else self.stamps.copy(), self.epoch

    def _true_factor(self, stamps: np.ndarray, l: int, e: int) -> np.ndarray:
        """prod_{k=s+1..e} c_k[l-1] in float64 for every node, from the list of fp32 factors (1 where s < 0)."""
        out = np.ones(stamps.shape[0])
        for s in np.unique(stamps[:, l - 1]):
            if s < 0:
                continue
            p = 1.0
            for k in range(int(s) + 1, e + 1):
                p *= float(self.factors[k][l - 1])
            out[stamps[:, l - 1] == s] = p
        return out

    def chain64(self, pre, tgt, oth, w, e_new):
        """Float64 truth of an update of the pre-call state ``pre``: per layer l, the target rows
        R = T + sum_j S_j w_j, the magnitude A = |T| + sum_j |S_j w_j| (T: the true decayed target, S_j: the true
        current sources) and the message count m per row.  Returns (R [L, N, rs], A [L, N, rs], m [N])."""
        from scipy.sparse import csr_matrix
        rows, stamps, _ = pre
        N = self.N
        keep = (tgt >= 0) & (tgt < N)
        tgt, oth, w = tgt[keep], oth[keep], np.asarray(w, np.float64)[keep]
        M = csr_matrix((w, (tgt, oth)), shape=(N, N))
        Ma = csr_matrix((np.abs(w), (tgt, oth)), shape=(N, N))
        true = [rows[:, 0, :].astype(np.float64)]
        for l in range(1, self.L + 1):
            true.append(rows[:, l, :].astype(np.float64) * self._true_factor(stamps, l, e_new)[:, None])
        R = np.zeros((self.L, N, self.rs))
        A = np.zeros((self.L, N, self.rs))
        for l in range(1, self.L + 1):
            R[l - 1] = true[l] + M @ true[l - 1]
            A[l - 1] = np.abs(true[l]) + Ma @ np.abs(true[l - 1])
        return R, A, np.bincount(tgt, minlength=N)

    # ------------------------------------------------------------------ readers
    def gather(self, ids) -> np.ndarray:
        """tpn_gather: [L+1, n, dim], negative ids wrap."""
        ids = np.asarray(ids, np.int64) % self.N
        return np.stack([self.current_layer(l)[ids, :self.d] for l in range(self.L + 1)])

    def gather_blocks(self, ids) -> np.ndarray:
        """tpn_gather_blocks: [n, node_stride] whole node blocks, rows 1..L current, everything else as stored."""
        ids = np.asarray(ids, np.int64) % self.N
        out = self.data[ids].copy()
        H = self.L + 1
        blk = out[:, :H * self.rs].reshape(len(ids), H, self.rs)
        for l in range(1, H):
            blk[:, l, :] = self.current_layer(l)[ids]
        return out

    def materialize(self) -> None:
        """tpn_materialize: every row with 0 <= stamp < epoch brought current and stamped; no-op at epoch 0."""
        if not self.lazy or self.epoch == 0:
            return
        R = self.rows()
        for l in range(1, self.L + 1):
            R[:, l, :] = self.current_layer(l)
        live = self.stamps >= 0
        self.stamps[live] = self.epoch

    def reset_epoch(self) -> None:
        """tpn_reset_epoch: stamps >= 0 -> 0, epoch 0, cum_floor 1.0 (the log's rows stay as they are)."""
        if not self.lazy:
            return
        self.stamps[self.stamps >= 0] = 0
        self.epoch = 0
        self.cum_floor = 1.0
        del self.factors[1:]


def anchor_bound(A: np.ndarray, m: np.ndarray, max_gap: int, max_abs: float) -> np.ndarray:
    """Bound on |kernel - chain64| of a target row with m messages (derivation: tests/test_gpu_update_lazy.py)."""
    u = 2.0 ** -24
    k = m + 3
    gamma = k * u / (1 - k * u)
    eta = (2 * max_gap + m + 4) * 2.0 ** -52
    return (gamma + eta) * A + (m + 1) * (max_abs + 2.0) * 2.0 ** -149

