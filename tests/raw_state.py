"""Hand-built tpn_state_t's for the GPU suites: any legal layout, hand-made stamps and decay logs, and thin wrappers of
the raw C ABI that synchronise and return host copies.

Layout conventions: rows [N, L+1, d] go to ``data[u * node_stride + l * row_stride + k]``; the pad columns
[d, row_stride) are 0; the node_stride gap and one node past num_nodes are NaN, so a kernel that reads outside a
node's L+1 rows shows NaN, and one that writes there changes bits that are compared.
"""
import ctypes

import numpy as np
import torch

from tpnet_b200 import _lib

DEV = 'cuda:0'
FACTOR_SET = np.float32([0.5, 0.37, 0.81, 0.62, 0.9])      # per-epoch fp32 factors far from 1


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dev(x, dtype):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).to(DEV)


class RawState:
    """A tpn_state_t over `rows` ([N, L+1, d] float32, the values in memory) in the given layout.

    ``lazy=True`` with no ``stamps`` / ``factors``: ``epoch`` random factors from FACTOR_SET and random stamps (the
    pair-wise suite's states).  ``stamps`` [N, L] and ``factors`` [epoch, L] (fp32; Q is their f64 running product)
    give the lazy bookkeeping explicitly; rows whose stamp is -1 are zeroed (the contract of a never-written row).
    ``log_capacity`` rows are allocated for the log (rows past the epoch hold -7.0 until an update writes them)."""

    def __init__(self, rows, rs, ns, lazy=False, rng=None, epoch=6, stamps=None, factors=None, log_capacity=None,
                 giant_chunk=0, cum_floor=None):
        N, H, d = rows.shape
        L = H - 1
        assert rs % 4 == 0 and rs >= d and ns % 4 == 0 and ns >= H * rs
        self.N, self.L, self.d, self.rs, self.ns = N, L, d, rs, ns
        host = np.full((N + 1, ns), np.nan, np.float32)          # gap and node N: NaN
        blk = host[:N, :H * rs].reshape(N, H, rs)
        blk[:] = 0
        blk[:, :, :d] = rows
        eff = rows.astype(np.float32).copy()
        self.stamps = self.qlog = None
        self.epoch = 0
        self.cum_floor = 1.0
        self.factors = np.zeros((0, L), np.float32)
        lazy = lazy or stamps is not None
        if lazy:
            rng = rng or np.random.default_rng(0)
            if factors is None:
                # per-epoch fp32 factors far from 1; Q[e] = product of the factors of epochs 1..e (f64), Q[0] = 1
                factors = rng.choice(FACTOR_SET, size=(epoch, L))
            factors = np.asarray(factors, np.float32).reshape(-1, L)
            epoch = len(factors)
            q = np.vstack([np.ones((1, L)), np.cumprod(factors.astype(np.float64), axis=0)])
            if stamps is None:
                stamps = rng.integers(-1, epoch + 1, (N, L)).astype(np.int32)
                stamps[rng.random((N, L)) < 0.3] = rng.integers(0, 2)     # gaps of several epochs
            stamps = np.asarray(stamps, np.int32).reshape(N, L)
            for l in range(1, H):
                dead = stamps[:, l - 1] < 0                            # never written: all zero by contract
                blk[dead, l, :] = 0
                eff[dead, l, :] = 0
                s = np.maximum(stamps[:, l - 1], 0)
                f = np.where(stamps[:, l - 1] >= 0, (q[epoch, l - 1] / q[s, l - 1]).astype(np.float32), 1.0)
                eff[:, l, :] = eff[:, l, :] * f.astype(np.float32)[:, None]     # fl32(x * fl32(Q[e] / Q[s]))
            cap = epoch + 1 if log_capacity is None else int(log_capacity)
            qfull = np.full((cap, L), -7.0)
            qfull[:epoch + 1] = q
            self.factors = factors
            self.stamps = torch.from_numpy(stamps.copy()).to(DEV)
            self.qlog = torch.from_numpy(qfull).to(DEV)
            self.epoch = epoch
            self.cum_floor = float(q.min()) if cum_floor is None else float(cum_floor)
        self.eff = eff
        self.host0 = host.copy()
        self.data = torch.from_numpy(host.reshape(-1)).to(DEV)
        self.err = torch.zeros(1, dtype=torch.int32, device=DEV)
        self.ws = None
        self.st = _lib.TpnState(
            data=self.data.data_ptr(), num_nodes=N, num_layer=L, dim=d, row_stride=rs, node_stride=ns,
            stamps=None if self.stamps is None else self.stamps.data_ptr(),
            decay_log=None if self.qlog is None else self.qlog.data_ptr(),
            log_capacity=0 if self.qlog is None else self.qlog.shape[0], epoch=self.epoch, cum_floor=self.cum_floor,
            err_flag=self.err.data_ptr(), giant_chunk=int(giant_chunk))

    # ------------------------------------------------------------------ snapshots of the device state
    def model_args(self):
        """Keyword arguments of oracle.lazy_decay.LazyDecayModel for this state as built."""
        return dict(data=self.host0, num_nodes=self.N, num_layer=self.L, dim=self.d, row_stride=self.rs,
                    node_stride=self.ns, stamps=None if self.stamps is None else self.stamps.cpu().numpy(),
                    factors=self.factors if self.stamps is not None else None,
                    log_capacity=0 if self.qlog is None else self.qlog.shape[0],
                    cum_floor=self.st.cum_floor, giant_chunk=self.st.giant_chunk)

    def host(self):
        """(data [N+1, ns], stamps or None, log or None, epoch, cum_floor, err) after a synchronise."""
        torch.cuda.synchronize()
        return (self.data.cpu().numpy().reshape(-1, self.ns).copy(),
                None if self.stamps is None else self.stamps.cpu().numpy().copy(),
                None if self.qlog is None else self.qlog.cpu().numpy().copy(),
                int(self.st.epoch), float(self.st.cum_floor), int(self.err.item()))

    # ------------------------------------------------------------------ the C ABI
    def workspace(self, batch):
        need = _lib.load().tpn_update_workspace_bytes(ctypes.byref(self.st), int(batch))
        if self.ws is None or self.ws.numel() < need:
            self.ws = torch.empty(max(int(need), 1 << 16), dtype=torch.uint8, device=DEV)
        return self.ws

    @staticmethod
    def _decay(decay):
        if decay is None:
            return None
        return (ctypes.c_float * len(decay))(*[float(np.float32(c)) for c in decay])

    def update(self, src, dst, t, lam, decay, phase=None, stream=None, keep=None):
        """tpn_update (phase None) or tpn_update_phase with t_last = t[-1]; returns the C return code.  `keep`:
        a list that holds the device arrays of a split call until its second half ran."""
        src_d, dst_d, t_d = _dev(src, np.int64), _dev(dst, np.int64), _dev(t, np.float64)
        ws = self.workspace(len(src))
        if stream is not None:
            torch.cuda.synchronize()                 # the uploads above ran on the current stream
        args = (ctypes.byref(self.st), src_d.data_ptr(), dst_d.data_ptr(), t_d.data_ptr(), len(src),
                float(np.float64(t[-1])), float(np.float32(-lam)), self._decay(decay), ws.data_ptr(), ws.numel(),
                self.err.data_ptr(), stream if stream is not None else _stream())
        lib = _lib.load()
        rc = lib.tpn_update(*args) if phase is None else lib.tpn_update_phase(*args, int(phase))
        if keep is not None:
            keep.append((src_d, dst_d, t_d))
        torch.cuda.synchronize()
        return rc

    def update_messages(self, tgt, src, t, t_last, lam, decay, num_local_rows, count=None):
        """tpn_update_messages; `count` (< len(tgt)): the real number of messages, passed on the device."""
        tgt_d, src_d, t_d = _dev(tgt, np.int64), _dev(src, np.int64), _dev(t, np.float64)
        n = len(tgt)
        cnt = None if count is None else torch.tensor([int(count)], dtype=torch.int32, device=DEV)
        ws = self.workspace((n + 1) // 2)
        rc = _lib.load().tpn_update_messages(ctypes.byref(self.st), tgt_d.data_ptr(), src_d.data_ptr(),
                                             t_d.data_ptr(), n, None if cnt is None else cnt.data_ptr(),
                                             int(num_local_rows), float(t_last), float(np.float32(-lam)),
                                             self._decay(decay), ws.data_ptr(), ws.numel(), self.err.data_ptr(),
                                             _stream())
        torch.cuda.synchronize()
        return rc

    def gather(self, ids):
        ids_d = _dev(ids, np.int64)
        out = torch.full((self.L + 1, len(ids), self.d), -7.0, device=DEV)
        rc = _lib.load().tpn_gather(ctypes.byref(self.st), ids_d.data_ptr(), len(ids), out.data_ptr(), _stream())
        assert rc == 0, rc
        torch.cuda.synchronize()
        return out.cpu().numpy()

    def gather_blocks(self, ids):
        ids_d = _dev(ids, np.int64)
        out = torch.full((len(ids), self.ns), -7.0, device=DEV)
        rc = _lib.load().tpn_gather_blocks(ctypes.byref(self.st), ids_d.data_ptr(), len(ids), out.data_ptr(),
                                           _stream())
        assert rc == 0, rc
        torch.cuda.synchronize()
        return out.cpu().numpy()

    def materialize(self):
        rc = _lib.load().tpn_materialize(ctypes.byref(self.st), _stream())
        torch.cuda.synchronize()
        return rc

    def reset_epoch(self):
        rc = _lib.load().tpn_reset_epoch(ctypes.byref(self.st), _stream())
        torch.cuda.synchronize()
        return rc

    # ------------------------------------------------------------------ pair-wise calls
    def pairwise(self, a, b, log):
        n = len(a)
        out = torch.full((n, 4 * (self.L + 1) ** 2), -7.0, device=DEV)
        ad, bd = (torch.from_numpy(np.asarray(x, np.int64)).to(DEV) for x in (a, b))
        rc = _lib.load().tpn_pairwise(ctypes.byref(self.st), ad.data_ptr(), bd.data_ptr(), n, None, int(log),
                                      out.data_ptr(), _stream())
        assert rc == 0, rc
        torch.cuda.synchronize()
        assert int(self.err.item()) == 0
        return out.cpu().numpy()

    def neighbors(self, nbr, src, dst, log):
        m, K = nbr.shape
        F = 4 * (self.L + 1) ** 2
        out = torch.full((m, K, 2, F), -7.0, device=DEV)
        t = [torch.from_numpy(np.ascontiguousarray(x, np.int64)).to(DEV) for x in (nbr, src, dst)]
        rc = _lib.load().tpn_pairwise_neighbors(ctypes.byref(self.st), t[0].data_ptr(), t[1].data_ptr(),
                                                t[2].data_ptr(), m, K, int(log), out.data_ptr(), _stream())
        torch.cuda.synchronize()
        if rc == 0:
            assert int(self.err.item()) == 0
        return rc, out.cpu().numpy()

    def reference(self, a, b, exact_nonfinite=False):
        """(G, sum |x_i y_i|) in float64 for pairs (a, b): [n, R*R] each.  Negative ids wrap."""
        x = np.concatenate([self.eff[np.asarray(a) % self.N], self.eff[np.asarray(b) % self.N]], axis=1)
        x = x.astype(np.float64)
        ax = np.abs(x)
        n = len(x)
        if exact_nonfinite:                      # plain loops, IEEE semantics for inf * 0 and inf - inf
            with np.errstate(invalid='ignore', over='ignore'):
                g = np.einsum('nrd,ncd->nrc', x, x, optimize=False)
                s = np.einsum('nrd,ncd->nrc', ax, ax, optimize=False)
        else:
            g = x @ x.transpose(0, 2, 1)
            s = ax @ ax.transpose(0, 2, 1)
        return g.reshape(n, -1), s.reshape(n, -1)
