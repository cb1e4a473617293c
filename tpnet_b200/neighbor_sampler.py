"""GPU version of the reference's `recent` historical-neighbour sampler
(``/root/reference/utils/utils.py:70-224`` with ``sample_neighbor_strategy='recent'``; SURVEY.md 8(f) N2).

Same constructor data and the same ``get_historical_neighbors(node_ids, node_interact_times,
num_neighbors)`` call and results as the reference class: for every (node, time) the most recent
``num_neighbors`` interactions strictly before ``time``, written to the back of zero rows — neighbour
ids, edge ids (int64) and times (float64), ``[n, num_neighbors]`` each.  The adjacency lives on the
device as one CSR (built here once, per node stably sorted by timestamp); a query batch is one kernel
(``tpn_sampler_recent``).  With ``as_tensors=True`` the results stay on the device and feed
``RandomProjectionModule.get_neighbor_pair_wise_feature`` without a host round trip.
``StreamingRecentSampler`` gives the same answers without the whole edge list: it is fed batch by batch
(``push``) and keeps O(num_nodes * max_neighbors) state on the device (``tpn_stream_sampler_*``).
``ShardedStreamingSampler`` splits that state over the GPUs of a node-sharded job (``tpn_stream_shard_*``).
Only the `recent` strategy exists (what TPNet uses); there is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Tuple, Union

import numpy as np
import torch

from . import _lib
from .peer import PeerShardMember, rows_on_rank

ArrayOrTensor = Union[np.ndarray, torch.Tensor]


def build_recent_csr(src: np.ndarray, dst: np.ndarray, eid: np.ndarray, t: np.ndarray, num_nodes: int):
    """(offsets[num_nodes+1], neighbour ids, edge ids, times) of the time-sorted adjacency.
    utils/utils.py:248-251: per edge, (dst, eid, t) joins src's list, then (src, eid, t) joins dst's list;
    :107-113: every list is stably sorted by time."""
    owner = np.stack([src, dst], axis=1).reshape(-1)
    other = np.stack([dst, src], axis=1).reshape(-1)
    e2, t2 = np.repeat(eid, 2), np.repeat(t, 2)
    order = np.lexsort((np.arange(owner.shape[0]), t2, owner))
    offsets = np.zeros(num_nodes + 1, dtype=np.int64)
    np.cumsum(np.bincount(owner, minlength=num_nodes), out=offsets[1:])
    return offsets, other[order], e2[order], t2[order]


class RecentNeighborSampler:
    def __init__(self, src_node_ids: np.ndarray, dst_node_ids: np.ndarray, edge_ids: np.ndarray,
                 node_interact_times: np.ndarray, device: Union[str, torch.device], num_nodes: int = None):
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise RuntimeError('tpnet_b200.RecentNeighborSampler samples on CUDA only (no CPU fallback)')
        src = np.asarray(src_node_ids, dtype=np.int64)
        dst = np.asarray(dst_node_ids, dtype=np.int64)
        eid = np.asarray(edge_ids, dtype=np.int64)
        t = np.asarray(node_interact_times, dtype=np.float64)
        if not (len(src) == len(dst) == len(eid) == len(t)):
            raise ValueError('src, dst, edge id and time arrays must have the same length')
        top = int(max(src.max(initial=0), dst.max(initial=0))) + 1
        self.num_nodes = top if num_nodes is None else int(num_nodes)
        if self.num_nodes < top or (len(src) and min(src.min(), dst.min()) < 0):
            raise IndexError('node id out of range')
        offsets, nbr, eids, times = build_recent_csr(src, dst, eid, t, self.num_nodes)
        self.device = dev
        self._offsets = torch.from_numpy(offsets).to(dev)
        self._nbr = torch.from_numpy(nbr).to(dev)
        self._eid = torch.from_numpy(eids).to(dev)
        self._times = torch.from_numpy(times).to(dev)
        if self._nbr.numel() == 0:                          # keep valid base pointers for an empty graph
            self._nbr = torch.zeros(1, dtype=torch.int64, device=dev)
            self._eid = torch.zeros(1, dtype=torch.int64, device=dev)
            self._times = torch.zeros(1, dtype=torch.float64, device=dev)
        self.sample_neighbor_strategy = 'recent'
        self.seed = None                                    # attributes / methods the reference's callers touch

    def reset_random_state(self) -> None:
        """`recent` sampling is deterministic: nothing to reset (utils/utils.py:316-321 exists for the random strategies)."""

    def _to_device(self, a: ArrayOrTensor, dtype: torch.dtype) -> torch.Tensor:
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=dtype).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64 if dtype == torch.int64 else np.float64)
                                ).to(self.device)

    def get_historical_neighbors(self, node_ids: ArrayOrTensor, node_interact_times: ArrayOrTensor,
                                 num_neighbors: int = 20, as_tensors: bool = False
                                 ) -> Tuple[ArrayOrTensor, ArrayOrTensor, ArrayOrTensor]:
        """utils/utils.py:160-224 for the `recent` strategy."""
        assert num_neighbors > 0, 'Number of sampled neighbors for each node should be greater than 0!'
        n = int(len(node_ids))
        if len(node_interact_times) != n:
            raise ValueError('node ids and times must have the same length')
        if not isinstance(node_ids, torch.Tensor) and n:
            ids = np.asarray(node_ids)
            if ids.min() < 0 or ids.max() >= self.num_nodes:     # the reference indexes a per-node list (utils.py:177)
                raise IndexError(f'node id out of range for a sampler over {self.num_nodes} nodes')
        qn = self._to_device(node_ids, torch.int64).reshape(-1)
        qt = self._to_device(node_interact_times, torch.float64).reshape(-1)
        out_n = torch.empty(n, num_neighbors, dtype=torch.int64, device=self.device)
        out_e = torch.empty(n, num_neighbors, dtype=torch.int64, device=self.device)
        out_t = torch.empty(n, num_neighbors, dtype=torch.float64, device=self.device)
        if n:
            dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
            stream = torch._C._cuda_getCurrentRawStream(dev_index)
            rc = _lib.load().tpn_sampler_recent(self._offsets.data_ptr(), self._nbr.data_ptr(), self._eid.data_ptr(),
                                                self._times.data_ptr(), self.num_nodes, qn.data_ptr(), qt.data_ptr(), n,
                                                int(num_neighbors), out_n.data_ptr(), out_e.data_ptr(), out_t.data_ptr(),
                                                stream)
            if rc:
                _lib.check(rc, 'tpn_sampler_recent')
        if as_tensors:
            return out_n, out_e, out_t
        return out_n.cpu().numpy(), out_e.cpu().numpy(), out_t.cpu().numpy()


class StreamingRecentSampler:
    """The `recent` sampler fed batch by batch: ``push(src, dst, edge_ids, t)`` appends one chronological batch,
    and ``get_historical_neighbors`` answers exactly what ``RecentNeighborSampler`` built over every edge pushed so
    far answers, for any query whose time is >= the node's newest time before the latest push.  TPNet's loop always
    meets that condition: push the batch, query its src / dst / negatives at the batch's times, push the next.  A query
    that breaks it cannot be answered exactly: it is flagged, and ``check_errors()`` raises.

    No adjacency of the whole stream is built: the state is two lists of ``max_neighbors`` entries per node on the
    device (48 * max_neighbors + 16 bytes per node) plus the latest batch (``tpn_stream_sampler_*``,
    include/tpnet_b200.h), so streams that never exist as a whole edge list can be sampled.  ``push`` and
    ``get_historical_neighbors`` with CUDA-tensor arguments never synchronise or allocate inside a CUDA-graph capture
    (push batches of at most ``max_batch`` edges there; larger batches grow the buffers outside captures).
    Host (numpy) arguments are validated before anything is launched; CUDA-tensor arguments are validated on the
    device (the offending edge or query is dropped and flagged)."""

    def __init__(self, num_nodes: int, max_neighbors: int, device: Union[str, torch.device], max_batch: int = 200_000):
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise RuntimeError('tpnet_b200.StreamingRecentSampler samples on CUDA only (no CPU fallback)')
        if num_nodes < 1 or num_nodes > 0xffffffff:
            raise ValueError('num_nodes must be in [1, 2**32)')
        if max_neighbors < 1:
            raise ValueError('max_neighbors must be positive')
        if max_batch < 1:
            raise ValueError('max_batch must be positive')
        if dev.index is None:
            dev = torch.device('cuda', torch.cuda.current_device())
        self.device = dev
        self.num_nodes = int(num_nodes)
        self.max_neighbors = int(max_neighbors)
        self._alloc_tables()
        i32, f64 = torch.int32, torch.float64
        self._pend_count = torch.zeros(1, dtype=i32, device=dev)
        self._last_time = torch.empty(1, dtype=f64, device=dev)
        self._err = torch.zeros(1, dtype=i32, device=dev)
        self.max_batch = 0
        self._ws = None
        self._grow(int(max_batch))
        self.sample_neighbor_strategy = 'recent'
        self.seed = None
        self.reset()

    def _alloc_tables(self) -> None:
        """The lists, counts and newest times of every node (num_nodes rows)."""
        N, C, dev = self.num_nodes, self.max_neighbors, self.device
        i64, f64, i32 = torch.int64, torch.float64, torch.int32
        self._lists = {k: torch.empty(N, C, dtype=d, device=dev) for k, d in
                       (('all_nbr', i64), ('all_eid', i64), ('all_t', f64),
                        ('old_nbr', i64), ('old_eid', i64), ('old_t', f64))}
        self._all_cnt = torch.empty(N, dtype=i32, device=dev)
        self._old_cnt = torch.empty(N, dtype=i32, device=dev)
        self._newest = torch.empty(N, dtype=f64, device=dev)

    def _grow(self, max_batch: int) -> None:
        """Pending arrays for 2 * max_batch entries (the current pending batch is kept) and the push workspace."""
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError(f'StreamingRecentSampler: a batch of {max_batch} edges exceeds max_batch='
                               f'{self.max_batch} inside a CUDA-graph capture; construct it with a larger max_batch')
        dev, cap = self.device, 2 * max_batch
        pend = {'pend_node': torch.empty(cap, dtype=torch.int32, device=dev),     # uint32 keys in the C struct
                'pend_nbr': torch.empty(cap, dtype=torch.int64, device=dev),
                'pend_eid': torch.empty(cap, dtype=torch.int64, device=dev),
                'pend_t': torch.empty(cap, dtype=torch.float64, device=dev)}
        if self.max_batch:
            for k, v in pend.items():
                v[:2 * self.max_batch].copy_(self._pend[k])
        self._pend = pend
        need = int(_lib.load().tpn_stream_sampler_workspace_bytes(max_batch))
        self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        self.max_batch = max_batch
        self._c = _lib.TpnStreamSampler(
            num_nodes=self.num_nodes, capacity=self.max_neighbors, max_batch=max_batch,
            **{k: v.data_ptr() for k, v in self._lists.items()}, **{k: v.data_ptr() for k, v in pend.items()},
            all_cnt=self._all_cnt.data_ptr(), old_cnt=self._old_cnt.data_ptr(), newest=self._newest.data_ptr(),
            pend_count=self._pend_count.data_ptr(), last_time=self._last_time.data_ptr(), err_flag=self._err.data_ptr())

    def _stream(self) -> int:
        return torch._C._cuda_getCurrentRawStream(self.device.index)

    def _to_device(self, a: ArrayOrTensor, dtype: torch.dtype) -> torch.Tensor:
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=dtype).contiguous().reshape(-1)
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64 if dtype == torch.int64 else np.float64)
                                ).reshape(-1).to(self.device)

    def reset_random_state(self) -> None:
        """`recent` sampling is deterministic: nothing to reset (as RecentNeighborSampler)."""

    def reset(self) -> None:
        """Forget every pushed edge (a new epoch restarts the stream); clears the error flag."""
        _lib.check(_lib.load().tpn_stream_sampler_reset(ctypes.byref(self._c), self._stream()),
                   'tpn_stream_sampler_reset')
        self._last_host = -np.inf           # last pushed time, when the host knows it (numpy pushes)

    def push(self, src_node_ids: ArrayOrTensor, dst_node_ids: ArrayOrTensor, edge_ids: ArrayOrTensor,
             node_interact_times: ArrayOrTensor) -> None:
        """Appends one batch; its times are non-decreasing and >= every earlier pushed time."""
        n = int(len(src_node_ids))
        if not (len(dst_node_ids) == len(edge_ids) == len(node_interact_times) == n):
            raise ValueError('src, dst, edge id and time arrays must have the same length')
        if n == 0:
            return
        host = [not isinstance(a, torch.Tensor) for a in (src_node_ids, dst_node_ids, node_interact_times)]
        if host[0] or host[1]:
            for a, h in zip((src_node_ids, dst_node_ids), host):
                if h:
                    ids = np.asarray(a)
                    if ids.min() < 0 or ids.max() >= self.num_nodes:
                        raise IndexError(f'node id out of range for a sampler over {self.num_nodes} nodes')
        if host[2]:
            t = np.asarray(node_interact_times, dtype=np.float64)
            if (n > 1 and bool((np.diff(t) < 0).any())) or t[0] < self._last_host:
                raise ValueError('pushed times must be non-decreasing and >= every earlier pushed time')
            self._last_host = float(t[-1])
        else:
            self._last_host = -np.inf           # unknown on the host: the device checks the order
        if n > self.max_batch:
            self._grow(n)
        src = self._to_device(src_node_ids, torch.int64)
        dst = self._to_device(dst_node_ids, torch.int64)
        eid = self._to_device(edge_ids, torch.int64)
        t = self._to_device(node_interact_times, torch.float64)
        self._push_launch(src, dst, eid, t, n)

    def _push_launch(self, src: torch.Tensor, dst: torch.Tensor, eid: torch.Tensor, t: torch.Tensor, n: int) -> None:
        rc = _lib.load().tpn_stream_sampler_push(ctypes.byref(self._c), src.data_ptr(), dst.data_ptr(), eid.data_ptr(),
                                                 t.data_ptr(), n, self._ws.data_ptr(), self._ws.numel(), self._stream())
        if rc:
            _lib.check(rc, 'tpn_stream_sampler_push')

    def get_historical_neighbors(self, node_ids: ArrayOrTensor, node_interact_times: ArrayOrTensor,
                                 num_neighbors: int = 20, as_tensors: bool = False
                                 ) -> Tuple[ArrayOrTensor, ArrayOrTensor, ArrayOrTensor]:
        """Same call and results as ``RecentNeighborSampler.get_historical_neighbors`` over the pushed edges.
        With numpy results the error flag is checked too (``check_errors``)."""
        n = self._check_query(node_ids, node_interact_times, num_neighbors)
        qn = self._to_device(node_ids, torch.int64)
        qt = self._to_device(node_interact_times, torch.float64)
        out_n = torch.empty(n, num_neighbors, dtype=torch.int64, device=self.device)
        out_e = torch.empty(n, num_neighbors, dtype=torch.int64, device=self.device)
        out_t = torch.empty(n, num_neighbors, dtype=torch.float64, device=self.device)
        if n:
            rc = _lib.load().tpn_stream_sampler_query(ctypes.byref(self._c), qn.data_ptr(), qt.data_ptr(), n,
                                                      int(num_neighbors), out_n.data_ptr(), out_e.data_ptr(),
                                                      out_t.data_ptr(), self._stream())
            if rc:
                _lib.check(rc, 'tpn_stream_sampler_query')
        if as_tensors:
            return out_n, out_e, out_t
        res = out_n.cpu().numpy(), out_e.cpu().numpy(), out_t.cpu().numpy()
        self.check_errors()
        return res

    def _check_query(self, node_ids: ArrayOrTensor, node_interact_times: ArrayOrTensor, num_neighbors: int) -> int:
        """Host-side checks of a query call (host ids against num_nodes, before anything is launched); its length."""
        assert num_neighbors > 0, 'Number of sampled neighbors for each node should be greater than 0!'
        if num_neighbors > self.max_neighbors:
            raise ValueError(f'num_neighbors={num_neighbors} exceeds max_neighbors={self.max_neighbors}')
        n = int(len(node_ids))
        if len(node_interact_times) != n:
            raise ValueError('node ids and times must have the same length')
        if not isinstance(node_ids, torch.Tensor) and n:
            ids = np.asarray(node_ids)
            if ids.min() < 0 or ids.max() >= self.num_nodes:
                raise IndexError(f'node id out of range for a sampler over {self.num_nodes} nodes')
        return n

    def check_errors(self) -> None:
        """Synchronises; raises (and clears the flag) if a device-resident input was flagged since the last check:
        IndexError for a node id outside [0, num_nodes), ValueError for a pushed time out of order or a query before
        the node's newest time of the previous batches."""
        code = int(self._err.item())
        if code == 0:
            return
        self._err.zero_()
        if code & _lib.STREAM_ERR_INDEX:
            raise IndexError(f'node id out of range for a sampler over {self.num_nodes} nodes (dropped)')
        if code & _lib.STREAM_ERR_ORDER:
            raise ValueError('pushed times decreased (the edge was dropped; answers are unspecified until reset())')
        raise ValueError('a query asked for a time before the newest time its node had before the latest push: '
                         'not answerable from the streaming state (a zero row was returned)')


class ShardedStreamingSampler(StreamingRecentSampler, PeerShardMember):
    """``StreamingRecentSampler`` over the node-sharded layout of ``ShardedRandomProjection``: node ``u``'s lists live
    on rank ``u % world`` at local row ``u // world``, so a rank holds ``ceil(num_nodes / world) + cache_rows`` list
    rows instead of ``num_nodes`` (``tpn_stream_shard_*``, include/tpnet_b200.h).

    ``push`` takes the replicated batch on every rank; each rank keeps the whole batch pending and folds only the nodes
    it owns.  ``get_historical_neighbors(node_ids, times, K)`` takes the replicated query list and answers the rows of
    this rank's positional slice ``[r * per, min((r + 1) * per, m))``, ``per = ceil(m / world)`` — the split
    ``ShardedRandomProjection`` gives the encoder call over the same rows, so the result feeds
    ``get_neighbor_pair_wise_feature(..., sliced_neighbors=True)`` with no all-gather.  It returns ``(positions, nbr,
    eid, t)``; the rows are bit-equal to ``StreamingRecentSampler``'s rows at those positions.  Remote lists are
    routed through the sampler's own mark table into ``cache_rows`` cache rows and pulled out of the owners' memory; a
    cached list stays valid until the next push.  Every rank calls ``push``, ``get_historical_neighbors`` and
    ``reset`` together (they may take a rank barrier).

    ``peers`` / ``group`` as for ``ShardedRandomProjection``; with a ``LocalPeerGroup`` (several ranks in one process)
    construct every rank, then ``connect()`` each.  World 1 is ``StreamingRecentSampler`` itself (no cache rows).
    ``exchange='nccl'`` at world > 1 raises ``NotImplementedError``: the sampler has only the peer data plane."""

    def __init__(self, num_nodes: int, max_neighbors: int, device: Union[str, torch.device], max_batch: int = 200_000,
                 peers=None, group=None, cache_rows: int = 1 << 16, exchange: str = 'auto'):
        if exchange not in ('auto', 'peer', 'nccl'):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        self._join(num_nodes, peers, group)
        if self.world > 1 and exchange == 'nccl':
            raise NotImplementedError("ShardedStreamingSampler with world > 1 needs exchange='peer' "
                                      "(the sampler pulls remote lists out of peer memory; it has no 'nccl' data plane)")
        if self.world > 1 and num_nodes > 0x7fffffff:
            raise ValueError('a sharded sampler routes node ids through int32 mark tables: num_nodes must be < 2**31')
        if cache_rows < 0:
            raise ValueError('cache_rows must be >= 0')
        self.cache_rows = int(cache_rows) if self.world > 1 else 0
        super().__init__(num_nodes, max_neighbors, device, max_batch)

    # ------------------------------------------------------------------ set-up
    def _alloc_tables(self) -> None:
        if self.world == 1:
            return super()._alloc_tables()
        dev, C = self.device, self.max_neighbors
        rows = self.n_local + self.cache_rows
        # one peer-visible buffer of the same size on every rank (symmetric memory needs it), the nine tables at the
        # same offsets everywhere: rank q's tables are its base pointer plus these offsets
        alloc = rows_on_rank(self.num_nodes, self.world, 0) + self.cache_rows
        sizes = [alloc * C * 8] * 6 + [alloc * 4, alloc * 4, alloc * 8]
        self._offsets, off = [], 0
        for b in sizes:
            self._offsets.append(off)
            off += (b + 255) // 256 * 256
        buf = self._peer_buffer('sampler_lists', off, dev)
        raw = buf.tensor((buf.nbytes,), torch.uint8)

        def view(i, dtype, shape):
            n = 1
            for s in shape:
                n *= s
            o = self._offsets[i]
            return raw[o:o + n * (8 if dtype != torch.int32 else 4)].view(dtype).view(*shape)

        i64, f64, i32 = torch.int64, torch.float64, torch.int32
        names = _lib.STREAM_PEER_TABLES
        self._lists = {k: view(i, d, (rows, C)) for i, (k, d) in enumerate(zip(names[:6], (i64, i64, f64) * 2))}
        self._all_cnt = view(6, i32, (rows,))
        self._old_cnt = view(7, i32, (rows,))
        self._newest = view(8, f64, (rows,))
        self._cs = _lib.TpnStreamShard()             # its `shard` is the tpn_shard_t of the base class (one struct)
        self._init_shard(dev, self.num_nodes, self.cache_rows, 'sampler_flags', self._cs.shard)

    @property
    def _counters(self) -> torch.Tensor:
        """The routing counters of the shard (``_shard_tensors['counters']``; ``SHARD_CTR_*`` index them)."""
        return self._shard_tensors['counters']

    def _grow(self, max_batch: int) -> None:
        super()._grow(max_batch)
        if self.world > 1:
            self._cs.local = self._c

    def _connect_tables(self, bases):
        lists = torch.tensor([b + o for b in bases['sampler_lists'] for o in self._offsets], dtype=torch.int64,
                             device=self.device)
        self._cs.peer_lists = lists.data_ptr()
        return {'lists': lists}

    # ------------------------------------------------------------------ API
    def reset(self) -> None:
        """Forget every pushed edge on every rank (collective at world > 1); clears the error flags."""
        if self.world == 1:
            return super().reset()
        if self._connected:
            self._barrier()              # no peer is still pulling the lists this rewrites
        _lib.check(_lib.load().tpn_stream_shard_reset(ctypes.byref(self._cs), self._stream()), 'tpn_stream_shard_reset')
        self._dirty = True
        self._last_host = -np.inf

    def _push_launch(self, src, dst, eid, t, n: int) -> None:
        if self.world == 1:
            return super()._push_launch(src, dst, eid, t, n)
        self._barrier()                  # every peer has finished pulling the lists this fold rewrites
        rc = _lib.load().tpn_stream_shard_push(ctypes.byref(self._cs), src.data_ptr(), dst.data_ptr(), eid.data_ptr(),
                                               t.data_ptr(), n, self._ws.data_ptr(), self._ws.numel(), self._stream())
        if rc:
            _lib.check(rc, 'tpn_stream_shard_push')
        self._dirty = True

    def get_historical_neighbors(self, node_ids: ArrayOrTensor, node_interact_times: ArrayOrTensor,
                                 num_neighbors: int = 20, as_tensors: bool = False):
        """This rank's slice of ``StreamingRecentSampler.get_historical_neighbors`` over the replicated call:
        ``(positions, nbr [rows, K], eid [rows, K], t [rows, K])`` (numpy, or CUDA tensors with ``as_tensors``).
        Host ids of the whole call are checked on every rank before anything is launched."""
        m = self._check_query(node_ids, node_interact_times, num_neighbors)
        per, lo, hi = self.row_split(m)
        keep = self._positions(lo, hi, self.device)
        if self.world == 1:
            res = super().get_historical_neighbors(node_ids, node_interact_times, num_neighbors, as_tensors)
            return (keep if as_tensors else keep.cpu().numpy(),) + tuple(res)
        n, K, dev = hi - lo, int(num_neighbors), self.device
        lib = _lib.load()
        qn = self._to_device(node_ids[lo:hi], torch.int64)
        qt = self._to_device(node_interact_times[lo:hi], torch.float64)
        rows = torch.empty(n, dtype=torch.int64, device=dev)
        out_n = torch.empty(n, K, dtype=torch.int64, device=dev)
        out_e = torch.empty(n, K, dtype=torch.int64, device=dev)
        out_t = torch.empty(n, K, dtype=torch.float64, device=dev)
        stream = self._stream()
        # route even an empty slice: the pull that follows then fetches nothing, and every rank takes the barrier
        rc = lib.tpn_route_nodes(self._c_shard(), qn.data_ptr() if n else None, n, rows.data_ptr() if n else None,
                                 stream)
        if rc:
            _lib.check(rc, 'tpn_route_nodes')
        self._before_pull()              # every rank's fold is done before anyone reads its lists
        _lib.check(lib.tpn_stream_shard_pull(ctypes.byref(self._cs), stream), 'tpn_stream_shard_pull')
        if n:
            rc = lib.tpn_stream_shard_query(ctypes.byref(self._cs), qn.data_ptr(), rows.data_ptr(), qt.data_ptr(), n, K,
                                            out_n.data_ptr(), out_e.data_ptr(), out_t.data_ptr(), stream)
            if rc:
                _lib.check(rc, 'tpn_stream_shard_query')
        if as_tensors:
            return keep, out_n, out_e, out_t
        res = keep.cpu().numpy(), out_n.cpu().numpy(), out_e.cpu().numpy(), out_t.cpu().numpy()
        self.check_errors()
        return res

    def check_errors(self) -> None:
        """``StreamingRecentSampler.check_errors``, then the routing flags: IndexError for an id outside the graph,
        RuntimeError when one generation's remote lists do not fit ``cache_rows``."""
        err = self._take_shard_error(               # cleared with the sampler's flag, by one call
            f'node id out of range for a sampler over {self.num_nodes} nodes (routing)',
            f'the remote lists one batch queries do not fit cache_rows={self.cache_rows}: construct '
            f'ShardedStreamingSampler with a larger cache_rows',
            'a peer rank never reached a barrier of the sharded sampler')
        super().check_errors()
        if err is not None:
            raise err


def get_neighbor_sampler(data, sample_neighbor_strategy: str = 'recent', device: Union[str, torch.device] = 'cuda:0',
                         **_unused) -> RecentNeighborSampler:
    """Counterpart of ``utils/utils.py:239-262`` for a reference ``Data`` object (fields src_node_ids,
    dst_node_ids, edge_ids, node_interact_times)."""
    if sample_neighbor_strategy != 'recent':
        raise NotImplementedError("only the 'recent' strategy (the one TPNet uses) has a GPU sampler")
    return RecentNeighborSampler(data.src_node_ids, data.dst_node_ids, data.edge_ids, data.node_interact_times, device)
