"""Node-sharded walk-projection state for graphs too large for one GPU (SURVEY.md §8e).

The reference is single-device; this file is the multi-GPU extension `north_star` asks for.
Rows of node ``u`` live on rank ``u % G`` at local row ``u // G`` (modulo placement balances
power-law hubs).  The edge batch / pair list is replicated on every rank (24 B/edge).

Data plane ``exchange='peer'`` (default on CUDA): everything of a call runs on the device, per rank, with
no host plan and no collective —
  1. ``tpn_route_update`` / ``tpn_route_pairs``: stable compaction of the items this rank owns (target /
     first endpoint owned) and a cache slot, in the extension rows behind the local rows, for every remote
     second endpoint (de-duplicated through a mark table; a slot lives until the next write to the state);
  2. ``tpn_pull_rows``: the new slots are filled straight out of the owners' HBM over NVLink (every rank's
     state and stamps are mapped into every other rank with CUDA IPC), stamps included, so a cached row is
     read exactly like a local row and sharded results equal the single-GPU ones bit for bit;
  3. ``tpn_peer_barrier`` (flag words in peer memory) where the protocol needs one: after a write before the
     peers' next pull, and between the pulls of an update and its writes;
  4. the rank-local kernels with the device-side item count (``tpn_update_messages`` / ``tpn_pairwise``).
The encoder's structured call and ``get_random_projections`` split their rows by position instead: every rank
routes the ids its slice reads with ``tpn_route_nodes`` (own rows, or cache slots of the same mark table), pulls,
and runs the plain kernels (``tpn_pairwise_neighbors`` / ``tpn_gather``) on the translated rows.
All of it is plain kernel launches on one stream: a whole step can be captured in a CUDA graph.

Data plane ``exchange='nccl'`` (portable; what the gloo CPU tests exercise): the routing plan is computed on
the host (``make_plan`` / ``tpn_plan``), senders pack whole node blocks (``tpn_gather_blocks``) and ONE
``all_to_all_single`` delivers them into the extension rows.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .peer import IpcPeerGroup, LocalPeerGroup, PeerBuffer, PeerGroup, SymmPeerGroup
from .random_projection import _DEFAULT_LOG_EPOCHS, RandomProjectionModule, _round_up


def owner_of(ids: np.ndarray, world: int) -> np.ndarray:
    return ids % world


def local_row(ids: np.ndarray, world: int) -> np.ndarray:
    return ids // world


def rows_on_rank(node_num: int, world: int, rank: int) -> int:
    """Number of global ids u < node_num with u % world == rank."""
    return (node_num - rank + world - 1) // world if node_num > rank else 0


@dataclass
class ShardPlan:
    """Routing of one call, identical on every rank up to the rank-specific parts."""
    keep: np.ndarray            # indices (into the call's message / pair list) owned by this rank, in order
    first_rows: np.ndarray      # int64[M] local row of the target (update) / a endpoint (pairwise)
    second_rows: np.ndarray     # int64[M] row of the source / b endpoint: local row, or n_local + receive slot
    send_rows: np.ndarray       # int64[S] local rows to pack, grouped by destination rank (ascending), then node id
    send_counts: List[int]      # rows per destination rank
    recv_counts: List[int]      # rows per source rank (they land at n_local + offset, grouped by rank, then node id)

    @property
    def num_recv(self) -> int:
        return int(sum(self.recv_counts))


def make_plan(first: np.ndarray, second: np.ndarray, world: int, rank: int, n_local: int) -> ShardPlan:
    """Plan for messages/pairs (first[m], second[m]): work item m belongs to owner(first[m]) and
    needs the rows of second[m].  Pure function of the replicated inputs: rank r's send list to
    rank q is, by construction, rank q's receive list from rank r (same set, same order)."""
    first = np.asarray(first, dtype=np.int64)
    second = np.asarray(second, dtype=np.int64)
    if world == 1:                                                   # everything is local
        return ShardPlan(keep=np.arange(first.shape[0]), first_rows=first, second_rows=second,
                         send_rows=np.zeros(0, dtype=np.int64), send_counts=[0], recv_counts=[0])
    of, os_ = first % world, second % world
    big = np.int64(max(int(first.max(initial=0)), int(second.max(initial=0))) + 1)

    keep = np.nonzero(of == rank)[0]
    sec = second[keep]
    sec_owner = os_[keep]
    remote = sec_owner != rank
    second_rows = sec // world
    recv_counts = [0] * world
    if remote.any():
        key = sec_owner[remote] * big + sec[remote]                  # group by owner, then node id
        uniq, inverse = np.unique(key, return_inverse=True)
        second_rows = second_rows.copy()
        second_rows[remote] = n_local + inverse
        recv_counts = np.bincount(uniq // big, minlength=world).astype(np.int64).tolist()

    need = (os_ == rank) & (of != rank)                              # my rows that other ranks need
    send_counts = [0] * world
    send_rows = np.zeros(0, dtype=np.int64)
    if need.any():
        key = of[need] * big + second[need]                          # group by destination, then node id
        uniq = np.unique(key)
        send_rows = (uniq % big) // world
        send_counts = np.bincount(uniq // big, minlength=world).astype(np.int64).tolist()
    return ShardPlan(keep=keep, first_rows=first[keep] // world, second_rows=second_rows,
                     send_rows=send_rows.astype(np.int64), send_counts=[int(c) for c in send_counts],
                     recv_counts=[int(c) for c in recv_counts])


class NativePlanner:
    """`make_plan` computed by the library (csrc/tpn_plan.cu: two linear passes, no sort of the batch) —
    same plan, field for field (tests/test_sharded_cpu.py), 10x faster on 100k-edge batches."""

    def __init__(self, global_node_num: int, world: int, rank: int):
        self._lib = _lib.load()
        self.world, self.rank = int(world), int(rank)
        self.handle = ctypes.c_void_p()
        _lib.check(self._lib.tpn_planner_create(ctypes.byref(self.handle), int(global_node_num), self.world, self.rank),
                   'tpn_planner_create')

    def plan(self, first: np.ndarray, second: np.ndarray, n_local: int) -> ShardPlan:
        first = np.ascontiguousarray(first, dtype=np.int64)
        second = np.ascontiguousarray(second, dtype=np.int64)
        m = int(first.shape[0])
        if second.shape[0] != m:
            raise ValueError('first and second must have the same length')
        keep, rows1, rows2, send = (np.empty(max(m, 1), dtype=np.int64) for _ in range(4))
        sc, rc_ = np.zeros(self.world, dtype=np.int64), np.zeros(self.world, dtype=np.int64)
        nk, ns = ctypes.c_int64(0), ctypes.c_int64(0)
        rc = self._lib.tpn_plan(self.handle, first.ctypes.data, second.ctypes.data, m, int(n_local), keep.ctypes.data,
                                rows1.ctypes.data, rows2.ctypes.data, ctypes.byref(nk), send.ctypes.data,
                                ctypes.byref(ns), sc.ctypes.data, rc_.ctypes.data)
        if rc == _lib.TPN_ERR_INDEX:
            raise IndexError('node id out of range in a sharded batch')
        _lib.check(rc, 'tpn_plan')
        return ShardPlan(keep=keep[:nk.value], first_rows=rows1[:nk.value], second_rows=rows2[:nk.value],
                         send_rows=send[:ns.value], send_counts=[int(c) for c in sc], recv_counts=[int(c) for c in rc_])

    def __del__(self):
        try:
            if self.handle:
                self._lib.tpn_planner_destroy(self.handle)
                self.handle = ctypes.c_void_p()
        except Exception:  # interpreter shutdown
            pass


def update_messages(src: np.ndarray, dst: np.ndarray, t: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """The 2B messages of one edge batch in the reference's accumulation order: all
    (target=src, source=dst) in batch order, then all (target=dst, source=src) — the two
    scatter_add_ calls of models/TPNet.py:93-96."""
    return np.concatenate([src, dst]), np.concatenate([dst, src]), np.concatenate([t, t])


def exchange_blocks(send: torch.Tensor, send_counts: Sequence[int], recv: torch.Tensor, recv_counts: Sequence[int],
                    group=None) -> None:
    """The one collective of the sharded path: rows of `send` ([S, W], grouped by destination
    rank) are delivered into `recv` ([R, W], grouped by source rank)."""
    if sum(send_counts) != send.shape[0] or sum(recv_counts) != recv.shape[0]:
        raise ValueError('split sizes do not match the buffers')
    dist.all_to_all_single(recv, send, output_split_sizes=list(recv_counts), input_split_sizes=list(send_counts),
                           group=group)


@dataclass
class RoutedPairs:
    """Result of a routed pair-wise call (peer data plane): the pairs this rank owns, padded to the capacity
    the call was sized for.  ``count`` (device int32[1]) is the number of valid rows; rows past it are zero."""
    keep: torch.Tensor          # int64 [cap]  position in the batch of the j-th kept pair
    feat: torch.Tensor          # float32 [cap, F]
    count: torch.Tensor         # int32 [1]

    def trimmed(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """(positions, features) of exactly the owned pairs — one device -> host read of the count."""
        m = int(self.count.item())
        if m > self.feat.shape[0]:
            raise RuntimeError(f'{m} pairs routed to this rank but the call was sized for {self.feat.shape[0]}: '
                               f'raise route_cap_factor')
        return self.keep[:m], self.feat[:m]


class ShardedRandomProjection(RandomProjectionModule):
    """Rank-local part of the node-sharded state.  Same constructor as the reference class plus
    the process group; ``node_num`` is the GLOBAL node count.  ``update`` and
    ``pair_wise_gram`` take the replicated global-id batch; ``pair_wise_gram`` returns the
    features of the pairs this rank owns together with their positions in the batch
    (``get_pair_wise_feature(..., gather=True)`` re-assembles the reference's ``[n, F]`` tensor on every rank).
    ``neighbor_pair_wise_gram`` / ``get_neighbor_pair_wise_feature`` / ``get_random_projections`` compute a positional
    slice of their rows on each rank and return it with its positions (``gather=True``: the reference's tensors).

    ``exchange``: 'peer' — routing, NVLink pulls and barriers on the device (module docstring; needs the state
    on CUDA); 'nccl' — host plan + one all_to_all_single; 'auto' — 'peer' when the state is created on a CUDA
    device (``state_device``), else 'nccl'.  ``peers``: a ``PeerGroup`` (default: ``IpcPeerGroup`` over
    ``group`` when torch.distributed is initialised; ``LocalPeerGroup`` views put several ranks in one
    process).  ``route_cap_factor`` bounds the share of a call's items one rank may own (the launches of the
    rank-local kernels are sized for ``min(1, factor / world)`` of the call; an overflow is flagged, never silent).
    """

    def __init__(self, node_num: int, edge_num: int, dim_factor: int, num_layer: int, time_decay_weight: float,
                 device: str, use_matrix: bool, beginning_time: np.float64, not_scale: bool, enforce_dim: int,
                 decay_mode: str = 'lazy', group=None, ext_rows: int = 1 << 16, p0: str = 'global',
                 state_device=None, exchange: str = 'auto', peers: Optional[PeerGroup] = None,
                 route_cap_factor: float = 3.5, accumulation: str = 'reference', giant_chunk: int = 1024):
        if use_matrix:
            raise ValueError('use_matrix keeps N x N matrices: not meaningful for a sharded state')
        if exchange not in ('auto', 'peer', 'nccl'):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        self.group = group
        if peers is not None:
            self.world, self.rank = int(peers.world), int(peers.rank)
        else:
            self.world = dist.get_world_size(group) if dist.is_initialized() else 1
            self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        sdev = torch.device(state_device) if state_device is not None else None
        if exchange == 'auto':
            exchange = 'peer' if (sdev is not None and sdev.type == 'cuda' and self.world > 1) else 'nccl'
        if exchange == 'peer' and (sdev is None or sdev.type != 'cuda'):
            raise ValueError("exchange='peer' needs the state on a CUDA device: pass state_device")
        self.exchange = exchange
        self.route_cap_factor = float(route_cap_factor)
        self.global_node_num = int(node_num)
        self.n_local = rows_on_rank(self.global_node_num, self.world, self.rank)
        self.ext_rows = int(ext_rows)
        # the width rule uses the GLOBAL node count (TPNet.py:30-33)
        dim = enforce_dim if enforce_dim != -1 else min(int(math.log(edge_num * 2)) * dim_factor, node_num)
        self._p0_mode = p0
        if p0 == 'global':
            # draw the global P_0 exactly like the single-GPU module and keep this rank's rows:
            # same values as an unsharded run with the same seed (parity tests)
            full = torch.normal(0, 1 / math.sqrt(dim), (self.global_node_num, dim))
            mine = full[self.rank::self.world].clone()
            del full
        else:
            mine = None
        state_buffer = None
        self._peer_bufs = {}
        # one process per GPU: symmetric memory (2 MiB pages; the legacy-IPC mapping is TLB-bound, peer.py);
        # an explicit PeerGroup (in-process ranks, IPC) brings its own kind of buffer
        self._symmetric = exchange == 'peer' and (peers is None or getattr(peers, 'symmetric', False))
        self._rows_alloc = rows_on_rank(self.global_node_num, self.world, 0) + self.ext_rows      # same on every rank
        if exchange == 'peer':
            rows = self.n_local + self.ext_rows
            stride = _round_up(dim, 8)
            buf = PeerBuffer(self._rows_alloc * (num_layer + 1) * stride * 4, sdev, symmetric=self._symmetric)
            self._peer_bufs['state'] = buf
            state_buffer = buf.tensor((rows, num_layer + 1, stride), torch.float32)
        super().__init__(node_num=self.n_local + self.ext_rows, edge_num=edge_num, dim_factor=dim_factor,
                         num_layer=num_layer, time_decay_weight=time_decay_weight, device=device, use_matrix=False,
                         beginning_time=beginning_time, not_scale=not_scale, enforce_dim=dim, decay_mode=decay_mode,
                         init_p0=False, state_device=state_device, accumulation=accumulation, giant_chunk=giant_chunk,
                         state_buffer=state_buffer)
        with torch.no_grad():
            if mine is not None:
                self.random_projections[0][:self.n_local].copy_(mine)
        self.exchanged_rows = 0          # rows received so far (bench accounting; 'nccl' data plane)
        self._send_buf: Optional[torch.Tensor] = None
        self._all_keep: Optional[np.ndarray] = None
        self._planner: Optional[NativePlanner] = None
        # ---- peer data plane
        self._peers = peers
        self._shard: Optional[_lib.TpnShard] = None
        self._shard_tensors = {}
        self._route = {}                 # cached routing buffers, keyed by (kind, items)
        self._dirty = True               # a rank may have written since the last barrier: barrier before pulling
        self.barriers = 0                # barriers issued so far (bench accounting)
        if exchange == 'peer':
            if self.lazy:
                # stamps live in peer memory too (a puller copies them with the rows); -1 = never written
                sb = PeerBuffer(self._rows_alloc * self.num_layer * 4, sdev, symmetric=self._symmetric)
                self._peer_bufs['stamps'] = sb
                self._stamps = sb.tensor((self.node_num, self.num_layer), torch.int32)
                self._stamps.fill_(-1)
                self._decay_log = torch.ones(_DEFAULT_LOG_EPOCHS, self.num_layer, dtype=torch.float64, device=sdev)
            self._peer_bufs['flags'] = PeerBuffer(4 * max(self.world, 16), sdev, symmetric=self._symmetric)

    # ------------------------------------------------------------------ helpers
    def init_p0_on_device(self, seed: int) -> None:
        """P_0 ~ N(0, 1/sqrt(d)) drawn directly on this rank's GPU (large graphs: no host pass)."""
        g = torch.Generator(device=self._state.device).manual_seed(seed * 1000003 + self.rank)
        with torch.no_grad():
            p0 = self.random_projections[0]
            block = 1 << 20
            for lo in range(0, self.n_local, block):
                hi = min(lo + block, self.n_local)
                p0[lo:hi].copy_(torch.randn(hi - lo, self.dim, device=p0.device, generator=g) / math.sqrt(self.dim))

    def _ext_view(self, rows: int) -> torch.Tensor:
        if rows > self.ext_rows:
            raise RuntimeError(f'{rows} remote rows needed but the extension region holds {self.ext_rows}: '
                               f'construct ShardedRandomProjection with a larger ext_rows')
        return self._state.view(self.node_num, self.node_stride)[self.n_local:self.n_local + rows]

    def _exchange(self, plan: ShardPlan) -> None:
        """Pack -> all-to-all -> received blocks sit in the extension rows."""
        self._require_cuda()
        lib = _lib.load()
        dev = self._state.device
        S, R = int(plan.send_rows.shape[0]), plan.num_recv
        if self._send_buf is None or self._send_buf.shape[0] < max(S, 1):
            self._send_buf = torch.empty(max(S, 1024), self.node_stride, dtype=torch.float32, device=dev)
        send = self._send_buf[:S]
        if S:
            ptr = self._ids_to_device([plan.send_rows], ['id'])[0]
            rc = lib.tpn_gather_blocks(self._c_state(), ptr, S, send.data_ptr(), self._stream())
            if rc:
                _lib.check(rc, 'tpn_gather_blocks')
        if self.world > 1 and dist.is_initialized():
            # decided collectively: a rank that raised alone would leave the others waiting in the all_to_all
            over = torch.tensor([1 if R > self.ext_rows else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(over, op=dist.ReduceOp.MAX, group=self.group)
            if int(over.item()):
                raise RuntimeError(f'a rank needs more remote rows than the {self.ext_rows} extension rows hold '
                                   f'(this rank: {R}): construct ShardedRandomProjection with a larger ext_rows')
        recv = self._ext_view(R)
        if self.world > 1:
            exchange_blocks(send, plan.send_counts, recv, plan.recv_counts, self.group)
        if self.lazy and R:
            self._c_state()                                   # makes sure the stamps exist
            self._stamps[self.n_local:self.n_local + R].fill_(self._h.epoch)     # received rows are current
        self.exchanged_rows += R

    # ------------------------------------------------------------------ peer data plane: set-up
    def connect(self) -> None:
        """Rendezvous of the peer-visible buffers (collective over the ranks of the group; the first routed call
        does it if the caller did not).  With a ``LocalPeerGroup`` every rank must be constructed first."""
        if self.exchange != 'peer' or self._shard is not None:
            return
        dev = self._require_cuda()
        if self._peers is None:
            if not dist.is_initialized():
                raise RuntimeError("exchange='peer' with world > 1 needs torch.distributed or a PeerGroup")
            self._peers = SymmPeerGroup(self.group)
        tables = {}
        for name in ('state', 'stamps', 'flags'):
            if name in self._peer_bufs:
                ptrs = self._peers.exchange(name, self._peer_bufs[name])
                tables[name] = torch.tensor(ptrs, dtype=torch.int64, device=dev)
        t = self._shard_tensors
        t['tables'] = tables
        t['mark'] = torch.zeros(self.global_node_num, dtype=torch.int32, device=dev)
        t['counters'] = torch.zeros(_lib.SHARD_COUNTERS, dtype=torch.int32, device=dev)
        t['need'] = torch.zeros(max(self.ext_rows, 1), dtype=torch.int64, device=dev)
        t['seq'] = torch.zeros(1, dtype=torch.int32, device=dev)
        sh = _lib.TpnShard()
        sh.world, sh.rank = self.world, self.rank
        sh.global_nodes = self.global_node_num
        sh.num_local_rows = self.n_local
        sh.ext_rows = self.ext_rows
        sh.peer_data = tables['state'].data_ptr()
        sh.peer_stamps = tables['stamps'].data_ptr() if 'stamps' in tables else None
        sh.peer_flags = tables['flags'].data_ptr()
        sh.mark = t['mark'].data_ptr()
        sh.counters = t['counters'].data_ptr()
        sh.need_nodes = t['need'].data_ptr()
        sh.barrier_seq = t['seq'].data_ptr()
        self._shard = sh
        self._peers.barrier()            # every rank has mapped every buffer before anyone launches a pull

    def close(self) -> None:
        """Collective teardown of the peer data plane: every rank stops using its peers' memory, unmaps it, and only
        then may anyone free its buffers (freeing an exported allocation that a peer still maps is undefined).  Call
        it on every rank before dropping the module when another sharded module will be created in the same job."""
        if self._shard is None or self._peers is None:
            return
        if self._state.is_cuda:
            torch.cuda.synchronize(self._state.device)
        self._peers.barrier()
        if hasattr(self._peers, 'close'):
            self._peers.close()
        self._peers.barrier()
        self._shard = None
        self._shard_tensors = {}

    def __del__(self):
        try:                                       # best effort without the barriers (interpreter shutdown, errors)
            if getattr(self, '_shard', None) is not None and hasattr(self._peers, 'close'):
                self._peers.close()
        except Exception:
            pass

    def _c_shard(self):
        if self._shard is None:
            self.connect()
        return ctypes.byref(self._shard)

    def _cap(self, items: int) -> int:
        """Launch capacity for the rank-local kernels of a call with `items` work items in total."""
        share = min(1.0, self.route_cap_factor / self.world)
        return int(min(items, math.ceil(items * share) + 1024))

    def _route_buffers(self, kind: str, items: int):
        key = (kind, items)
        buf = self._route.get(key)
        if buf is None:
            dev = self._state.device
            lib = _lib.load()
            buf = dict(first=torch.empty(items, dtype=torch.int64, device=dev),
                       second=torch.empty(items, dtype=torch.int64, device=dev),
                       count=torch.zeros(1, dtype=torch.int32, device=dev),
                       ws=torch.empty(lib.tpn_route_workspace_bytes(items), dtype=torch.uint8, device=dev))
            if kind == 'update':
                buf['t'] = torch.empty(items, dtype=torch.float64, device=dev)
            if len(self._route) > 8:
                self._route.clear()
            self._route[key] = buf
        return buf

    def _barrier(self) -> None:
        self.barriers += 1
        if getattr(self._peers, 'host_barriers', False):
            return          # LocalPeerGroup: the driver of the in-process ranks orders the phases itself (peer.py)
        _lib.check(_lib.load().tpn_peer_barrier(self._c_shard(), self._stream()), 'tpn_peer_barrier')

    def _pull(self) -> None:
        """Peers' writes are ordered before this rank's reads of their rows (one barrier after any write), then the
        cache slots handed out by the latest routing call are filled from the owners' memory."""
        if self._dirty:
            self._barrier()
            self._dirty = False
        _lib.check(_lib.load().tpn_pull_rows(self._c_state(), self._c_shard(), self._stream()), 'tpn_pull_rows')

    def _state_written(self) -> None:
        """After any write to the local rows: cached copies held by (and of) other ranks are stale."""
        self._dirty = True
        if self._shard is not None:
            _lib.check(_lib.load().tpn_shard_new_generation(self._c_shard(), self._stream()), 'tpn_shard_new_generation')

    def _update_peer(self, src_node_ids, dst_node_ids, node_interact_times, next_time) -> None:
        pending = self.update_begin(src_node_ids, dst_node_ids, node_interact_times, next_time)
        self._barrier()                       # every rank has pulled its pre-batch rows: now the writes may start
        self.update_end(pending)

    def update_begin(self, src_node_ids, dst_node_ids, node_interact_times, next_time=None):
        """First half of a routed update: routing + pulls of the pre-batch remote rows (reads only).  ``update`` is
        ``update_begin`` -> rank barrier -> ``update_end``; a driver that runs several ranks in one process calls
        the halves itself (all ranks' ``update_begin``, then all ranks' ``update_end``)."""
        dev = self._require_cuda()
        lib = _lib.load()
        n = int(len(src_node_ids))
        if n == 0:
            raise IndexError('index -1 is out of bounds for axis 0 with size 0')
        if len(dst_node_ids) != n or len(node_interact_times) != n:
            raise ValueError('src, dst and time arrays must have the same length')
        if next_time is None:
            last = node_interact_times[-1]
            next_time = float(last.item()) if isinstance(last, torch.Tensor) else float(last)
        h = self._h
        lam = self.time_decay_weight
        base = np.exp(-lam * (np.float64(next_time) - np.float64(h.now)))
        factors = (ctypes.c_float * self.num_layer)(*[float(np.float32(np.power(base, i)))
                                                      for i in range(1, self.num_layer + 1)])
        ptrs = self._global_ids_to_device([src_node_ids, dst_node_ids, node_interact_times], ['id', 'id', 'time'])
        st = self._c_state()
        sh = self._c_shard()
        stream = self._stream()
        rb = self._route_buffers('update', 2 * n)
        rc = lib.tpn_route_update(sh, ptrs[0], ptrs[1], ptrs[2], n, rb['first'].data_ptr(), rb['second'].data_ptr(),
                                  rb['t'].data_ptr(), rb['count'].data_ptr(), rb['ws'].data_ptr(), rb['ws'].numel(),
                                  stream)
        if rc:
            _lib.check(rc, 'tpn_route_update')
        self._pull()
        return dict(n=n, rb=rb, next_time=float(next_time), factors=factors, lam=lam)

    def update_end(self, pending) -> None:
        """Second half of a routed update: the rank-local kernels (writes) and the new cache generation."""
        dev = self._state.device
        lib = _lib.load()
        h = self._h
        n, rb, next_time, factors, lam = (pending[k] for k in ('n', 'rb', 'next_time', 'factors', 'lam'))
        st = self._c_state()
        stream = self._stream()
        cap = self._cap(2 * n)
        need = lib.tpn_update_workspace_bytes(st, (cap + 1) // 2)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=dev)
        args = (rb['first'].data_ptr(), rb['second'].data_ptr(), rb['t'].data_ptr(), cap, rb['count'].data_ptr(),
                self.n_local, float(next_time), float(np.float32(-lam)), factors, self._ws.data_ptr(),
                self._ws.numel(), self._err.data_ptr(), stream)
        rc = lib.tpn_update_messages(st, *args)
        if rc == _lib.TPN_ERR_LOG_FULL:       # same epoch, same factors on every rank: they all restart together
            self._restart_log()
            st = self._c_state()
            rc = lib.tpn_update_messages(st, *args)
        if rc:
            _lib.check(rc, 'tpn_update_messages')
        h.epoch = int(h.st.epoch)
        h.launches += 1
        h.now = float(next_time)
        self.now_time.data.fill_(h.now)
        self._state_written()

    #: host arrays at least this long are uploaded in slices (1/world per rank) and all-gathered over NVLink
    SLICED_UPLOAD_MIN = 32768

    def _sliced_upload(self, arrays, kinds):
        """The batch is replicated on every rank's HOST; uploading all of it on every rank would move world x the
        bytes over PCIe.  Rank r stages only elements [r*per, (r+1)*per) of each array (pinned memory, validated
        on the way) and one all_gather per array over NVLink rebuilds the full arrays on every device."""
        dev = self._state.device
        n = int(arrays[0].shape[0])
        per = (n + self.world - 1) // self.world
        lo, hi = min(self.rank * per, n), min((self.rank + 1) * per, n)
        key = ('upload', per, len(arrays))
        ring = self._route.get(key)
        if ring is None:
            ring = dict(cursor=0, slots=[])
            for _ in range(4):
                ring['slots'].append(dict(
                    host=[torch.empty(per, dtype=torch.int64).pin_memory() for _ in arrays],
                    dev=[torch.empty(per, dtype=torch.int64, device=dev) for _ in arrays],
                    full=[torch.empty(per * self.world, dtype=torch.int64, device=dev) for _ in arrays],
                    done=torch.cuda.Event()))
            self._route[key] = ring
        slot = ring['slots'][ring['cursor']]
        ring['cursor'] = (ring['cursor'] + 1) % len(ring['slots'])
        slot['done'].synchronize()                       # the copies out of this slot's pinned memory have left
        bad = False
        for a, kind, h, d in zip(arrays, kinds, slot['host'], slot['dev']):
            want = np.int64 if kind == 'id' else np.float64
            part = np.ascontiguousarray(a[lo:hi], dtype=want)
            if kind == 'id' and part.size and (part.min() < 0 or part.max() >= self.global_node_num):
                bad = True
            h.numpy().view(want)[:hi - lo] = part
            d.copy_(h, non_blocking=True)
        slot['done'].record()
        out = []
        for d, f in zip(slot['dev'], slot['full']):
            dist.all_gather_into_tensor(f, d, group=self.group)
            out.append(f.data_ptr())
        self._h.keepalive = slot
        if bad:                                          # after the collectives: the other ranks are not left waiting
            raise IndexError(f'index out of range for node_num {self.global_node_num}')
        return out

    def _global_ids_to_device(self, arrays, kinds):
        """Like _ids_to_device, for GLOBAL ids: host arrays are range-checked against the global node count."""
        if (self.exchange == 'peer' and self.world > 1 and dist.is_initialized()
                and isinstance(self._peers, (IpcPeerGroup, SymmPeerGroup))
                and all(isinstance(a, np.ndarray) and a.ndim == 1 for a in arrays)
                and arrays[0].shape[0] >= self.SLICED_UPLOAD_MIN
                and all(a.shape[0] == arrays[0].shape[0] for a in arrays)):
            return self._sliced_upload(arrays, kinds)
        return self._rank_ids_to_device(arrays, kinds)

    def _rank_ids_to_device(self, arrays, kinds):
        """Global ids of this rank's own lists (never the sliced upload of a replicated batch): host arrays are
        range-checked against the global node count before anything is launched."""
        keep = self.node_num
        self.node_num = self.global_node_num          # the stager validates against node_num
        try:
            return self._ids_to_device(arrays, kinds, wrap_negative=False)
        finally:
            self.node_num = keep

    def _pairs_peer(self, a_ids, b_ids) -> RoutedPairs:
        dev = self._require_cuda()
        lib = _lib.load()
        n = int(len(a_ids))
        if len(b_ids) != n:
            raise ValueError('src and dst id arrays must have the same length')
        cap = self._cap(max(n, 1))
        out = torch.zeros(cap, self.pair_wise_feature_dim, dtype=torch.float32, device=dev)
        rb = self._route_buffers('pairs', max(n, 1))
        keep = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        if n == 0:
            rb['count'].zero_()
            return RoutedPairs(keep[:0], out[:0], rb['count'])
        ptrs = self._global_ids_to_device([a_ids, b_ids], ['id', 'id'])
        st = self._c_state()
        sh = self._c_shard()
        stream = self._stream()
        count = torch.zeros(1, dtype=torch.int32, device=dev)      # per call: results of several calls stay alive
        rc = lib.tpn_route_pairs(sh, ptrs[0], ptrs[1], n, rb['first'].data_ptr(), rb['second'].data_ptr(),
                                 keep.data_ptr(), count.data_ptr(), rb['ws'].data_ptr(), rb['ws'].numel(), stream)
        if rc:
            _lib.check(rc, 'tpn_route_pairs')
        self._pull()
        rc = lib.tpn_pairwise(st, rb['first'].data_ptr(), rb['second'].data_ptr(), cap, count.data_ptr(),
                              0 if self.not_scale else 1, out.data_ptr(), stream)
        if rc:
            _lib.check(rc, 'tpn_pairwise')
        self._h.launches += 1
        return RoutedPairs(keep[:cap], out, count)

    def routed_pair_wise_gram(self, src_node_ids, dst_node_ids) -> RoutedPairs:
        """Peer data plane, no host synchronisation: padded features of the owned pairs + device-side count."""
        return self._pairs_peer(src_node_ids, dst_node_ids)

    def routed_pair_wise_feature(self, src_node_ids, dst_node_ids) -> RoutedPairs:
        r = self._pairs_peer(src_node_ids, dst_node_ids)
        return RoutedPairs(r.keep, self._head(r.feat, r.count), r.count)

    def assemble(self, routed: RoutedPairs, n: int) -> torch.Tensor:
        """The reference's ``[n, F]`` result on every rank: each rank contributes the rows of the pairs it owns
        (one all_gather of the padded blocks; collective over the process group)."""
        cap, F = routed.feat.shape
        if self.world == 1 or not dist.is_initialized():
            keep, feat = routed.trimmed()
            full = torch.zeros(n, F, dtype=torch.float32, device=feat.device)
            full[keep] = feat
            return full
        feats = torch.empty(self.world, cap, F, dtype=torch.float32, device=routed.feat.device)
        keeps = torch.empty(self.world, cap, dtype=torch.int64, device=routed.feat.device)
        counts = torch.empty(self.world, dtype=torch.int32, device=routed.feat.device)
        dist.all_gather_into_tensor(feats, routed.feat.contiguous(), group=self.group)
        dist.all_gather_into_tensor(keeps, routed.keep.contiguous(), group=self.group)
        dist.all_gather_into_tensor(counts, routed.count, group=self.group)
        full = torch.zeros(n, F, dtype=torch.float32, device=routed.feat.device)
        valid = torch.arange(cap, device=counts.device)[None, :] < counts[:, None]
        full[keeps[valid]] = feats[valid]
        return full

    # ------------------------------------------------------------------ API
    def _make_plan(self, first: np.ndarray, second: np.ndarray) -> ShardPlan:
        if self.world == 1:
            return make_plan(first, second, 1, 0, self.n_local)
        if self._planner is None:
            self._planner = NativePlanner(self.global_node_num, self.world, self.rank)
        return self._planner.plan(first, second, self.n_local)

    def plan_update(self, src: np.ndarray, dst: np.ndarray, t: np.ndarray):
        tgt, oth, tm = update_messages(np.asarray(src, dtype=np.int64), np.asarray(dst, dtype=np.int64),
                                       np.asarray(t, dtype=np.float64))
        plan = self._make_plan(tgt, oth)
        return plan, np.ascontiguousarray(tm[plan.keep])

    def update_prepare(self, src_node_ids, dst_node_ids, node_interact_times, next_time=None) -> bool:
        """One shard: the plain module's early half.  Several shards: not split (routing and the pulls of the update
        follow the pair-wise calls of the batch, whose cached rows they reuse) — returns False."""
        if self.world == 1:
            return RandomProjectionModule.update_prepare(self, src_node_ids, dst_node_ids, node_interact_times, next_time)
        return False

    def update(self, src_node_ids, dst_node_ids, node_interact_times, next_time=None, plan=None):
        """TPNet.py:67-99 on the sharded state.  All ranks must call it with the same batch."""
        if self.world == 1 and plan is None:
            # one shard = the whole graph: the plain edge-batch path (no message list, no exchange)
            return RandomProjectionModule.update(self, src_node_ids, dst_node_ids, node_interact_times, next_time)
        if self.exchange == 'peer' and plan is None:
            return self._update_peer(src_node_ids, dst_node_ids, node_interact_times, next_time)
        dev = self._require_cuda()
        lib = _lib.load()
        t = np.asarray(node_interact_times, dtype=np.float64)
        if len(t) == 0:
            raise IndexError('index -1 is out of bounds for axis 0 with size 0')
        if plan is None:
            src = np.asarray(src_node_ids, dtype=np.int64)
            dst = np.asarray(dst_node_ids, dtype=np.int64)
            if src.min() < 0 or dst.min() < 0 or src.max() >= self.global_node_num or \
                    dst.max() >= self.global_node_num:
                raise IndexError(f'index out of range for node_num {self.global_node_num}')
            plan = self.plan_update(src, dst, t)
        plan, t_msg = plan
        next_time = float(t[-1]) if next_time is None else float(next_time)
        h = self._h
        lam = self.time_decay_weight
        base = np.exp(-lam * (np.float64(next_time) - np.float64(h.now)))
        factors = (ctypes.c_float * self.num_layer)(*[float(np.float32(np.power(base, i)))
                                                      for i in range(1, self.num_layer + 1)])
        self._exchange(plan)                                  # pre-batch rows, before the clock moves
        M = int(plan.first_rows.shape[0])
        if M:
            ptrs = self._ids_to_device([plan.first_rows, plan.second_rows, t_msg], ['id', 'id', 'time'],
                                       wrap_negative=False)
            st = self._c_state()
            need = lib.tpn_update_workspace_bytes(st, (M + 1) // 2)
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=dev)
            args = (ptrs[0], ptrs[1], ptrs[2], M, None, self.n_local, next_time, float(np.float32(-lam)), factors,
                    self._ws.data_ptr(), self._ws.numel(), self._err.data_ptr(), self._stream())
            rc = lib.tpn_update_messages(st, *args)
            if rc == _lib.TPN_ERR_LOG_FULL:
                self._restart_log()
                st = self._c_state()
                rc = lib.tpn_update_messages(st, *args)
            if rc:
                _lib.check(rc, 'tpn_update_messages')
            h.epoch = int(h.st.epoch)
            h.launches += 1
        else:
            # no local message: the clock (and the lazy epoch) must still advance identically
            self._advance_clock_only(factors)
        h.now = next_time
        self.now_time.data.fill_(h.now)

    def _advance_clock_only(self, factors) -> None:
        """Decay without any local message (keeps epochs aligned across ranks)."""
        if all(f == 1.0 for f in factors):
            return
        if self.lazy:
            self._c_state()
            if self._h.epoch + 1 >= self._decay_log.shape[0]:
                self._restart_log()
            if self._h.st.cum_floor * min(factors) < 1e-200:
                self._restart_log()
            self._h.epoch += 1
            f = torch.tensor([float(x) for x in factors], dtype=torch.float64, device=self._decay_log.device)
            self._decay_log[self._h.epoch] = self._decay_log[self._h.epoch - 1] * f      # cumulative products
            self._h.st.cum_floor *= float(min(factors))
        else:
            with torch.no_grad():
                for i in range(1, self.num_layer + 1):
                    self.random_projections[i].mul_(float(factors[i - 1]))

    def plan_pairs(self, a_ids: np.ndarray, b_ids: np.ndarray) -> ShardPlan:
        return self._make_plan(np.asarray(a_ids, dtype=np.int64), np.asarray(b_ids, dtype=np.int64))

    def pair_wise_gram(self, src_node_ids, dst_node_ids, plan: Optional[ShardPlan] = None):
        """Features (input of self.mlp, TPNet.py:119-128) of the pairs whose first endpoint this
        rank owns.  Returns (positions in the batch, float32 [m, (2L+2)^2])."""
        if self.world == 1 and plan is None:
            n = int(len(src_node_ids))
            if self._all_keep is None or self._all_keep.shape[0] != n:
                self._all_keep = np.arange(n)
            return self._all_keep, RandomProjectionModule.pair_wise_gram(self, src_node_ids, dst_node_ids)
        if self.exchange == 'peer' and plan is None:
            keep, feat = self._pairs_peer(src_node_ids, dst_node_ids).trimmed()      # one read of the count
            return keep, feat
        dev = self._require_cuda()
        lib = _lib.load()
        if plan is None:
            plan = self.plan_pairs(src_node_ids, dst_node_ids)
        self._exchange(plan)
        m = int(plan.first_rows.shape[0])
        out = torch.empty(m, self.pair_wise_feature_dim, dtype=torch.float32, device=dev)
        if m:
            ptrs = self._ids_to_device([plan.first_rows, plan.second_rows], ['id', 'id'])
            rc = lib.tpn_pairwise(self._c_state(), ptrs[0], ptrs[1], m, None, 0 if self.not_scale else 1, out.data_ptr(),
                                  self._stream())
            if rc:
                _lib.check(rc, 'tpn_pairwise')
            self._h.launches += 1
        return plan.keep, out

    def get_pair_wise_feature(self, src_node_ids, dst_node_ids, gather: bool = False):
        """Features of the pairs this rank owns, as ``(positions in the batch, [m, F])``; ``gather=True`` returns
        the reference's ``[n, F]`` tensor (TPNet.py:112-129) on every rank (collective)."""
        n = int(len(src_node_ids))
        if self.exchange == 'peer' and self.world > 1:
            routed = self.routed_pair_wise_feature(src_node_ids, dst_node_ids)
            return self.assemble(routed, n) if gather else routed.trimmed()
        keep, feat = self.pair_wise_gram(src_node_ids, dst_node_ids)
        feat = self._head(feat)
        if not gather:
            return keep, feat
        keep_t = keep if isinstance(keep, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(keep)).to(feat.device)
        return self.assemble(RoutedPairs(keep_t, feat, torch.tensor([feat.shape[0]], dtype=torch.int32,
                                                                    device=feat.device)), n) \
            if self.world == 1 else self._assemble_ragged(keep_t, feat, n)

    def _assemble_ragged(self, keep: torch.Tensor, feat: torch.Tensor, n: int) -> torch.Tensor:
        """'nccl' data plane: ranks hold different numbers of rows — pad to the largest, then assemble."""
        m = torch.tensor([feat.shape[0]], dtype=torch.int64, device=feat.device)
        dist.all_reduce(m, op=dist.ReduceOp.MAX, group=self.group)
        cap = int(m.item())
        pf = torch.zeros(cap, feat.shape[1], dtype=torch.float32, device=feat.device)
        pk = torch.zeros(cap, dtype=torch.int64, device=feat.device)
        pf[:feat.shape[0]] = feat
        pk[:feat.shape[0]] = keep
        return self.assemble(RoutedPairs(pk, pf, torch.tensor([feat.shape[0]], dtype=torch.int32, device=feat.device)), n)

    # ------------------------------------------------------------------ node-list calls: encoder features, row reads
    # A call with m rows (encoder rows, or ids of get_random_projections) is split by POSITION: rank r computes rows
    # [r*per, min((r+1)*per, m)), per = ceil(m / world).  Every encoder row reads K + 2 node blocks wherever it runs, so
    # no owner rule saves the pulls; the positional split balances the work exactly, and its size is known on the host
    # (no device count, no capacity padding, no device -> host read).  The rows a rank reads are routed
    # (tpn_route_nodes: own rows, or cache slots of the current generation) and pulled, then the plain kernels run on
    # the translated rows of the local state.
    def _row_split(self, m: int) -> Tuple[int, int, int]:
        """(per, lo, hi): this rank computes rows [lo, hi) of a call with m rows."""
        per = -(-m // self.world)
        lo = min(self.rank * per, m)
        return per, lo, min(lo + per, m)

    def _positions(self, lo: int, hi: int) -> torch.Tensor:
        """Device int64 [lo, hi) (cached: the same split recurs every batch)."""
        key = ('positions', lo, hi)
        t = self._route.get(key)
        if t is None:
            t = torch.arange(lo, hi, dtype=torch.int64, device=self._state.device)
            if len(self._route) > 8:
                self._route.clear()
            self._route[key] = t
        return t

    def _check_node_call(self, what: str) -> None:
        if self.world > 1 and self.exchange != 'peer':
            raise NotImplementedError(f"{what} on a sharded state with world > 1 needs exchange='peer' "
                                      f"(the 'nccl' data plane routes only update and the decoder pairs)")

    def _route_node_rows(self, ids) -> torch.Tensor:
        """Peer data plane: this rank's list of global ids (host array or CUDA tensor) -> int64 rows of the local state,
        every remote row pulled into its cache slot.  Collective: every rank calls it (with its own list, possibly
        empty), because the pull may take a barrier."""
        lib = _lib.load()
        n = int(len(ids))
        rows = torch.empty(n, dtype=torch.int64, device=self._state.device)
        ptr = self._rank_ids_to_device([ids], ['id'])[0] if n else None
        rc = lib.tpn_route_nodes(self._c_shard(), ptr, n, rows.data_ptr() if n else None, self._stream())
        if rc:
            _lib.check(rc, 'tpn_route_nodes')
        self._pull()
        return rows

    def _gather_slices(self, local: torch.Tensor, per: int, m: int) -> torch.Tensor:
        """Every rank's slice of a positional split -> the [m, ...] tensor on every rank (one all_gather of the slices
        padded to `per`; collective).  Not differentiable: the result is detached."""
        if self.world == 1:
            return local.detach()
        if not dist.is_initialized():
            raise RuntimeError('gather=True with world > 1 needs torch.distributed (one process per rank)')
        rest = tuple(local.shape[1:])
        if per == 0:
            return local.detach()
        pad = local.new_zeros((per,) + rest)
        pad[:local.shape[0]] = local.detach()
        full = local.new_empty((self.world * per,) + rest)
        dist.all_gather_into_tensor(full, pad, group=self.group)
        return full[:m]

    def _nbr_gram_rows(self, lists, m: int, k: int) -> torch.Tensor:
        """tpn_pairwise_neighbors on rows of the local state: lists = (nbr [m*K], src [m], dst [m]) as CUDA tensors or
        already validated host arrays (staged here).  Node blocks too wide for the shared-memory staging take the plain
        module's fallback, tpn_pairwise on the expanded row lists."""
        dev = self._state.device
        lib = _lib.load()
        f = self.pair_wise_feature_dim
        out = torch.empty(m, k, 2, f, dtype=torch.float32, device=dev)
        if m == 0 or k == 0:
            return out
        ptrs = self._rank_ids_to_device(list(lists), ['id', 'id', 'id'])
        st, stream, scale = self._c_state(), self._stream(), 0 if self.not_scale else 1
        rc = lib.tpn_pairwise_neighbors(st, ptrs[0], ptrs[1], ptrs[2], m, k, scale, out.data_ptr(), stream)
        if rc == _lib.TPN_ERR_UNSUPPORTED:
            on_dev = [(a.to(dev) if isinstance(a, torch.Tensor) else
                       torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(dev)).contiguous() for a in lists]
            tmp = torch.empty(m * k, f, dtype=torch.float32, device=dev)
            for j, e in enumerate(on_dev[1:]):
                e = e.repeat_interleave(k)
                rc = lib.tpn_pairwise(st, on_dev[0].data_ptr(), e.data_ptr(), m * k, None, scale, tmp.data_ptr(), stream)
                if rc:
                    _lib.check(rc, 'tpn_pairwise')
                out[:, :, j, :] = tmp.view(m, k, f)
            self._h.launches += 2
            return out
        if rc:
            _lib.check(rc, 'tpn_pairwise_neighbors')
        self._h.launches += 1
        return out

    def neighbor_pair_wise_gram(self, neighbor_node_ids, src_node_ids, dst_node_ids, sliced_neighbors: bool = False):
        """The encoder's structured call (TPNet.py:313-324) without the head, on the sharded state.  ``[m, K]`` global
        neighbour ids and ``[m]`` src / dst ids, replicated on every rank; this rank computes the rows of its positional
        slice.  Returns ``(positions in the batch, [rows, K, 2, F])``, the ``(keep, feat)`` convention of
        ``pair_wise_gram``: block ``[j, k, 0]`` is the pair ``(nbr[keep[j], k], src[keep[j]])``, ``[j, k, 1]`` the pair
        with ``dst``.  ``sliced_neighbors=True``: ``neighbor_node_ids`` holds only the ``[rows, K]`` of this rank's slice
        (what ``ShardedStreamingSampler`` answers on this rank), src / dst stay the whole ``[m]``.  Peer data plane (or
        world 1); all ranks call it together."""
        self._check_node_call('neighbor_pair_wise_gram')
        dev = self._require_cuda()
        if neighbor_node_ids.ndim != 2:
            raise ValueError('neighbor_node_ids must be [m, num_neighbors]')
        m = int(len(src_node_ids)) if sliced_neighbors else int(neighbor_node_ids.shape[0])
        k = int(neighbor_node_ids.shape[1])
        if len(src_node_ids) != m or len(dst_node_ids) != m:
            raise ValueError('src and dst id arrays must have one entry per row of neighbor_node_ids')
        per, lo, hi = self._row_split(m)
        n = hi - lo
        if sliced_neighbors and int(neighbor_node_ids.shape[0]) != n:
            raise ValueError(f'sliced_neighbors: this rank computes rows [{lo}, {hi}) of {m}, so neighbor_node_ids must '
                             f'have {n} rows (it has {int(neighbor_node_ids.shape[0])})')
        nbr = neighbor_node_ids if sliced_neighbors else neighbor_node_ids[lo:hi]
        keep = self._positions(lo, hi)
        resident = all(isinstance(a, torch.Tensor) and a.is_cuda for a in (neighbor_node_ids, src_node_ids, dst_node_ids))
        if self.world == 1:
            flat = neighbor_node_ids.reshape(-1)
            return keep, self._nbr_gram_rows((flat, src_node_ids, dst_node_ids), m, k)
        if resident:
            ids = torch.cat([nbr.reshape(-1), src_node_ids[lo:hi], dst_node_ids[lo:hi]])
        else:
            host = [a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
                    for a in (nbr, src_node_ids, dst_node_ids)]
            ids = np.concatenate([host[0].reshape(-1), host[1][lo:hi], host[2][lo:hi]]).astype(np.int64, copy=False)
        rows = self._route_node_rows(ids)
        nk = n * k
        return keep, self._nbr_gram_rows((rows[:nk], rows[nk:nk + n], rows[nk + n:]), n, k)

    def get_neighbor_pair_wise_feature(self, neighbor_node_ids, src_node_ids, dst_node_ids,
                                       out: Optional[torch.Tensor] = None, gather: bool = False,
                                       sliced_neighbors: bool = False):
        """TPNet.py:313-324 on the sharded state: ``self.mlp`` on the ``[rows*K*2, F]`` view of
        ``neighbor_pair_wise_gram``.  Returns ``(positions in the batch, [rows, K, 2F])`` for this rank's slice (``out``:
        the buffer for that slice); ``gather=True`` returns the reference's ``[m, K, 2F]`` on every rank (one
        all_gather; collective).  The gathered tensor carries no gradient: training through a sharded state needs
        the per-rank slices.  ``sliced_neighbors``: as in ``neighbor_pair_wise_gram``."""
        keep, g = self.neighbor_pair_wise_gram(neighbor_node_ids, src_node_ids, dst_node_ids, sliced_neighbors)
        n, k = g.shape[0], g.shape[1]
        f = self.pair_wise_feature_dim
        flat_out = None if out is None else out.view(n * k * 2, f)
        feat = self._head(g.view(n * k * 2, f), out=flat_out).view(n, k, 2 * f)
        if not gather:
            return keep, feat
        m = int(len(src_node_ids))
        return self._gather_slices(feat, self._row_split(m)[0], m)

    def _gather_state_rows(self, ptr: int, n: int) -> torch.Tensor:
        out = torch.empty(self.num_layer + 1, n, self.dim, dtype=torch.float32, device=self._state.device)
        if n:
            rc = _lib.load().tpn_gather(self._c_state(), ptr, n, out.data_ptr(), self._stream())
            if rc:
                _lib.check(rc, 'tpn_gather')
            self._h.launches += 1
        return out

    def get_random_projections(self, node_ids, gather: bool = False):
        """TPNet.py:101-110 on the sharded state: the L+1 rows of global ids, decay applied.  World 1 (the whole graph
        is this rank's): the reference's list of L+1 ``[n, d]`` tensors, as on the plain module, ids checked against
        the global node count.  World > 1 (peer data plane; all ranks call it together): this rank reads its positional
        slice of ``node_ids`` and returns ``(positions, [L+1 tensors of shape rows x d])``; ``gather=True`` returns the
        reference's list on every rank (one all_gather; collective, no gradient — the layers have none anyway)."""
        self._check_node_call('get_random_projections')
        dev = self._require_cuda()
        n = int(len(node_ids))
        if self.world == 1:
            ptr = self._rank_ids_to_device([node_ids], ['id'])[0] if n else 0
            out = self._gather_state_rows(ptr, n)
            return [out[i] for i in range(self.num_layer + 1)]
        per, lo, hi = self._row_split(n)
        rows = self._route_node_rows(node_ids[lo:hi])
        out = self._gather_state_rows(rows.data_ptr(), hi - lo)
        if gather:
            full = self._gather_slices(out.transpose(0, 1), per, n).transpose(0, 1).contiguous()
            return [full[i] for i in range(self.num_layer + 1)]
        return self._positions(lo, hi), [out[i] for i in range(self.num_layer + 1)]

    # ------------------------------------------------------------------ state changes invalidate the remote-row caches
    def _before_write(self) -> None:
        """A write to the local rows outside update(): every peer must have finished the pulls it issued before."""
        if self.exchange == 'peer' and self.world > 1 and self._state.is_cuda:
            self._barrier()

    def reset_random_projections(self):
        self._before_write()
        super().reset_random_projections()         # tpn_clear_walk_layers also sets every stamp to -1
        self._state_written()

    def reload_random_projections(self, random_projections):
        self._before_write()
        super().reload_random_projections(random_projections)
        self._state_written()

    def materialize(self) -> None:
        """Collective in the peer data plane (every rank calls it at the same point, as backup / state_dict do):
        the write-back of the pending decay must not race with a peer's pull."""
        if self.exchange != 'peer' or self.world == 1 or not self._state.is_cuda:
            return super().materialize()
        self._before_write()
        super().materialize()
        self._state_written()

    def _restart_log(self) -> None:
        super()._restart_log()                     # every row rewritten, stamps restarted: cached copies are stale
        self._state_written()

    def check_errors(self) -> None:
        super().check_errors()
        if self._shard is not None:
            code = int(self._shard_tensors['counters'][_lib.SHARD_CTR_ERROR].item())
            if code:
                self._shard_tensors['counters'][_lib.SHARD_CTR_ERROR] = 0
                if code == 1:
                    raise IndexError(f'node id out of range for node_num {self.global_node_num} in a sharded batch')
                if code == 2:
                    raise RuntimeError(f'the {self.ext_rows} extension rows cannot hold the remote rows of one '
                                       f'generation: construct ShardedRandomProjection with a larger ext_rows')
                raise RuntimeError('a peer rank never reached a barrier of the sharded data plane')

    def gather_global(self) -> List[torch.Tensor]:
        """All-gathers the L+1 global [N, d] matrices (tests / small graphs only)."""
        self.materialize()
        out = []
        for i in range(self.num_layer + 1):
            mine = self.random_projections[i].data[:self.n_local].contiguous()
            full = torch.zeros(self.global_node_num, self.dim, dtype=torch.float32, device=mine.device)
            if self.world == 1:
                full.copy_(mine)
            else:
                pad = rows_on_rank(self.global_node_num, self.world, 0)
                buf = torch.zeros(pad, self.dim, dtype=torch.float32, device=mine.device)
                buf[:self.n_local].copy_(mine)
                parts = [torch.empty_like(buf) for _ in range(self.world)]
                dist.all_gather(parts, buf, group=self.group)
                for r in range(self.world):
                    n_r = rows_on_rank(self.global_node_num, self.world, r)
                    full[r::self.world] = parts[r][:n_r]
            out.append(full)
        return out
