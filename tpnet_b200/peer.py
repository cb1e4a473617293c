"""Peer-visible device memory for the node-sharded state (tpnet_b200/sharded.py, SURVEY.md §8e).

The sharded data plane reads other ranks' rows straight out of their HBM over NVLink, so every rank's state,
stamps and barrier words must be mapped into every other rank's address space:

  * ``PeerBuffer``      — peer-visible device memory, handed to PyTorch as a tensor.  ``symmetric=True`` (what a
                          one-process-per-GPU job uses): ``torch.distributed._symmetric_memory.empty`` —
                          cuMemCreate / cuMemMap allocations with 2 MiB pages.  Otherwise memory owned by the
                          library (``tpn_peer_alloc``: plain ``cudaMalloc``, exportable with legacy CUDA IPC),
                          viewed through ``__cuda_array_interface__``.
  * ``SymmPeerGroup``   — one process per GPU (torchrun), the default: ``symmetric_memory.rendezvous`` maps every
                          rank's buffer into every other rank and returns plain device pointers.  MEASURED
                          (scripts/peer_probe.py, profiles/r02_peer_probe.json): random 3.4 KB row blocks out of a
                          14 GB peer buffer are pulled at 640 GB/s through this mapping, but only at 171 GB/s
                          through a legacy-IPC mapping of the same buffer (consecutive rows: 647 GB/s on both) —
                          the IPC mapping is TLB-bound for random access.
  * ``IpcPeerGroup``    — the same rendezvous with legacy CUDA IPC handles (``cudaIpcOpenMemHandle``), kept for
                          setups without symmetric-memory support; see the measurement above.
  * ``LocalPeerGroup``  — all ranks inside ONE process (several ranks may even share one GPU): the "peer"
                          pointers are simply the other ranks' pointers.  This is how the single-GPU test box
                          runs the complete routed data plane (routing, pulls, barriers, device-side counts);
                          only the NVLink transport itself needs more than one GPU.

``PeerShardMember`` is the rank-local side of that protocol, shared by the sharded state and the sharded sampler.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib

_TYPESTR = {torch.float32: '<f4', torch.int32: '<i4', torch.uint8: '|u1', torch.int64: '<i8', torch.float64: '<f8'}
_ITEMSIZE = {torch.float32: 4, torch.int32: 4, torch.uint8: 1, torch.int64: 8, torch.float64: 8}


class PeerBuffer:
    """Zero-filled device memory from ``tpn_peer_alloc`` on ``device``; ``tensor(shape, dtype)`` views it."""

    def __init__(self, nbytes: int, device: torch.device, symmetric: bool = False):
        self._lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('peer-visible memory lives on CUDA devices only')
        self.nbytes = (max(int(nbytes), 16) + 15) // 16 * 16
        self.symmetric = bool(symmetric)
        self._t = None
        if self.symmetric:
            import torch.distributed._symmetric_memory as symm_mem
            self._t = symm_mem.empty(self.nbytes, dtype=torch.uint8, device=self.device)
            self._t.zero_()
            self.ptr = int(self._t.data_ptr())
            return
        ptr = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.tpn_peer_alloc(ctypes.byref(ptr), self.nbytes), 'tpn_peer_alloc')
        self.ptr = int(ptr.value)

    def tensor(self, shape, dtype: torch.dtype) -> torch.Tensor:
        numel = 1
        for s in shape:
            numel *= int(s)
        if numel * _ITEMSIZE[dtype] > self.nbytes:
            raise ValueError('view larger than the buffer')
        if self._t is not None:
            return self._t[:numel * _ITEMSIZE[dtype]].view(dtype).view(*[int(s) for s in shape])
        holder = _ArrayView(self, tuple(int(s) for s in shape), _TYPESTR[dtype])
        return torch.as_tensor(holder, device=self.device)

    def ipc_handle(self) -> bytes:
        buf = (ctypes.c_ubyte * 64)()
        _lib.check(self._lib.tpn_ipc_export(self.ptr, buf), 'tpn_ipc_export')
        return bytes(buf)

    def __del__(self):
        try:
            if getattr(self, '_t', None) is not None:
                self._t = None
                self.ptr = 0
            elif getattr(self, 'ptr', 0):
                self._lib.tpn_peer_free(self.ptr)
                self.ptr = 0
        except Exception:  # interpreter shutdown
            pass


class _ArrayView:
    """What ``torch.as_tensor`` consumes; keeps the buffer alive as long as the tensor lives."""

    def __init__(self, buf: PeerBuffer, shape, typestr: str):
        self._buf = buf
        self.__cuda_array_interface__ = {'shape': shape, 'typestr': typestr, 'data': (buf.ptr, False), 'version': 2,
                                         'strides': None}


class PeerGroup:
    """Rendezvous of the per-rank buffers of one sharded module."""
    world: int
    rank: int

    def exchange(self, name: str, buf: PeerBuffer) -> List[int]:
        """Device pointers, valid in THIS process, of every rank's buffer ``name`` (index = rank)."""
        raise NotImplementedError

    def barrier(self) -> None:
        """Host-level barrier (set-up only; the data path uses tpn_peer_barrier)."""


class LocalPeerGroup(PeerGroup):
    """All ranks in one process.  ``LocalPeerGroup.create(world)`` returns one view per rank; every rank
    registers its buffers (``publish``) before any of them resolves the table (``exchange``).

    ``host_barriers``: ranks that share ONE GPU cannot use the spinning flag barrier (``tpn_peer_barrier``): a
    kernel of rank A that waits for rank B can sit in front of rank B's work in the same hardware queue.  The
    driver of the ranks orders the phases instead — every rank finishes its reads (``update_begin``, pair-wise
    calls) before any rank writes (``update_end``) — and the module skips the device barrier."""
    host_barriers = True

    def __init__(self, world: int, rank: int, table: Dict[str, List[Optional[int]]]):
        self.world, self.rank, self._table = int(world), int(rank), table

    @staticmethod
    def create(world: int) -> List['LocalPeerGroup']:
        table: Dict[str, List[Optional[int]]] = {}
        return [LocalPeerGroup(world, r, table) for r in range(world)]

    def publish(self, name: str, buf: PeerBuffer) -> None:
        self._table.setdefault(name, [None] * self.world)[self.rank] = buf.ptr

    def exchange(self, name: str, buf: PeerBuffer) -> List[int]:
        self.publish(name, buf)
        ptrs = self._table[name]
        missing = [r for r, p in enumerate(ptrs) if p is None]
        if missing:
            raise RuntimeError(f'ranks {missing} have not published "{name}" yet: construct every rank, then connect()')
        return [int(p) for p in ptrs]


class SymmPeerGroup(PeerGroup):
    """One process per GPU: torch symmetric memory maps every rank's buffer into every other rank (2 MiB pages).
    Buffers must be ``PeerBuffer(..., symmetric=True)`` of the same size on every rank; ``exchange`` is collective."""
    symmetric = True

    def __init__(self, group=None):
        self._dist = dist
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self._handles = []

    def exchange(self, name: str, buf: PeerBuffer) -> List[int]:
        import torch.distributed._symmetric_memory as symm_mem
        if buf._t is None:
            raise ValueError('SymmPeerGroup needs PeerBuffer(..., symmetric=True)')
        hdl = symm_mem.rendezvous(buf._t, self.group)
        self._handles.append(hdl)
        ptrs = [int(p) for p in hdl.buffer_ptrs]
        if len(ptrs) != self.world or ptrs[self.rank] != buf.ptr:
            raise RuntimeError(f'symmetric-memory rendezvous of "{name}" returned an unexpected pointer table')
        return ptrs

    def barrier(self) -> None:
        self._dist.barrier(group=self.group)

    def close(self) -> None:
        self._handles = []


class IpcPeerGroup(PeerGroup):
    """One process per GPU: pointers of the other ranks' buffers through legacy CUDA IPC (see the module docstring
    for why this is not the default)."""

    def __init__(self, group=None):
        self._dist = dist
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self._opened: List[int] = []
        self._lib = _lib.load()

    def exchange(self, name: str, buf: PeerBuffer) -> List[int]:
        handles: List[Optional[bytes]] = [None] * self.world
        self._dist.all_gather_object(handles, (name, buf.ipc_handle()), group=self.group)
        out = []
        with torch.cuda.device(buf.device):
            for r, item in enumerate(handles):
                if r == self.rank:
                    out.append(buf.ptr)
                    continue
                peer_name, handle = item
                if peer_name != name:
                    raise RuntimeError(f'rank {r} exchanged "{peer_name}" while rank {self.rank} exchanged "{name}"')
                ptr = ctypes.c_void_p()
                raw = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
                _lib.check(self._lib.tpn_ipc_open(raw, ctypes.byref(ptr)), f'tpn_ipc_open (buffer "{name}" of rank {r})')
                self._opened.append(int(ptr.value))
                out.append(int(ptr.value))
        return out

    def barrier(self) -> None:
        self._dist.barrier(group=self.group)

    def close(self) -> None:
        for p in self._opened:
            self._lib.tpn_ipc_close(p)
        self._opened = []


def rows_on_rank(node_num: int, world: int, rank: int) -> int:
    """Number of global ids u < node_num with u % world == rank (node u lives on rank u % world, row u // world)."""
    return (node_num - rank + world - 1) // world if node_num > rank else 0


class PeerShardMember:
    """One rank of a node-sharded module with a peer data plane: the rank-local side of the "Barrier protocol" of
    include/tpnet_b200.h, shared by ``ShardedRandomProjection`` and ``ShardedStreamingSampler``.

    The owner calls ``_join`` first (world, rank, ``n_local``), allocates its peer-visible memory with
    ``_peer_buffer`` and ``_init_shard`` (the flags buffer and the routing shard: mark table, counters, need list and
    barrier sequence in ``_shard_tensors``, described by the ``tpn_shard_t`` ``_shard``), and turns the exchanged base
    pointers into its own tables in ``_connect_tables``.  A module without a peer data plane (world 1, or the 'nccl'
    plane of the state) calls ``_join`` only: ``_shard`` stays None and nothing peer-visible is allocated."""

    def _join(self, node_num: int, peers: Optional[PeerGroup], group) -> None:
        """World and rank from ``peers``, else from torch.distributed (world 1 without it); the rows this rank owns."""
        if peers is not None:
            self.world, self.rank = int(peers.world), int(peers.rank)
        else:
            self.world = dist.get_world_size(group) if dist.is_initialized() else 1
            self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.group = group
        self._peers = peers
        self.n_local = rows_on_rank(node_num, self.world, self.rank)
        self._peer_bufs: Dict[str, PeerBuffer] = {}
        self._shard: Optional[_lib.TpnShard] = None
        self._shard_tensors = {}
        self._connected = False
        self._route = {}                 # cached device buffers, keyed by (kind, ...)
        self._dirty = True               # a rank may have written since the last barrier: barrier before pulling
        self.barriers = 0                # barriers issued so far (bench accounting)

    def _peer_buffer(self, name: str, nbytes: int, device) -> PeerBuffer:
        """Zero-filled peer-visible buffer ``name``.  ``nbytes`` must be the same on every rank (symmetric memory
        needs it).  In-process ranks publish it at once, so every rank constructed can connect."""
        symmetric = self._peers is None or getattr(self._peers, 'symmetric', False)
        buf = self._peer_bufs[name] = PeerBuffer(nbytes, device, symmetric=symmetric)
        if isinstance(self._peers, LocalPeerGroup):
            self._peers.publish(name, buf)
        return buf

    def _init_shard(self, device, global_nodes: int, ext_rows: int, flags: str,
                    shard: Optional[_lib.TpnShard] = None) -> None:
        """The flags buffer ``flags`` (one barrier word per rank) and the routing shard over ``global_nodes`` ids with
        ``ext_rows`` cache rows, described in ``shard`` (a new ``TpnShard`` unless the owner embeds one)."""
        self._flags_name = flags
        self._peer_buffer(flags, 4 * max(self.world, 16), device)
        t = self._shard_tensors
        t['mark'] = torch.zeros(global_nodes, dtype=torch.int32, device=device)
        t['counters'] = torch.zeros(_lib.SHARD_COUNTERS, dtype=torch.int32, device=device)
        t['need'] = torch.zeros(max(ext_rows, 1), dtype=torch.int64, device=device)
        t['seq'] = torch.zeros(1, dtype=torch.int32, device=device)
        sh = shard if shard is not None else _lib.TpnShard()
        sh.world, sh.rank, sh.global_nodes = self.world, self.rank, global_nodes
        sh.num_local_rows, sh.ext_rows = self.n_local, ext_rows
        sh.mark, sh.counters = t['mark'].data_ptr(), t['counters'].data_ptr()
        sh.need_nodes, sh.barrier_seq = t['need'].data_ptr(), t['seq'].data_ptr()
        self._shard = sh

    def _connect_tables(self, bases: Dict[str, List[int]]) -> Dict[str, torch.Tensor]:
        """The owner's device tables built from every rank's base pointer of each of its buffers (flags excluded),
        written into its C structs; returned to be kept alive in ``_shard_tensors['tables']``."""
        raise NotImplementedError

    def connect(self) -> None:
        """Rendezvous of the peer-visible buffers (collective over the ranks; the first call that needs the peers does
        it if the caller did not).  With a ``LocalPeerGroup`` every rank must be constructed first."""
        if self._shard is None or self._connected:
            return
        if self._peers is None:
            if not dist.is_initialized():
                raise RuntimeError(f'{type(self).__name__} with world > 1 needs torch.distributed or a PeerGroup')
            self._peers = SymmPeerGroup(self.group)
        bases = {name: self._peers.exchange(name, buf) for name, buf in self._peer_bufs.items()}
        flags = torch.tensor(bases.pop(self._flags_name), dtype=torch.int64, device=self._shard_tensors['mark'].device)
        tables = dict(self._connect_tables(bases), flags=flags)
        self._shard.peer_flags = flags.data_ptr()
        self._shard_tensors['tables'] = tables
        self._connected = True
        self._peers.barrier()            # every rank has mapped every buffer before anyone launches a pull

    def close(self) -> None:
        """Collective teardown of the peer data plane: every rank stops using its peers' memory, unmaps it, and only
        then may anyone free its buffers (freeing an exported allocation that a peer still maps is undefined).  Call
        it on every rank before dropping the module when another sharded module will be created in the same job."""
        if not self._connected:
            return
        torch.cuda.synchronize(self._shard_tensors['mark'].device)
        self._peers.barrier()
        if hasattr(self._peers, 'close'):
            self._peers.close()
        self._peers.barrier()
        self._connected = False
        del self._shard_tensors['tables']

    def __del__(self):
        try:                                       # best effort without the barriers (interpreter shutdown, errors)
            if getattr(self, '_connected', False) and hasattr(self._peers, 'close'):
                self._peers.close()
        except Exception:
            pass

    def _c_shard(self):
        """byref of the ``tpn_shard_t``, connected."""
        if not self._connected:
            self.connect()
        return ctypes.byref(self._shard)

    def _barrier(self) -> None:
        self.barriers += 1
        if getattr(self._peers, 'host_barriers', False):
            return          # LocalPeerGroup: the driver of the in-process ranks orders the phases itself
        _lib.check(_lib.load().tpn_peer_barrier(self._c_shard(), self._stream()), 'tpn_peer_barrier')

    def _before_pull(self) -> None:
        """Peers' writes are ordered before this rank's reads of their rows: one barrier after any write."""
        if self._dirty:
            self._barrier()
            self._dirty = False

    def _take_shard_error(self, out_of_range: str, cache_full: str, no_barrier: str) -> Optional[Exception]:
        """Reads and clears the sticky routing error ``counters[SHARD_CTR_ERROR]``; the exception it stands for, with
        the owner's text: IndexError for an id outside the graph (1), RuntimeError when one generation's remote rows do
        not fit the cache (2) or a peer never reached a barrier (3)."""
        if self._shard is None:
            return None
        ctr = self._shard_tensors['counters']
        code = int(ctr[_lib.SHARD_CTR_ERROR].item())
        if code == 0:
            return None
        ctr[_lib.SHARD_CTR_ERROR] = 0
        if code == 1:
            return IndexError(out_of_range)
        return RuntimeError(cache_full if code == 2 else no_barrier)

    def row_split(self, m: int) -> Tuple[int, int, int]:
        """(per, lo, hi): this rank computes rows [lo, hi) of a call with m rows, per = ceil(m / world)."""
        per = -(-m // self.world)
        lo = min(self.rank * per, m)
        return per, lo, min(lo + per, m)

    def _positions(self, lo: int, hi: int, device) -> torch.Tensor:
        """Device int64 [lo, hi) (cached: the same split recurs every batch)."""
        key = ('positions', lo, hi)
        t = self._route.get(key)
        if t is None:
            if len(self._route) > 8:
                self._route.clear()
            t = self._route[key] = torch.arange(lo, hi, dtype=torch.int64, device=device)
        return t
