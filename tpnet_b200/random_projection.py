"""Drop-in replacement for the reference's ``RandomProjectionModule``
(``/root/reference/models/TPNet.py:9-157``) backed by the sm_100a CUDA library.

Same constructor arguments, attributes, ``state_dict`` keys and method names as
the reference, so ``train_link_prediction.py`` / ``evaluate_link_prediction.py``
run on it unmodified (see INTEGRATION.md for the two-line patch).  All arithmetic
of the hot path runs in the hand-written kernels reached through the C ABI
(``include/tpnet_b200.h``); PyTorch only owns memory, streams and the trainable
``self.mlp`` head.  There is no CPU path: calling a compute method while the
state is not on a CUDA device raises.

Differences a caller can observe (documented, none on the reference's own call
sites):
  * the L+1 projection matrices live in ONE packed node-major buffer
    ``[N, L+1, row_stride]``; ``self.random_projections[i]`` are strided ``[N, d]``
    views of it (values, shapes, dtypes and state_dict keys are the reference's);
  * ``decay_mode='lazy'`` defers the per-update whole-matrix rescale
    (TPNet.py:83-85) to the rows that are touched (one multiply by the product of
    the skipped factors: same value up to one fp32 rounding per skipped update,
    identical when at most one update was skipped); reads through this class's
    methods are always current, raw reads of ``random_projections[i]`` need
    ``materialize()`` first (``state_dict()`` and ``backup_…`` do it themselves);
  * ids may also be passed as int64 CUDA tensors (device-resident pipelines).
"""
from __future__ import annotations

import ctypes
import math
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import TpnState

IdArray = Union[np.ndarray, torch.Tensor]

#: state size above which 'auto' picks lazy decay (the eager sweep of a state
#: this small stays in L2 and costs a few microseconds)
AUTO_LAZY_BYTES = 256 << 20
_DEFAULT_LOG_EPOCHS = 4096


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


class _Stager:
    """Thin owner of the C-side pinned staging ring (csrc/tpn_stage.cu): one ctypes call copies
    the per-call id / timestamp arrays into pinned memory (validating ids on the way) and issues
    one async H2D copy on the current stream."""

    def __init__(self, dev_index: int, slot_bytes: int = 1 << 20, slots: int = 8):
        self._lib = _lib.load()
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(dev_index):       # the ring's device slots live on the module's device
            _lib.check(self._lib.tpn_stager_create(ctypes.byref(self.handle), slot_bytes, slots), 'tpn_stager_create')
        self.host = (ctypes.c_void_p * 8)()
        self.elems = (ctypes.c_int64 * 8)()
        self.kinds = (ctypes.c_int * 8)()
        self.out = (ctypes.c_void_p * 8)()

    def upload(self, arrays: Sequence[np.ndarray], kinds: Sequence[int], num_nodes: int, stream: int) -> List[int]:
        for i, a in enumerate(arrays):
            self.host[i] = a.__array_interface__['data'][0]
            self.elems[i] = a.shape[0]
            self.kinds[i] = kinds[i]
        rc = self._lib.tpn_stage(self.handle, self.host, self.elems, self.kinds, len(arrays), num_nodes, self.out,
                                 stream)
        if rc:
            if rc == _lib.TPN_ERR_INDEX:
                raise IndexError(f'index out of range for node_num {num_nodes}')
            _lib.check(rc, 'tpn_stage')
        return [self.out[i] for i in range(len(arrays))]

    def __del__(self):
        try:
            if self.handle:
                self._lib.tpn_stager_destroy(self.handle)
                self.handle = ctypes.c_void_p()
        except Exception:  # interpreter shutdown
            pass


class _Host:
    """Mutable host-side bookkeeping kept off the nn.Module (its __setattr__ is slow)."""
    __slots__ = ('now', 'begin', 'epoch', 'launches', 'stager', 'stager2', 'st', 'st_ref', 'dev_index', 'keepalive',
                 'device_ids_seen')

    def __init__(self, t0: float):
        self.now = t0
        self.begin = t0
        self.epoch = 0
        self.launches = 0
        self.stager: Optional[_Stager] = None
        self.stager2: Optional[_Stager] = None       # ring of the calls issued on the feature stream
        self.st: Optional[TpnState] = None
        self.st_ref = None
        self.dev_index = -1
        self.keepalive = None
        self.device_ids_seen = False     # a device-resident id array was used since the last check_errors()


class RandomProjectionModule(nn.Module):
    def __init__(self, node_num: int, edge_num: int, dim_factor: int, num_layer: int, time_decay_weight: float,
                 device: str, use_matrix: bool, beginning_time: np.float64, not_scale: bool, enforce_dim: int,
                 decay_mode: str = 'auto', init_p0: bool = True, state_device=None,
                 accumulation: str = 'reference', giant_chunk: int = 1024,
                 state_buffer: Optional[torch.Tensor] = None, p0_seed: Optional[int] = None):
        """Arguments as the reference constructor (TPNet.py:10-26).  ``decay_mode`` in
        {'auto', 'eager', 'lazy'} selects how the time decay of TPNet.py:83-85 is
        realised; all modes produce the same values.  ``init_p0=False`` leaves P_0 zero for the
        caller to fill and ``state_device`` allocates the packed state directly on a device
        (both for states too large to stage through host memory).  ``accumulation`` selects the order
        in which the messages of ONE target row are added inside an update: ``'reference'`` (default)
        adds them one at a time in the reference's order (CPU ``scatter_add_``, TPNet.py:93-96), bit for
        bit; ``'chunked'`` cuts the messages of a row that receives >= 2048 of them in one call into
        chunks of ``giant_chunk``, sums each chunk in order and adds the chunk sums in order —
        deterministic, within fp32 rounding of the reference order (include/tpnet_b200.h,
        ``tpn_state_t::giant_chunk``), and free of the hub's sequential add chain.  ``state_buffer``: a
        zero-filled float32 tensor ``[node_num, num_layer + 1, row_stride]`` to use as the packed state
        (the sharded module passes peer-visible memory).  ``p0_seed``: an int in [0, 2^64) draws P_0 on the state's
        device from the counter-based generator of ``tpn_init_projection`` (include/tpnet_b200.h) instead of torch's
        RNG — draw 0 here, draw ``p0_draw`` after ``p0_draw`` resets — so every placement of the rows, sharded at any
        world size or not, holds the same bits; no torch RNG state is consumed.  Needs ``state_device`` on CUDA."""
        super().__init__()
        if p0_seed is not None:
            if use_matrix:
                raise ValueError('p0_seed: use_matrix has P_0 = I, there is nothing to draw')
            if not init_p0:
                raise ValueError('p0_seed draws P_0: it cannot be combined with init_p0=False')
            sdev = state_buffer.device if state_buffer is not None else (
                torch.device(state_device) if state_device is not None else None)
            if sdev is None or sdev.type != 'cuda':
                raise ValueError('p0_seed draws P_0 on the GPU: create the state there with state_device')
            if not 0 <= int(p0_seed) < 1 << 64:
                raise ValueError('p0_seed must be in [0, 2^64)')
        self.p0_seed = None if p0_seed is None else int(p0_seed)
        self.p0_draw = 0
        if not 1 <= num_layer <= _lib.TPN_MAX_LAYERS:
            raise ValueError(f'num_layer must be in 1..{_lib.TPN_MAX_LAYERS}')
        if decay_mode not in ('auto', 'eager', 'lazy'):
            raise ValueError("decay_mode must be 'auto', 'eager' or 'lazy'")
        if accumulation not in ('reference', 'chunked'):
            raise ValueError("accumulation must be 'reference' or 'chunked'")
        if accumulation == 'chunked' and not (256 <= giant_chunk <= 2048 and giant_chunk % 32 == 0):
            raise ValueError('giant_chunk must be a multiple of 32 in 256..2048')
        self.accumulation = accumulation
        self.giant_chunk = int(giant_chunk)
        self.node_num = node_num
        self.edge_num = edge_num
        if enforce_dim != -1:                                             # TPNet.py:30-33
            self.dim = enforce_dim
        else:
            self.dim = min(int(math.log(self.edge_num * 2)) * dim_factor, node_num)
        self.num_layer = num_layer
        self.time_decay_weight = time_decay_weight
        self.begging_time = nn.Parameter(torch.tensor(beginning_time), requires_grad=False)   # (sic) TPNet.py:36
        self.now_time = nn.Parameter(torch.tensor(beginning_time), requires_grad=False)
        self.device = device
        self.use_matrix = use_matrix
        self.node_feature_dim = 128
        self.not_scale = not_scale
        if self.use_matrix:                                               # TPNet.py:44-45
            self.dim = self.node_num
        self.row_stride = _round_up(self.dim, 8)          # 32-byte sectors; pad columns stay zero
        self.node_stride = (self.num_layer + 1) * self.row_stride
        self.decay_mode = decay_mode

        # packed node-major state; P_l[u] = _state[u, l, :dim]
        if state_buffer is not None:
            if state_buffer.shape != (self.node_num, self.num_layer + 1, self.row_stride) or \
                    state_buffer.dtype != torch.float32 or not state_buffer.is_contiguous():
                raise ValueError('state_buffer must be a contiguous float32 [node_num, num_layer + 1, row_stride] tensor')
            self._state = state_buffer
        else:
            self._state = torch.zeros(self.node_num, self.num_layer + 1, self.row_stride, dtype=torch.float32,
                                      device=state_device)
        if self.use_matrix:
            self._state[:, 0, :self.dim] = torch.eye(self.node_num)      # TPNet.py:48-49
        elif init_p0 and self.p0_seed is None:
            # same RNG call as TPNet.py:58 so a seeded run draws the same P_0
            self._state[:, 0, :self.dim] = torch.normal(0, 1 / math.sqrt(self.dim), (self.node_num, self.dim))
        self.random_projections = nn.ParameterList(
            [nn.Parameter(self._state[:, i, :self.dim], requires_grad=False) for i in range(self.num_layer + 1)])
        self.pair_wise_feature_dim = (2 * self.num_layer + 2) ** 2        # TPNet.py:63
        self.mlp = nn.Sequential(nn.Linear(self.pair_wise_feature_dim, self.pair_wise_feature_dim * 4), nn.ReLU(),
                                 nn.Linear(self.pair_wise_feature_dim * 4, self.pair_wise_feature_dim))

        # host mirrors / device scratch (not part of state_dict)
        self._h = _Host(float(beginning_time))
        if self._state.is_cuda:
            self._h.dev_index = self._state.device.index if self._state.device.index is not None \
                else torch.cuda.current_device()
        self._stamps: Optional[torch.Tensor] = None
        self._decay_log: Optional[torch.Tensor] = None
        self._ws: Optional[torch.Tensor] = None
        self._ws_batch = 0
        self._err: Optional[torch.Tensor] = None
        self._pending = None            # update_prepare: (array ids, n, next_time, C arguments) of the half in flight
        self._prep_stream: Optional[torch.cuda.Stream] = None
        self._prep_done: Optional[torch.cuda.Event] = None
        self._feature_stream: Optional[torch.cuda.Stream] = None
        self.validate_ids = True
        self.fused_head = True          # no-grad calls: fused fp32 head kernel when the head has the default shape
        self.register_state_dict_pre_hook(lambda module, prefix, keep_vars: module.materialize())
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._after_external_write())
        if self.p0_seed is not None:
            self._write_counter_p0()

    # ------------------------------------------------------------------ plumbing
    @property
    def _now_host(self) -> float:
        return self._h.now

    @property
    def launches(self) -> int:
        """C-ABI calls that launched kernels so far (bench accounting)."""
        return self._h.launches

    @property
    def lazy(self) -> bool:
        if self.decay_mode == 'auto':
            return self._state.numel() * 4 > AUTO_LAZY_BYTES
        return self.decay_mode == 'lazy'

    def _apply(self, fn, recurse=True):
        # nn.Module.to()/cuda()/cpu(): parameters are converted one by one (the views
        # become independent tensors); gather them back into one packed buffer.
        super()._apply(fn, recurse)
        self._repack()
        return self

    def _is_packed(self) -> bool:
        st = self._state
        for i, p in enumerate(self.random_projections):
            if (p.device != st.device or p.dtype != torch.float32 or p.shape != (self.node_num, self.dim)
                    or p.stride() != (self.node_stride, 1)
                    or p.data_ptr() != st.data_ptr() + 4 * i * self.row_stride):
                return False
        return True

    def _repack(self) -> None:
        if self._is_packed():
            return
        dev = self.random_projections[0].device
        for p in self.random_projections:
            if p.dtype != torch.float32:
                raise TypeError('RandomProjectionModule state must stay float32')
        new_state = torch.zeros(self.node_num, self.num_layer + 1, self.row_stride, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for i, p in enumerate(self.random_projections):
                new_state[:, i, :self.dim].copy_(p.data)
                p.data = new_state[:, i, :self.dim]
        self._state = new_state
        self._stamps = None
        self._decay_log = None
        self._cancel_prepare()
        self._ws = None
        self._ws_batch = 0
        self._err = None
        self._h.epoch = 0
        self._h.st = None
        self._h.stager = None
        self._h.dev_index = dev.index if dev.type == 'cuda' and dev.index is not None else (
            torch.cuda.current_device() if dev.type == 'cuda' else -1)

    def _after_external_write(self) -> None:
        """load_state_dict / reload wrote fully materialised values: refresh mirrors."""
        self._repack()
        self._h.now = float(self.now_time.item())
        self._h.begin = float(self.begging_time.item())
        if self._stamps is not None:
            self._stamps.zero_()
        self._h.epoch = 0

    def _require_cuda(self) -> torch.device:
        dev = self._state.device
        if dev.type != 'cuda':
            raise RuntimeError('tpnet_b200.RandomProjectionModule computes on CUDA only (no CPU fallback): '
                               'move the module with .to("cuda") first')
        return dev

    def _stream(self) -> int:
        h = self._h
        if h.dev_index < 0:
            dev = self._state.device
            h.dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        return torch._C._cuda_getCurrentRawStream(h.dev_index)

    def _c_state(self):
        """ctypes view of the state (cached; rebuilt when a buffer changes). Returns byref(struct)."""
        h = self._h
        st = h.st
        if st is None:
            st = TpnState()
            st.data = self._state.data_ptr()
            st.num_nodes = self.node_num
            st.num_layer = self.num_layer
            st.dim = self.dim
            st.row_stride = self.row_stride
            st.node_stride = self.node_stride
            if self.lazy:
                if self._stamps is None:
                    # -1 = row known to be all zero (never written); rows holding data start at epoch 0
                    has_data = bool((self._state[:, 1:, :] != 0).any().item()) if self._state.numel() else False
                    self._stamps = torch.full((self.node_num, self.num_layer), 0 if has_data else -1,
                                              dtype=torch.int32, device=self._state.device)
                    # f64 cumulative products of the per-update fp32 factors; row 0 = 1.0
                    self._decay_log = torch.ones(_DEFAULT_LOG_EPOCHS, self.num_layer, dtype=torch.float64,
                                                 device=self._state.device)
                    h.epoch = 0
                st.stamps = self._stamps.data_ptr()
                st.decay_log = self._decay_log.data_ptr()
                st.log_capacity = self._decay_log.shape[0]
                st.cum_floor = 1.0
            else:
                st.stamps = None
                st.decay_log = None
                st.log_capacity = 0
            if self._err is None:
                self._err = torch.zeros(1, dtype=torch.int32, device=self._state.device)
            st.err_flag = self._err.data_ptr()
            st.giant_chunk = self.giant_chunk if self.accumulation == 'chunked' else 0
            h.st = st
            h.st_ref = ctypes.byref(st)
        st.epoch = h.epoch
        return h.st_ref

    def _ids_to_device(self, arrays: Sequence[IdArray], kinds: Sequence[str], wrap_negative: bool = True) -> List[int]:
        """Returns device addresses for id (int64) / time (float64) arrays given as
        numpy arrays (staged through pinned memory) or CUDA tensors (used in place)."""
        dev = self._state.device
        if isinstance(arrays[0], torch.Tensor) and all(isinstance(a, torch.Tensor) and a.is_cuda for a in arrays):
            out = []
            for a, kind in zip(arrays, kinds):
                want = torch.int64 if kind == 'id' else torch.float64
                if a.device != dev or a.dtype != want or not a.is_contiguous():
                    raise TypeError(f'device-resident {kind} arrays must be contiguous {want} tensors on {dev}')
                out.append(a.data_ptr())
            self._h.keepalive = arrays
            self._h.device_ids_seen = True
            return out
        host, ck = [], []
        id_kind = _lib.STAGE_ID_WRAP if wrap_negative else _lib.STAGE_ID
        if not self.validate_ids:
            id_kind = _lib.STAGE_RAW
        for a, kind in zip(arrays, kinds):
            if isinstance(a, torch.Tensor):
                a = a.detach().cpu().numpy()
            want = np.int64 if kind == 'id' else np.float64
            if not (isinstance(a, np.ndarray) and a.dtype == want and a.ndim == 1 and a.flags.c_contiguous):
                a = np.ascontiguousarray(a, dtype=want).reshape(-1)
            host.append(a)
            ck.append(id_kind if kind == 'id' else _lib.STAGE_RAW)
        h = self._h
        raw = self._stream()                            # also resolves dev_index
        if self._feature_stream is not None and raw == self._feature_stream.cuda_stream:
            # a staging ring orders the reuse of its slots against ONE caller stream: calls on the feature stream
            # (pipeline.tpnet_step) get their own
            if h.stager2 is None:
                h.stager2 = _Stager(h.dev_index)
            return h.stager2.upload(host, ck, self.node_num, raw)
        if h.stager is None:
            h.stager = _Stager(h.dev_index)
        return h.stager.upload(host, ck, self.node_num, raw)

    # ------------------------------------------------------------------ reference API
    def _cancel_prepare(self) -> None:
        """A prepared half (update_prepare) is dropped before anything else rewrites the state or its bookkeeping;
        the next update then runs whole."""
        if getattr(self, '_pending', None) is not None:
            torch.cuda.current_stream(self._state.device).wait_event(self._prep_done)
            self._pending = None

    def _update_args(self, src_node_ids: IdArray, dst_node_ids: IdArray, node_interact_times: IdArray,
                     next_time: Optional[float]):
        """Host half of TPNet.py:67-99: argument checks, the f64 decay factors, ids / timestamps on the device, the
        workspace.  Returns (n, next_time, C arguments after the state pointer and before the stream)."""
        dev = self._require_cuda()
        lib = _lib.load()
        n = int(len(src_node_ids))
        if n == 0:
            raise IndexError('index -1 is out of bounds for axis 0 with size 0')      # what TPNet.py:76 raises
        if len(dst_node_ids) != n or len(node_interact_times) != n:
            raise ValueError('src, dst and time arrays must have the same length')
        if next_time is None:
            last = node_interact_times[-1]
            next_time = float(last.item()) if isinstance(last, torch.Tensor) else float(last)
        lam = self.time_decay_weight
        # c_l = f32(pow(exp(-lambda*(t_last - now)), l)) computed in f64 on the host, TPNet.py:84-85
        h = self._h
        base = np.exp(-lam * (np.float64(next_time) - np.float64(h.now)))
        factors = (ctypes.c_float * self.num_layer)(*[float(np.float32(np.power(base, i)))
                                                      for i in range(1, self.num_layer + 1)])
        ptrs = self._ids_to_device([src_node_ids, dst_node_ids, node_interact_times], ['id', 'id', 'time'],
                                   wrap_negative=False)
        st = self._c_state()
        if self._ws is None or self._ws_batch < n:
            need = lib.tpn_update_workspace_bytes(st, n)
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=dev)
            self._ws_batch = n
        args = (ptrs[0], ptrs[1], ptrs[2], n, float(next_time), float(np.float32(-lam)), factors,
                self._ws.data_ptr(), self._ws.numel(), self._err.data_ptr())
        return n, float(next_time), args

    def update_prepare(self, src_node_ids: IdArray, dst_node_ids: IdArray, node_interact_times: IdArray,
                       next_time: Optional[float] = None) -> bool:
        """Optional, no reference counterpart: starts the half of the NEXT ``update`` that does not write the state
        (weights, stable sort by target, work lists, lazy mode: the pre-batch snapshot) on a side stream, so that it
        overlaps the calls that still read the pre-batch state — the reference's loop computes the pair-wise features
        of a batch and then updates with the same batch (train_link_prediction.py:370-373,
        evaluate_models_utils.py:182-184).  The following ``update`` call with the same arrays only runs the rest.
        Results are identical with or without it; any other ``update`` call falls back to the whole update.
        Returns False when nothing was started (small batch, or the decay log must be restarted first)."""
        dev = self._require_cuda()
        lib = _lib.load()
        self._pending = None
        n, next_time, args = self._update_args(src_node_ids, dst_node_ids, node_interact_times, next_time)
        if 2 * n <= 4096:
            return False
        if self._prep_stream is None:
            self._prep_stream = torch.cuda.Stream(dev, priority=-1)      # its CTAs go first when SM slots free up
            self._prep_done = torch.cuda.Event()
        cur = torch.cuda.current_stream(dev)
        side = self._prep_stream
        side.wait_stream(cur)                        # fork: the staged ids and every earlier write of the state
        rc = lib.tpn_update_phase(self._c_state(), *args, side.cuda_stream, _lib.UPDATE_PREPARE)
        if rc == _lib.TPN_ERR_LOG_FULL:              # the log restart rewrites the state: not while it is being read
            cur.wait_stream(side)
            return False
        if rc:
            _lib.check(rc, 'tpn_update_phase(prepare)')
        self._prep_done.record(side)
        self._pending = (id(src_node_ids), id(dst_node_ids), id(node_interact_times), n, next_time, args)
        return True

    def update(self, src_node_ids: IdArray, dst_node_ids: IdArray, node_interact_times: IdArray,
               next_time: Optional[float] = None):
        """TPNet.py:67-99.  ``next_time`` is only needed when the arrays are CUDA tensors
        (it is ``node_interact_times[-1]``, which the host needs for the f64 decay factors)."""
        dev = self._require_cuda()
        lib = _lib.load()
        pend, self._pending = self._pending, None
        phase = _lib.UPDATE_WHOLE
        if pend is not None:
            torch.cuda.current_stream(dev).wait_event(self._prep_done)       # join (also frees the workspace)
            if pend[:4] == (id(src_node_ids), id(dst_node_ids), id(node_interact_times), int(len(src_node_ids))) and \
                    (next_time is None or float(next_time) == pend[4]):
                n, next_time, args = pend[3], pend[4], pend[5]
                phase = _lib.UPDATE_APPLY
        if phase == _lib.UPDATE_WHOLE:
            n, next_time, args = self._update_args(src_node_ids, dst_node_ids, node_interact_times, next_time)
        st = self._c_state()
        rc = lib.tpn_update_phase(st, *args, self._stream(), phase)
        if rc == _lib.TPN_ERR_LOG_FULL:
            self._restart_log()
            st = self._c_state()
            rc = lib.tpn_update_phase(st, *args, self._stream(), _lib.UPDATE_WHOLE)
        if rc:
            _lib.check(rc, 'tpn_update')
        h = self._h
        h.epoch = int(h.st.epoch)
        h.launches += 1
        h.now = float(next_time)
        self.now_time.data.fill_(h.now)                                                # TPNet.py:99

    def get_random_projections(self, node_ids: IdArray) -> List[torch.Tensor]:
        """TPNet.py:101-110: list of L+1 tensors [n, dim]."""
        dev = self._require_cuda()
        lib = _lib.load()
        n = int(len(node_ids))
        out = torch.empty(self.num_layer + 1, n, self.dim, dtype=torch.float32, device=dev)
        if n:
            ptrs = self._ids_to_device([node_ids], ['id'])
            rc = lib.tpn_gather(self._c_state(), ptrs[0], n, out.data_ptr(), self._stream())
            if rc:
                _lib.check(rc, 'tpn_gather')
            self._h.launches += 1
        return [out[i] for i in range(self.num_layer + 1)]

    def _out(self, out: Optional[torch.Tensor], shape) -> torch.Tensor:
        """Result buffer of a feature call: a fresh tensor, or the caller's (``out=``: fixed addresses for CUDA graphs)."""
        dev = self._state.device
        if out is None:
            return torch.empty(*shape, dtype=torch.float32, device=dev)
        if tuple(out.shape) != tuple(shape) or out.dtype != torch.float32 or out.device != dev or not out.is_contiguous():
            raise ValueError(f'out must be a contiguous float32 tensor of shape {tuple(shape)} on {dev}')
        return out

    def feature_stream(self) -> torch.cuda.Stream:
        """A second stream for feature calls that are independent of each other (no reference counterpart): the two
        decoder calls of a batch — (src, dst) and (src, neg) — only read the state, so one can run here while the other
        runs on the current stream; the tensor-core head of one call then overlaps the HBM-bound gather of the other.
        The caller forks and joins: ``fs.wait_stream(cur)`` ... ``cur.wait_stream(fs)`` (``pipeline.tpnet_step``)."""
        dev = self._require_cuda()
        if self._feature_stream is None:
            self._feature_stream = torch.cuda.Stream(dev)
        return self._feature_stream

    def pair_wise_gram(self, src_node_ids: IdArray, dst_node_ids: IdArray, out: Optional[torch.Tensor] = None
                       ) -> torch.Tensor:
        """The input of ``self.mlp``: TPNet.py:119-128 (everything before the head)."""
        dev = self._require_cuda()
        lib = _lib.load()
        n = int(len(src_node_ids))
        if len(dst_node_ids) != n:
            raise ValueError('src and dst id arrays must have the same length')
        out = self._out(out, (n, self.pair_wise_feature_dim))
        if n:
            ptrs = self._ids_to_device([src_node_ids, dst_node_ids], ['id', 'id'])
            rc = lib.tpn_pairwise(self._c_state(), ptrs[0], ptrs[1], n, None, 0 if self.not_scale else 1,
                                  out.data_ptr(), self._stream())
            if rc:
                _lib.check(rc, 'tpn_pairwise')
            self._h.launches += 1
        return out

    def _head(self, gram: torch.Tensor, count: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None
              ) -> torch.Tensor:
        """``self.mlp`` on ``[n, F]`` features (TPNet.py:125/:129).  With autograd on (training) it is
        the PyTorch module; under ``torch.no_grad()`` the default-shape head (F = 64) runs as one
        fused fp32 kernel (``tpn_head_forward``).  ``count``: device int32 with the number of valid rows
        (routed calls of the sharded module; rows past it are left zero by the fused kernel)."""
        if torch.is_grad_enabled() or not self.fused_head or gram.shape[0] == 0:
            res = self.mlp(gram)
            return res if out is None else out.copy_(res)
        mlp = self.mlp
        if not (isinstance(mlp, nn.Sequential) and len(mlp) == 3 and isinstance(mlp[0], nn.Linear)
                and isinstance(mlp[1], nn.ReLU) and isinstance(mlp[2], nn.Linear)):
            return self.mlp(gram)
        l1, l2 = mlp[0], mlp[2]
        f, hid = l1.in_features, l1.out_features
        ok = (l2.in_features == hid and l2.out_features == f and gram.shape[1] == f and l1.bias is not None
              and l2.bias is not None and gram.is_contiguous()
              and all(t.dtype == torch.float32 and t.is_cuda and t.is_contiguous() and t.device == gram.device
                      for t in (gram, l1.weight, l1.bias, l2.weight, l2.bias)))
        if ok:
            if out is None:
                out = torch.empty_like(gram) if count is None else torch.zeros_like(gram)
            elif out.shape != gram.shape or out.dtype != torch.float32 or not out.is_contiguous():
                raise ValueError('out must be a contiguous float32 tensor of the shape of the features')
            rc = _lib.load().tpn_head_forward(gram.data_ptr(), gram.shape[0],
                                              None if count is None else count.data_ptr(), f, hid,
                                              l1.weight.data_ptr(),
                                              l1.bias.data_ptr(), l2.weight.data_ptr(), l2.bias.data_ptr(),
                                              out.data_ptr(), self._stream())
            if rc == _lib.TPN_OK:
                self._h.launches += 1
                return out
            if rc != _lib.TPN_ERR_UNSUPPORTED:
                _lib.check(rc, 'tpn_head_forward')
        res = self.mlp(gram)
        return res if out is None else out.copy_(res)

    def get_pair_wise_feature(self, src_node_ids: IdArray, dst_node_ids: IdArray, out: Optional[torch.Tensor] = None
                              ) -> torch.Tensor:
        """TPNet.py:112-129.  Gradients flow to ``self.mlp`` only, as in the reference
        (the projections are ``requires_grad=False``).  ``out`` (no-grad calls): result buffer to write into."""
        return self._head(self.pair_wise_gram(src_node_ids, dst_node_ids), out=out)

    def neighbor_pair_wise_gram(self, neighbor_node_ids: IdArray, src_node_ids: IdArray,
                                dst_node_ids: IdArray) -> torch.Tensor:
        """Input of ``self.mlp`` for the encoder's structured call (TPNet.py:313-324), as
        ``[m, K, 2, F]``: block ``[n, k, 0]`` is the pair ``(nbr[n, k], src[n])`` and block
        ``[n, k, 1]`` the pair ``(nbr[n, k], dst[n])``.  One kernel, no index lists, no re-split."""
        dev = self._require_cuda()
        lib = _lib.load()
        if neighbor_node_ids.ndim != 2:
            raise ValueError('neighbor_node_ids must be [m, num_neighbors]')
        m, k = int(neighbor_node_ids.shape[0]), int(neighbor_node_ids.shape[1])
        if len(src_node_ids) != m or len(dst_node_ids) != m:
            raise ValueError('src and dst id arrays must have one entry per row of neighbor_node_ids')
        f = self.pair_wise_feature_dim
        out = torch.empty(m, k, 2, f, dtype=torch.float32, device=dev)
        if m == 0 or k == 0:
            return out
        flat = neighbor_node_ids.reshape(-1)
        ptrs = self._ids_to_device([flat, src_node_ids, dst_node_ids], ['id', 'id', 'id'])
        rc = lib.tpn_pairwise_neighbors(self._c_state(), ptrs[0], ptrs[1], ptrs[2], m, k, 0 if self.not_scale else 1,
                                        out.data_ptr(), self._stream())
        if rc == _lib.TPN_ERR_UNSUPPORTED:
            # node blocks too wide for the shared-memory staging (use_matrix on a large graph):
            # the generic pair kernel on device-built index lists, as TPNet.py:313-316 builds them
            nb = torch.from_numpy(np.ascontiguousarray(flat)).to(dev) if isinstance(flat, np.ndarray) else flat
            for j, ids in enumerate((src_node_ids, dst_node_ids)):
                e = torch.from_numpy(np.ascontiguousarray(ids)).to(dev) if isinstance(ids, np.ndarray) else ids
                out[:, :, j, :] = self.pair_wise_gram(nb, e.repeat_interleave(k).contiguous()).view(m, k, f)
            return out
        if rc:
            _lib.check(rc, 'tpn_pairwise_neighbors')
        self._h.launches += 1
        return out

    def get_neighbor_pair_wise_feature(self, neighbor_node_ids: IdArray, src_node_ids: IdArray,
                                       dst_node_ids: IdArray, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Drop-in for TPNet.py:313-324: returns ``neighbor_random_features`` ``[m, K, 2F]`` — what
        the reference obtains from ``get_pair_wise_feature(np.tile(nbr.reshape(-1), 2),
        np.concatenate([np.repeat(src, K), np.repeat(dst, K)]))`` followed by the split / ``cat`` /
        ``reshape``.  ``self.mlp`` acts on every F-block on its own, so it is applied to the
        ``[m*K*2, F]`` view (same values, same gradients to the head)."""
        g = self.neighbor_pair_wise_gram(neighbor_node_ids, src_node_ids, dst_node_ids)
        m, k = g.shape[0], g.shape[1]
        f = self.pair_wise_feature_dim
        flat_out = None if out is None else out.view(m * k * 2, f)
        return self._head(g.view(m * k * 2, f), out=flat_out).view(m, k, 2 * f)

    def reset_random_projections(self):
        """TPNet.py:131-139.  (Called once per epoch by train_link_prediction.py:248: also the point where
        an out-of-range id of a device-resident batch — which a kernel can only flag — is raised.)"""
        self._cancel_prepare()
        self._require_cuda()
        if self._h.device_ids_seen:
            self.check_errors()
        lib = _lib.load()
        _lib.check(lib.tpn_clear_walk_layers(self._c_state(), self._stream()), 'tpn_clear_walk_layers')
        self._h.epoch = 0
        self._h.now = self._h.begin
        self.now_time.data.copy_(self.begging_time.data)     # in place: the parameter keeps its storage (CUDA graphs)
        if self.use_matrix:
            return
        if self.p0_seed is not None:
            self.p0_draw += 1
            self._write_counter_p0()
            return
        self._redraw_p0()

    def _redraw_p0(self) -> None:
        """P_0 of a reset drawn with torch's RNG (TPNet.py:139)."""
        std = 1 / math.sqrt(self.dim)
        p0 = self.random_projections[0]
        with torch.no_grad():
            if self.node_num * self.dim * 4 <= (2 << 30):
                # draw into a contiguous [N, d] tensor exactly like nn.init.normal_ on the
                # reference's contiguous parameter (same generator stream), then place it
                p0.copy_(torch.empty(self.node_num, self.dim, dtype=torch.float32, device=p0.device)
                         .normal_(mean=0, std=std))
            else:
                p0.normal_(mean=0, std=std)

    def _p0_rows(self) -> Tuple[int, int, int]:
        """(rows, first node, node step) of the P_0 rows this module owns: all of them, node j at row j."""
        return self.node_num, 0, 1

    def _write_counter_p0(self) -> None:
        """Draw ``p0_draw`` of the counter-based generator into the owned rows of P_0 (tpn_init_projection)."""
        self._require_cuda()
        rows, first, step = self._p0_rows()
        # a layout-only view: the kernel reads no stamps, and the module's cached C state is left alone
        st = TpnState(data=self._state.data_ptr(), num_nodes=self.node_num, num_layer=self.num_layer, dim=self.dim,
                      row_stride=self.row_stride, node_stride=self.node_stride)
        rc = _lib.load().tpn_init_projection(ctypes.byref(st), rows, first, step, self.p0_seed, self.p0_draw,
                                             self._stream())
        _lib.check(rc, 'tpn_init_projection')

    def backup_random_projections(self) -> Tuple[torch.Tensor, List[torch.Tensor]]:
        """TPNet.py:141-147: (now_time, [P_1..P_L]) — P_0 is not part of the backup."""
        self.materialize()
        return self.now_time.clone(), [self.random_projections[i].clone() for i in range(1, self.num_layer + 1)]

    def reload_random_projections(self, random_projections):
        """TPNet.py:149-157."""
        self._cancel_prepare()
        now_time, layers = random_projections
        with torch.no_grad():
            self.now_time.data.copy_(now_time.to(self.now_time.device))       # in place: same storage (CUDA graphs)
            for i in range(1, self.num_layer + 1):
                self.random_projections[i].copy_(layers[i - 1])
        self._after_external_write()

    def _warm_buffers(self, batch: int) -> None:
        """Everything a later call would allocate lazily, allocated now (before a CUDA-graph capture): the C state
        mirror, the error flag, the update workspace for `batch` edges; one read-only feature call initialises the
        kernels' per-device attributes."""
        dev = self._require_cuda()
        lib = _lib.load()
        st = self._c_state()
        need = lib.tpn_update_workspace_bytes(st, max(int(batch), 1))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=dev)
        self._ws_batch = max(self._ws_batch, int(batch))
        if self._prep_stream is None:
            self._prep_stream = torch.cuda.Stream(dev, priority=-1)      # its CTAs go first when SM slots free up
            self._prep_done = torch.cuda.Event()
        self.feature_stream()
        ids = torch.zeros(max(int(batch), 1), dtype=torch.int64, device=dev)
        with torch.no_grad():
            self.get_pair_wise_feature(ids, ids)

    # ------------------------------------------------------------------ lazy-decay maintenance
    def materialize(self) -> None:
        """Bring every row current (no-op in eager mode or off-GPU)."""
        self._cancel_prepare()
        if self._state.device.type != 'cuda' or not self.lazy or self._stamps is None or self._h.epoch == 0:
            return
        lib = _lib.load()
        _lib.check(lib.tpn_materialize(self._c_state(), self._stream()), 'tpn_materialize')
        self._h.launches += 1

    def _restart_log(self) -> None:
        self._cancel_prepare()
        lib = _lib.load()
        self.materialize()
        _lib.check(lib.tpn_reset_epoch(self._c_state(), self._stream()), 'tpn_reset_epoch')
        self._h.epoch = 0

    def check_errors(self) -> None:
        """Synchronises and raises IndexError if a device-resident id was out of range in any call since the
        last check (update drops such edges; pair-wise / gather calls clamp the access).  Host (numpy) ids are
        validated before anything is launched and raise at once, like the reference."""
        self._h.device_ids_seen = False
        code = int(self._err.item()) if self._err is not None else 0
        if code != 0:
            self._err.zero_()
            if code == 4:
                raise RuntimeError('a routed call of the sharded state owned more items than it was sized for '
                                   '(raise route_cap_factor); the excess was dropped')
            if code == 8:
                raise RuntimeError('tpn_update: the grid barrier of the fused sort front end timed out (its CTAs were '
                                   'not co-resident); the update of that call is invalid')
            if code == 2:
                raise RuntimeError('tpn_update_messages: a local source row was not a target of the same call '
                                   '(lazy decay needs both directions of every edge in the message list)')
            raise IndexError(f'node id out of range for node_num {self.node_num} in a device-resident batch')
