"""GPU version of the reference's negative edge sampler (DyGLib's ``NegativeEdgeSampler``, the reference's
utils/utils.py:315-505) with its three strategies, ``random``, ``historical`` and ``inductive``.

The constructor, ``sample`` and ``reset_random_state`` take the reference's arguments.  The tables are built once on
the device (``tpn_neg_sampler_build``): the edges sorted by time, and the distinct edges sorted by their first time,
so that ``W(earliest, s)`` is a prefix and no set of ``unique_src x unique_dst`` is ever built.  A call draws from the
same sets as the reference, with the same sizes and the same ordering rule (random fill first, then all of the
historical edges), but from a counter-based generator keyed by ``(seed, call index)`` instead of numpy's MT19937:
the same distribution, not the same draws (DESIGN.md §3).  The draws do not depend on the grid, the device or the
world size.

A call never reads a count back to the host, so with CUDA-tensor batch arguments and 0-d CUDA-tensor times (for
example ``t[0]`` and ``t[-1]`` of a resident batch) it can be captured in a CUDA graph.  The call index advances on
the host per ``sample`` call and is baked into a captured graph: replaying graphs captured after a
``reset_random_state()`` in capture order reproduces the eager calls.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple, Union

import numpy as np
import torch

from . import _lib

ArrayOrTensor = Union[np.ndarray, torch.Tensor]
STRATEGIES = {'random': 0, 'historical': 1, 'inductive': 2}
NEG_ERR_EMPTY = 1
MAX_EDGES = 0x7fffffff - 4096


def _ids(a, name: str) -> np.ndarray:
    a = np.asarray(a)
    if a.ndim != 1:
        raise ValueError(f'{name} must be one-dimensional')
    if a.dtype.kind not in 'iu':
        if a.size and not np.array_equal(a, np.round(a)):
            raise ValueError(f'{name} must hold integer node ids')
    a = a.astype(np.int64)
    if a.size and (a.min() < 0 or a.max() > 0xffffffff):
        raise IndexError(f'{name}: node ids must lie in [0, 2**32)')
    return a


class NegativeEdgeSampler:
    def __init__(self, src_node_ids, dst_node_ids, interact_times=None, last_observed_time=None,
                 negative_sample_strategy: str = 'random', seed: Optional[int] = None,
                 device: Union[str, torch.device] = 'cuda'):
        if negative_sample_strategy not in STRATEGIES:
            raise ValueError(f'negative_sample_strategy must be one of {tuple(STRATEGIES)}')
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise RuntimeError('tpnet_b200.NegativeEdgeSampler samples on CUDA only (no CPU fallback)')
        src = _ids(src_node_ids, 'src_node_ids')
        dst = _ids(dst_node_ids, 'dst_node_ids')
        if len(src) != len(dst):
            raise ValueError('src_node_ids and dst_node_ids must have the same length')
        if len(src) < 1 or len(src) > MAX_EDGES:
            raise ValueError(f'the sampler needs 1 .. {MAX_EDGES} edges')
        timed = negative_sample_strategy != 'random'
        t = None
        if interact_times is not None:
            t = np.asarray(interact_times, dtype=np.float64).reshape(-1)
            if len(t) != len(src):
                raise ValueError('interact_times must have one time per edge')
            if np.isnan(t).any():
                raise ValueError('interact_times must not be NaN')
        elif timed:
            raise ValueError(f'the {negative_sample_strategy!r} strategy needs interact_times')
        if negative_sample_strategy == 'inductive' and last_observed_time is None:
            raise ValueError("the 'inductive' strategy needs last_observed_time")
        if seed is not None and (int(seed) != seed or seed < 0):
            raise ValueError('seed must be a non-negative integer or None')

        if dev.index is None:
            dev = torch.device('cuda', torch.cuda.current_device())
        # attributes the reference's callers read
        self.negative_sample_strategy = negative_sample_strategy
        self.seed = seed
        self.src_node_ids, self.dst_node_ids, self.interact_times = src_node_ids, dst_node_ids, interact_times
        self.earliest_time = None if t is None else float(t.min())
        self.last_observed_time = last_observed_time
        self.device = dev
        # seed None: one key from numpy's global generator, so np.random.seed still governs the draws
        self.key = int(seed) & 0xffffffffffffffff if seed is not None else \
            int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
        self._call = 0

        E = len(src)
        id_bits = max(1, int(max(src.max(), dst.max())).bit_length())
        uniq_cap = min(E, 1 << id_bits)
        u32, f64 = torch.int32, torch.float64

        def buf(n, dtype):
            return torch.empty(n, dtype=dtype, device=dev)

        self._tables = {'uniq_src': buf(uniq_cap, u32), 'uniq_dst': buf(uniq_cap, u32),
                        'counts': torch.zeros(4, dtype=torch.int32, device=dev)}
        if timed:
            for name, dtype in (('t_src', u32), ('t_dst', u32), ('t_time', f64), ('t_fpos', u32), ('f_src', u32),
                                ('f_dst', u32), ('f_time', f64), ('mark', u32)):
                self._tables[name] = buf(E, dtype)
        c = _lib.TpnNegSampler()
        c.num_edges, c.id_bits, c.timed, c.seed = E, id_bits, int(timed), self.key
        c.last_observed_time = float(last_observed_time) if last_observed_time is not None else -np.inf
        for name, tensor in self._tables.items():
            setattr(c, name, tensor.data_ptr())
        self._c = c
        lib = _lib.load()
        self._ws = torch.empty(int(lib.tpn_neg_sampler_workspace_bytes(E, 0, 0)), dtype=torch.uint8, device=dev)
        src_d = torch.from_numpy(src).to(dev)
        dst_d = torch.from_numpy(dst).to(dev)
        t_d = torch.from_numpy(t).to(dev) if timed else None
        with torch.cuda.device(dev):
            rc = lib.tpn_neg_sampler_build(ctypes.byref(c), src_d.data_ptr(), dst_d.data_ptr(),
                                           t_d.data_ptr() if timed else None, self._ws.data_ptr(), self._ws.numel(),
                                           self._stream())
        _lib.check(rc, 'tpn_neg_sampler_build')
        counts = self._tables['counts'].cpu().numpy()          # one synchronisation, at construction
        self.num_unique_edges = int(counts[0]) if timed else None
        self.unique_src_node_ids = self._tables['uniq_src'][:int(counts[1])].cpu().numpy().view(np.uint32).astype(np.int64)
        self.unique_dst_node_ids = self._tables['uniq_dst'][:int(counts[2])].cpu().numpy().view(np.uint32).astype(np.int64)
        del src_d, dst_d, t_d
        self._ws = torch.empty(0, dtype=torch.uint8, device=dev)   # the build's scratch is not kept

    def _stream(self) -> int:
        return torch._C._cuda_getCurrentRawStream(self.device.index)

    def reset_random_state(self) -> None:
        """The next call draws what the first call after construction drew (utils/utils.py's reset_random_state)."""
        self._call = 0

    @property
    def call_index(self) -> int:
        return self._call

    def _batch(self, a: ArrayOrTensor, name: str) -> torch.Tensor:
        if isinstance(a, torch.Tensor):
            if a.device != self.device:
                raise ValueError(f'{name} is on {a.device}, the sampler on {self.device}')
            return a.reshape(-1).to(torch.int64).contiguous()
        a = np.asarray(a)
        if a.ndim != 1:
            raise ValueError(f'{name} must be one-dimensional')
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(self.device)

    def _time(self, x, name: str):
        """(host value, device pointer or None) of a batch time."""
        if isinstance(x, torch.Tensor):
            if x.numel() != 1 or x.device != self.device or x.dtype != torch.float64:
                raise ValueError(f'{name} must be a float or a one-element float64 tensor on {self.device}')
            return 0.0, x
        v = float(x)
        if np.isnan(v):
            raise ValueError(f'{name} must not be NaN')
        return v, None

    def sample(self, size: int, batch_src_node_ids: ArrayOrTensor = None, batch_dst_node_ids: ArrayOrTensor = None,
               current_batch_start_time=0.0, current_batch_end_time=0.0, as_tensors: bool = False
               ) -> Tuple[ArrayOrTensor, ArrayOrTensor]:
        """(negative src ids, negative dst ids), int64 numpy arrays (CUDA tensors with ``as_tensors=True``)."""
        if int(size) != size or size < 0 or size > MAX_EDGES:
            raise ValueError(f'size must be an integer in [0, {MAX_EDGES}]')
        size = int(size)
        strategy = STRATEGIES[self.negative_sample_strategy]
        out_src = torch.empty(size, dtype=torch.int64, device=self.device)
        out_dst = torch.empty(size, dtype=torch.int64, device=self.device)
        bs = bd = s_dev = e_dev = None
        s = e = 0.0
        batch = 0
        if strategy:
            if self.seed is None:
                raise ValueError('Random state is not initialized! The historical and inductive strategies need a seed')
            if batch_src_node_ids is None or batch_dst_node_ids is None:
                raise ValueError('the historical and inductive strategies need the batch source and destination ids')
            bs = self._batch(batch_src_node_ids, 'batch_src_node_ids')
            bd = self._batch(batch_dst_node_ids, 'batch_dst_node_ids')
            if bs.numel() != bd.numel():
                raise ValueError('batch_src_node_ids and batch_dst_node_ids must have the same length')
            if bs.numel() > MAX_EDGES:
                raise ValueError(f'a batch holds at most {MAX_EDGES} edges')
            batch = bs.numel()
            s, s_dev = self._time(current_batch_start_time, 'current_batch_start_time')
            e, e_dev = self._time(current_batch_end_time, 'current_batch_end_time')
            lib = _lib.load()
            need = int(lib.tpn_neg_sampler_workspace_bytes(0, size, batch))
            if self._ws.numel() < need:
                if torch.cuda.is_current_stream_capturing():
                    raise RuntimeError('NegativeEdgeSampler: the workspace must grow, which is not allowed inside a '
                                       'CUDA-graph capture; make one eager call of this size first')
                self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        call = self._call
        self._call += 1
        if size:
            lib = _lib.load()
            with torch.cuda.device(self.device):
                rc = lib.tpn_neg_sampler_sample(
                    ctypes.byref(self._c), strategy, call, size,
                    bs.data_ptr() if bs is not None else None, bd.data_ptr() if bd is not None else None, batch,
                    s, e, s_dev.data_ptr() if s_dev is not None else None,
                    e_dev.data_ptr() if e_dev is not None else None, out_src.data_ptr(), out_dst.data_ptr(),
                    self._ws.data_ptr() if self._ws.numel() else None, self._ws.numel(), self._stream())
            _lib.check(rc, 'tpn_neg_sampler_sample')
        if as_tensors:
            return out_src, out_dst
        src_np, dst_np = out_src.cpu().numpy(), out_dst.cpu().numpy()
        self.check_errors()
        return src_np, dst_np

    def check_errors(self) -> None:
        """Raises (and clears) a flag a call left on the device: a fill found every pair of unique_src x unique_dst in
        the batch, where the reference's assert fails (its outputs were written as -1)."""
        counts = self._tables['counts']
        err = int(counts[3].item())
        if err:
            counts[3].zero_()
            raise ValueError('NegativeEdgeSampler: every pair of unique_src_node_ids x unique_dst_node_ids is an edge '
                             'of the batch, so no random negative can be drawn (the reference asserts here)')
