"""ctypes binding of the C ABI declared in include/tpnet_b200.h.

There is no CPU fallback: if the shared library is missing, or it cannot be
loaded, every entry point raises.  The library is built in-tree by
``tpnet_b200.build`` (nvcc, sm_100a) and lives at tpnet_b200/_C/libtpnet_b200.so.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p
from typing import Optional

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, '_C', 'libtpnet_b200.so')

TPN_OK = 0
TPN_ERR_LOG_FULL = -3
TPN_ERR_UNSUPPORTED = -5
TPN_ERR_INDEX = -6
STAGE_RAW, STAGE_ID_WRAP, STAGE_ID = 0, 1, 2
TPN_MAX_LAYERS = 4
UPDATE_WHOLE, UPDATE_PREPARE, UPDATE_APPLY = 0, 1, 2
ABI_VERSION = 16

#: every symbol include/tpnet_b200.h declares (tests assert the .so exports all of them)
EXPORTED_SYMBOLS = (
    'tpn_version', 'tpn_error_string', 'tpn_last_cuda_error', 'tpn_device_info',
    'tpn_update_workspace_bytes', 'tpn_update', 'tpn_update_phase', 'tpn_pairwise', 'tpn_gather',
    'tpn_materialize', 'tpn_reset_epoch', 'tpn_clear_walk_layers',
    'tpn_stager_create', 'tpn_stager_destroy', 'tpn_stage',
    'tpn_update_messages', 'tpn_gather_blocks', 'tpn_set_debug_flags', 'tpn_pairwise_neighbors', 'tpn_head_forward',
    'tpn_planner_create', 'tpn_planner_destroy', 'tpn_plan', 'tpn_sampler_recent',
    'tpn_route_workspace_bytes', 'tpn_route_update', 'tpn_route_pairs', 'tpn_route_nodes', 'tpn_pull_rows',
    'tpn_peer_barrier', 'tpn_shard_new_generation', 'tpn_peer_alloc', 'tpn_peer_free', 'tpn_ipc_export', 'tpn_ipc_open',
    'tpn_ipc_close', 'tpn_stream_sampler_workspace_bytes', 'tpn_stream_sampler_reset', 'tpn_stream_sampler_push',
    'tpn_stream_sampler_query', 'tpn_stream_shard_reset', 'tpn_stream_shard_push', 'tpn_stream_shard_pull',
    'tpn_stream_shard_query', 'tpn_init_projection', 'tpn_neg_sampler_workspace_bytes', 'tpn_neg_sampler_build',
    'tpn_neg_sampler_sample',
)

SHARD_CTR_NEED, SHARD_CTR_PREV, SHARD_CTR_ERROR, SHARD_COUNTERS = 0, 1, 2, 8
STREAM_ERR_INDEX, STREAM_ERR_ORDER, STREAM_ERR_PAST = 1, 2, 4
#: per rank, the tables of tpn_stream_shard_t.peer_lists, in this order
STREAM_PEER_TABLES = ('all_nbr', 'all_eid', 'all_t', 'old_nbr', 'old_eid', 'old_t', 'all_cnt', 'old_cnt', 'newest')


class TpnState(ctypes.Structure):
    """Mirror of ``tpn_state_t`` (include/tpnet_b200.h)."""
    _fields_ = [
        ('data', c_void_p),
        ('num_nodes', c_int64),
        ('num_layer', c_int32),
        ('dim', c_int32),
        ('row_stride', c_int64),
        ('node_stride', c_int64),
        ('stamps', c_void_p),
        ('decay_log', c_void_p),
        ('log_capacity', c_int64),
        ('epoch', c_int64),
        ('cum_floor', c_double),
        ('err_flag', c_void_p),
        ('giant_chunk', c_int32),
        ('reserved0', c_int32),
    ]


class TpnShard(ctypes.Structure):
    """Mirror of ``tpn_shard_t`` (include/tpnet_b200.h)."""
    _fields_ = [
        ('world', c_int32),
        ('rank', c_int32),
        ('global_nodes', c_int64),
        ('num_local_rows', c_int64),
        ('ext_rows', c_int64),
        ('peer_data', c_void_p),
        ('peer_stamps', c_void_p),
        ('peer_flags', c_void_p),
        ('mark', c_void_p),
        ('counters', c_void_p),
        ('need_nodes', c_void_p),
        ('barrier_seq', c_void_p),
    ]


class TpnStreamSampler(ctypes.Structure):
    """Mirror of ``tpn_stream_sampler_t`` (include/tpnet_b200.h)."""
    _fields_ = [
        ('num_nodes', c_int64),
        ('capacity', c_int32),
        ('reserved0', c_int32),
        ('max_batch', c_int64),
        ('all_nbr', c_void_p),
        ('all_eid', c_void_p),
        ('all_t', c_void_p),
        ('old_nbr', c_void_p),
        ('old_eid', c_void_p),
        ('old_t', c_void_p),
        ('all_cnt', c_void_p),
        ('old_cnt', c_void_p),
        ('newest', c_void_p),
        ('pend_node', c_void_p),
        ('pend_nbr', c_void_p),
        ('pend_eid', c_void_p),
        ('pend_t', c_void_p),
        ('pend_count', c_void_p),
        ('last_time', c_void_p),
        ('err_flag', c_void_p),
    ]


class TpnStreamShard(ctypes.Structure):
    """Mirror of ``tpn_stream_shard_t`` (include/tpnet_b200.h)."""
    _fields_ = [
        ('local', TpnStreamSampler),
        ('shard', TpnShard),
        ('peer_lists', c_void_p),
    ]


class TpnNegSampler(ctypes.Structure):
    """Mirror of ``tpn_neg_sampler_t`` (include/tpnet_b200.h)."""
    _fields_ = [
        ('num_edges', c_int64),
        ('id_bits', c_int32),
        ('timed', c_int32),
        ('seed', c_uint64),
        ('last_observed_time', c_double),
        ('t_src', c_void_p),
        ('t_dst', c_void_p),
        ('t_time', c_void_p),
        ('t_fpos', c_void_p),
        ('f_src', c_void_p),
        ('f_dst', c_void_p),
        ('f_time', c_void_p),
        ('mark', c_void_p),
        ('uniq_src', c_void_p),
        ('uniq_dst', c_void_p),
        ('counts', c_void_p),
    ]


class TpnError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ''):
        self.code = code
        super().__init__(f'{where} failed: {detail} (code {code})')


_lib: Optional[ctypes.CDLL] = None


def _declare(lib: ctypes.CDLL) -> None:
    lib.tpn_version.restype = c_int
    lib.tpn_version.argtypes = []
    lib.tpn_error_string.restype = c_char_p
    lib.tpn_error_string.argtypes = [c_int]
    lib.tpn_last_cuda_error.restype = c_char_p
    lib.tpn_last_cuda_error.argtypes = []
    lib.tpn_device_info.restype = c_int
    lib.tpn_device_info.argtypes = [POINTER(c_int), POINTER(c_int), POINTER(c_int)]
    lib.tpn_update_workspace_bytes.restype = c_size_t
    lib.tpn_update_workspace_bytes.argtypes = [POINTER(TpnState), c_int64]
    lib.tpn_update.restype = c_int
    lib.tpn_update.argtypes = [POINTER(TpnState), c_void_p, c_void_p, c_void_p, c_int64, c_double, c_float,
                               POINTER(c_float), c_void_p, c_size_t, c_void_p, c_void_p]
    lib.tpn_update_phase.restype = c_int
    lib.tpn_update_phase.argtypes = [POINTER(TpnState), c_void_p, c_void_p, c_void_p, c_int64, c_double, c_float,
                                     POINTER(c_float), c_void_p, c_size_t, c_void_p, c_void_p, c_int]
    lib.tpn_update_messages.restype = c_int
    lib.tpn_update_messages.argtypes = [POINTER(TpnState), c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                        c_double, c_float, POINTER(c_float), c_void_p, c_size_t, c_void_p, c_void_p]
    lib.tpn_set_debug_flags.restype = c_int
    lib.tpn_set_debug_flags.argtypes = [c_int]
    lib.tpn_gather_blocks.restype = c_int
    lib.tpn_gather_blocks.argtypes = [POINTER(TpnState), c_void_p, c_int64, c_void_p, c_void_p]
    lib.tpn_pairwise.restype = c_int
    lib.tpn_pairwise.argtypes = [POINTER(TpnState), c_void_p, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p]
    lib.tpn_pairwise_neighbors.restype = c_int
    lib.tpn_pairwise_neighbors.argtypes = [POINTER(TpnState), c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int,
                                           c_void_p, c_void_p]
    lib.tpn_head_forward.restype = c_int
    lib.tpn_head_forward.argtypes = [c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p]
    lib.tpn_gather.restype = c_int
    lib.tpn_gather.argtypes = [POINTER(TpnState), c_void_p, c_int64, c_void_p, c_void_p]
    for name in ('tpn_materialize', 'tpn_reset_epoch', 'tpn_clear_walk_layers'):
        fn = getattr(lib, name)
        fn.restype = c_int
        fn.argtypes = [POINTER(TpnState), c_void_p]
    lib.tpn_init_projection.restype = c_int
    lib.tpn_init_projection.argtypes = [POINTER(TpnState), c_int64, c_int64, c_int64, c_uint64, c_uint64, c_void_p]
    lib.tpn_neg_sampler_workspace_bytes.restype = c_size_t
    lib.tpn_neg_sampler_workspace_bytes.argtypes = [c_int64, c_int64, c_int64]
    lib.tpn_neg_sampler_build.restype = c_int
    lib.tpn_neg_sampler_build.argtypes = [POINTER(TpnNegSampler), c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                          c_void_p]
    lib.tpn_neg_sampler_sample.restype = c_int
    lib.tpn_neg_sampler_sample.argtypes = [POINTER(TpnNegSampler), c_int, c_uint64, c_int64, c_void_p, c_void_p, c_int64,
                                           c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_size_t, c_void_p]
    lib.tpn_sampler_recent.restype = c_int
    lib.tpn_sampler_recent.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                       c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.tpn_stream_sampler_workspace_bytes.restype = c_size_t
    lib.tpn_stream_sampler_workspace_bytes.argtypes = [c_int64]
    lib.tpn_stream_sampler_reset.restype = c_int
    lib.tpn_stream_sampler_reset.argtypes = [POINTER(TpnStreamSampler), c_void_p]
    lib.tpn_stream_sampler_push.restype = c_int
    lib.tpn_stream_sampler_push.argtypes = [POINTER(TpnStreamSampler), c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                            c_void_p, c_size_t, c_void_p]
    lib.tpn_stream_sampler_query.restype = c_int
    lib.tpn_stream_sampler_query.argtypes = [POINTER(TpnStreamSampler), c_void_p, c_void_p, c_int64, c_int, c_void_p,
                                             c_void_p, c_void_p, c_void_p]
    for name in ('tpn_stream_shard_reset', 'tpn_stream_shard_pull'):
        fn = getattr(lib, name)
        fn.restype = c_int
        fn.argtypes = [POINTER(TpnStreamShard), c_void_p]
    lib.tpn_stream_shard_push.restype = c_int
    lib.tpn_stream_shard_push.argtypes = [POINTER(TpnStreamShard), c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                          c_void_p, c_size_t, c_void_p]
    lib.tpn_stream_shard_query.restype = c_int
    lib.tpn_stream_shard_query.argtypes = [POINTER(TpnStreamShard), c_void_p, c_void_p, c_void_p, c_int64, c_int,
                                           c_void_p, c_void_p, c_void_p, c_void_p]
    lib.tpn_planner_create.restype = c_int
    lib.tpn_planner_create.argtypes = [POINTER(c_void_p), c_int64, c_int, c_int]
    lib.tpn_planner_destroy.restype = None
    lib.tpn_planner_destroy.argtypes = [c_void_p]
    lib.tpn_plan.restype = c_int
    lib.tpn_plan.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                             POINTER(c_int64), c_void_p, POINTER(c_int64), c_void_p, c_void_p]
    lib.tpn_route_workspace_bytes.restype = c_size_t
    lib.tpn_route_workspace_bytes.argtypes = [c_int64]
    lib.tpn_route_update.restype = c_int
    lib.tpn_route_update.argtypes = [POINTER(TpnShard), c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.tpn_route_pairs.restype = c_int
    lib.tpn_route_pairs.argtypes = [POINTER(TpnShard), c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_size_t, c_void_p]
    lib.tpn_route_nodes.restype = c_int
    lib.tpn_route_nodes.argtypes = [POINTER(TpnShard), c_void_p, c_int64, c_void_p, c_void_p]
    lib.tpn_pull_rows.restype = c_int
    lib.tpn_pull_rows.argtypes = [POINTER(TpnState), POINTER(TpnShard), c_void_p]
    lib.tpn_peer_barrier.restype = c_int
    lib.tpn_peer_barrier.argtypes = [POINTER(TpnShard), c_void_p]
    lib.tpn_shard_new_generation.restype = c_int
    lib.tpn_shard_new_generation.argtypes = [POINTER(TpnShard), c_void_p]
    lib.tpn_peer_alloc.restype = c_int
    lib.tpn_peer_alloc.argtypes = [POINTER(c_void_p), c_size_t]
    lib.tpn_peer_free.restype = c_int
    lib.tpn_peer_free.argtypes = [c_void_p]
    lib.tpn_ipc_export.restype = c_int
    lib.tpn_ipc_export.argtypes = [c_void_p, c_void_p]
    lib.tpn_ipc_open.restype = c_int
    lib.tpn_ipc_open.argtypes = [c_void_p, POINTER(c_void_p)]
    lib.tpn_ipc_close.restype = c_int
    lib.tpn_ipc_close.argtypes = [c_void_p]
    lib.tpn_stager_create.restype = c_int
    lib.tpn_stager_create.argtypes = [POINTER(c_void_p), c_size_t, c_int]
    lib.tpn_stager_destroy.restype = None
    lib.tpn_stager_destroy.argtypes = [c_void_p]
    lib.tpn_stage.restype = c_int
    lib.tpn_stage.argtypes = [c_void_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int), c_int, c_int64,
                              POINTER(c_void_p), c_void_p]


def load() -> ctypes.CDLL:
    """Load the CUDA library or raise — never falls back to anything else."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'tpnet_b200 CUDA library not found at {LIB_PATH}. Build it with '
            f'`python -m tpnet_b200.build` (needs nvcc); there is no CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    missing = [s for s in EXPORTED_SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise RuntimeError(f'{LIB_PATH} does not export {missing}; rebuild with `python -m tpnet_b200.build --force`')
    _declare(lib)
    if lib.tpn_version() != ABI_VERSION:
        raise RuntimeError(f'{LIB_PATH} has ABI version {lib.tpn_version()}, expected {ABI_VERSION}; rebuild')
    if os.environ.get('TPN_DEBUG_FLAGS'):           # A/B measurements only (include/tpnet_b200.h, TPN_DEBUG_*)
        lib.tpn_set_debug_flags(int(os.environ['TPN_DEBUG_FLAGS']))
    _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code == TPN_OK:
        return
    if code == TPN_ERR_INDEX:
        raise IndexError(f'{where}: node id out of range')
    lib = load()
    detail = lib.tpn_error_string(code).decode()
    cuda = lib.tpn_last_cuda_error().decode()
    if cuda:
        detail += f' [{cuda}]'
    raise TpnError(code, where, detail)
