"""Packed checkpoints of the walk-projection state (SURVEY.md 8(f) N4).

The reference checkpoints ``model.state_dict()`` (``utils/EarlyStopping.py:64-87``).  Its
``RandomProjectionModule`` is registered under three parents (the backbone, the link predictor and
the model itself), so the L+1 ``[N, d]`` matrices appear three times in that dict — 3 x 33.6 GB for
the 10M-node graph — and a node-sharded state has no single ``state_dict`` at all.  This format
stores the state ONCE, one file per rank, and can be read back into any number of ranks:

    <dir>/<tag>.rank<r>-of-<G>.pt     torch.save of the header
        {'format', 'world', 'rank', 'global_node_num', 'dim', 'num_layer', 'now_time', 'begging_time', 'rows',
         'mlp': state_dict of the trainable head,
         'p0': {'seed', 'draw'} of a module with a counter-based P_0 (``p0_seed``), else None; absent in older files}
    <dir>/<tag>.rank<r>-of-<G>.state  raw little-endian float32 [rows, L+1, dim], C order
                                      (row j of rank r = node j*G + r; pending lazy decay applied)

The state file is written and read in CHUNKS of rows through a bounded host buffer (``chunk_bytes``, default
64 MiB): a 34.6 GB GPU-resident state is saved and restored without ever holding a whole shard in host memory.
(v1 files, which kept the state inside the .pt header, still load.)

``state_dict()`` / ``load_state_dict()`` of the module keep the reference's keys and remain the way
the unmodified reference scripts checkpoint small graphs; this is the path for states that do not
fit one host copy three times, or are sharded.

The streaming neighbour sampler (``StreamingRecentSampler`` / ``ShardedStreamingSampler``) is saved the same way,
so a stream job resumes where it stopped, at any world size (``save_sampler`` / ``load_sampler``):

    <dir>/<tag>.rank<r>-of-<G>.pt     torch.save of the header
        {'format', 'world', 'rank', 'num_nodes', 'capacity', 'rows', 'last_time', 'pend_count',
         'pend_node', 'pend_nbr', 'pend_eid', 'pend_t': the pending batch as sorted on the device}
    <dir>/<tag>.rank<r>-of-<G>.lists  raw little-endian row records, 48 * capacity + 16 bytes each
                                      (row j of rank r = node j*G + r; ``sampler_record_dtype``)
"""
from __future__ import annotations

import glob
import os
import re
from typing import Callable, Dict, Iterator, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .peer import rows_on_rank

FORMAT_V1 = 'tpnet_b200.shard.v1'
FORMAT = 'tpnet_b200.shard.v2'
SAMPLER_FORMAT = 'tpnet_b200.sampler.v1'
DEFAULT_CHUNK_BYTES = 64 << 20


def _shard_info(obj, num_nodes: int) -> Tuple[int, int, int]:
    """(world, rank, rows this rank owns) of a plain or sharded state or sampler over ``num_nodes`` nodes; cache rows
    are not owned."""
    return int(getattr(obj, 'world', 1)), int(getattr(obj, 'rank', 0)), int(getattr(obj, 'n_local', num_nodes))


def shard_path(directory: str, tag: str, rank: int, world: int) -> str:
    return os.path.join(directory, f'{tag}.rank{rank}-of-{world}.pt')


def pack_shard(state_rows: torch.Tensor, world: int, rank: int, global_node_num: int, now_time: float,
               begging_time: float, head: Dict[str, torch.Tensor]) -> dict:
    """Payload of one rank.  ``state_rows``: float32 [rows, L+1, dim] of the nodes rank, rank+world, ..."""
    rows_expected = rows_on_rank(global_node_num, world, rank)
    if state_rows.dim() != 3 or state_rows.shape[0] != rows_expected or state_rows.dtype != torch.float32:
        raise ValueError(f'rank {rank} of {world} owns {rows_expected} of {global_node_num} nodes; got state '
                         f'{tuple(state_rows.shape)} {state_rows.dtype}')
    return {'format': FORMAT_V1, 'world': int(world), 'rank': int(rank), 'global_node_num': int(global_node_num),
            'dim': int(state_rows.shape[2]), 'num_layer': int(state_rows.shape[1]) - 1, 'now_time': float(now_time),
            'begging_time': float(begging_time), 'state': state_rows.detach().to('cpu').contiguous(),
            'mlp': {k: v.detach().to('cpu') for k, v in head.items()}}


def scatter_rows(dst: Union[torch.Tensor, Sequence[torch.Tensor]], world: int, rank: int, saved_world: int,
                 saved_rank: int, src: Union[torch.Tensor, Sequence[torch.Tensor]], first_row: int = 0) -> int:
    """Re-sharding by node id.  ``src``: rows [first_row, first_row + n) of the shard saved by ``saved_rank`` of
    ``saved_world`` (its row j is node j * saved_world + saved_rank).  Copies those that rank ``rank`` of ``world``
    owns into ``dst`` (local row u // world of node u).  Returns the number of rows copied.
    ``dst`` / ``src`` are one tensor each, or sequences of tensors paired in order (the sampler's tables), indexed by
    row along dim 0.  A ``dst`` row wider than its ``src`` row in the last dimension (the state's padded row stride)
    receives the leading columns."""
    pairs = list(zip(dst, src)) if isinstance(dst, (list, tuple)) else [(dst, src)]
    n = int(pairs[0][1].shape[0])
    ids = saved_rank + saved_world * torch.arange(first_row, first_row + n, dtype=torch.int64)
    sel = torch.nonzero((ids % world) == rank).squeeze(1)
    if len(sel):
        local = torch.div(ids[sel], world, rounding_mode='floor')
        for d, s in pairs:
            if d.shape[1:] != s.shape[1:]:
                d = d[..., :s.shape[-1]]
            d[local.to(d.device)] = s[sel.to(s.device)].to(d.device)
    return int(len(sel))


def scatter_shard(dst_rows: torch.Tensor, world: int, rank: int, payload: dict) -> int:
    """v1 payload (state inside the header): see ``scatter_rows``."""
    return scatter_rows(dst_rows, world, rank, int(payload['world']), int(payload['rank']), payload['state'])


def state_path(header_path: str) -> str:
    return header_path[:-3] + '.state'


def _write_rows(path: str, rows: int, per: int, row_shape: Tuple[int, ...], dtype: torch.dtype, on_gpu: bool,
                fill: Callable[[int, int, torch.Tensor], None]) -> None:
    """Writes ``rows`` rows of ``row_shape`` to ``path`` in chunks of ``per`` rows through two (pinned) host buffers.
    ``fill(lo, hi, buf)`` enqueues the copy of rows [lo, hi) into ``buf``; the device -> host copy of chunk k+1 runs
    while chunk k is written, and host memory stays at two chunks whatever the table size."""
    bufs = [torch.empty((min(per, max(rows, 1)),) + tuple(row_shape), dtype=dtype, pin_memory=on_gpu)
            for _ in range(2)]
    events = [torch.cuda.Event() if on_gpu else None for _ in range(2)]

    def fetch(k: int):
        lo, hi = k * per, min((k + 1) * per, rows)
        fill(lo, hi, bufs[k & 1][:hi - lo])
        if on_gpu:
            events[k & 1].record()
        return lo, hi

    nchunks = (rows + per - 1) // per
    with open(path, 'wb') as fh:
        pending = fetch(0) if nchunks else None
        for k in range(nchunks):
            lo, hi = pending
            if on_gpu:
                events[k & 1].synchronize()
            if k + 1 < nchunks:
                pending = fetch(k + 1)
            fh.write(memoryview(bufs[k & 1][:hi - lo].numpy()).cast('B'))      # leading rows of a contiguous buffer


def _p0_header(module) -> Optional[Dict[str, int]]:
    """Seed and draw of a module whose P_0 comes from the counter-based generator (``p0_seed``), else None."""
    seed = getattr(module, 'p0_seed', None)
    return None if seed is None else {'seed': int(seed), 'draw': int(module.p0_draw)}


def save_checkpoint(module, directory: str, tag: str = 'walk_state', chunk_bytes: int = DEFAULT_CHUNK_BYTES) -> str:
    """Writes this rank's header + state file (every rank of a sharded state calls it).  The state streams to disk
    in chunks of rows through two pinned host buffers (device -> host copy of chunk k+1 overlaps the write of chunk
    k).  Returns the header path."""
    os.makedirs(directory, exist_ok=True)
    module.materialize()                                    # lazy decay: bring every row current first
    global_n = int(getattr(module, 'global_node_num', module.node_num))
    world, rank, rows = _shard_info(module, global_n)
    L1, d = module.num_layer + 1, module.dim
    path = shard_path(directory, tag, rank, world)
    spath = state_path(path)
    per = max(1, int(chunk_bytes) // (L1 * d * 4))
    state = module._state
    on_gpu = state.is_cuda
    _write_rows(spath + '.tmp', rows, per, (L1, d), torch.float32, on_gpu,
                lambda lo, hi, buf: buf.copy_(state[lo:hi, :, :d], non_blocking=on_gpu))
    header = {'format': FORMAT, 'world': int(world), 'rank': int(rank), 'global_node_num': int(global_n), 'dim': int(d),
              'num_layer': int(module.num_layer), 'now_time': float(module._now_host),
              'begging_time': float(module.begging_time.item()), 'rows': int(rows),
              'mlp': {k: v.detach().to('cpu') for k, v in module.mlp.state_dict().items()},
              'p0': _p0_header(module)}
    torch.save(header, path + '.tmp')
    os.replace(spath + '.tmp', spath)
    os.replace(path + '.tmp', path)                         # the header appears last: a reader never sees half a shard
    return path


def list_shards(directory: str, tag: str) -> List[str]:
    """The complete, consistent set of shard files of a checkpoint (raises if ranks are missing or mixed)."""
    pat = re.compile(re.escape(tag) + r'\.rank(\d+)-of-(\d+)\.pt$')
    found = {}
    for p in glob.glob(os.path.join(directory, tag + '.rank*-of-*.pt')):
        m = pat.search(os.path.basename(p))
        if m:
            found[(int(m.group(1)), int(m.group(2)))] = p
    worlds = {w for _, w in found}
    if not found:
        raise FileNotFoundError(f'no checkpoint {tag!r} in {directory}')
    if len(worlds) != 1:
        raise ValueError(f'checkpoint {tag!r} in {directory} mixes world sizes {sorted(worlds)}')
    world = worlds.pop()
    missing = [r for r in range(world) if (r, world) not in found]
    if missing:
        raise FileNotFoundError(f'checkpoint {tag!r}: shards of ranks {missing} of {world} are missing')
    return [found[(r, world)] for r in range(world)]


def load_checkpoint(module, directory: str, tag: str = 'walk_state', load_head: bool = True,
                    chunk_bytes: int = DEFAULT_CHUNK_BYTES) -> None:
    """Reads a checkpoint written with ANY number of ranks into this module's rows (re-sharding by node id:
    a single-GPU state can be loaded into 8 shards and back).  State files are memory-mapped and copied in chunks."""
    global_n = int(getattr(module, 'global_node_num', module.node_num))
    world, rank, rows = _shard_info(module, global_n)
    total = 0
    header = None
    with torch.no_grad():
        for path in list_shards(directory, tag):
            payload = torch.load(path, map_location='cpu', mmap=True, weights_only=True)
            if payload.get('format') not in (FORMAT, FORMAT_V1):
                raise ValueError(f'{path}: not a {FORMAT} file')
            if (int(payload['global_node_num']) != global_n or int(payload['dim']) != module.dim
                    or int(payload['num_layer']) != module.num_layer):
                raise ValueError(f'{path}: checkpoint is for {payload["global_node_num"]} nodes, dim {payload["dim"]}, '
                                 f'{payload["num_layer"]} layers; the module has {global_n}, {module.dim}, '
                                 f'{module.num_layer}')
            if payload['format'] == FORMAT_V1:
                total += scatter_shard(module._state[:rows], world, rank, payload)
            else:
                n, L1, d = int(payload['rows']), int(payload['num_layer']) + 1, int(payload['dim'])
                if n:
                    want = n * L1 * d * 4
                    if os.path.getsize(state_path(path)) != want:
                        raise ValueError(f'{state_path(path)}: {os.path.getsize(state_path(path))} bytes, expected {want}')
                    mm = np.memmap(state_path(path), dtype='<f4', mode='r', shape=(n, L1, d))
                    per = max(1, int(chunk_bytes) // (L1 * d * 4))
                    for lo in range(0, n, per):
                        chunk = torch.from_numpy(np.array(mm[lo:lo + per]))       # one bounded host copy
                        total += scatter_rows(module._state[:rows], world, rank, int(payload['world']),
                                              int(payload['rank']), chunk, first_row=lo)
                    del mm
            header = payload
        if total != rows:
            raise ValueError(f'checkpoint covers {total} of the {rows} rows of rank {rank}')
        module.now_time.data.fill_(header['now_time'])
        module.begging_time.data.fill_(header['begging_time'])
        if load_head:
            module.mlp.load_state_dict(header['mlp'])
        # a counter-mode module continues the saved generator: its next reset draws what the saved job's would
        if getattr(module, 'p0_seed', None) is not None and header.get('p0') is not None:
            module.p0_seed = int(header['p0']['seed'])
            module.p0_draw = int(header['p0']['draw'])
    module._after_external_write()                          # host clock mirror, lazy bookkeeping restart


# ---------------------------------------------------------------------------------------------- streaming sampler
_LIST_FIELDS = ('all_nbr', 'all_eid', 'all_t', 'old_nbr', 'old_eid', 'old_t')
_PEND_FIELDS = ('pend_node', 'pend_nbr', 'pend_eid', 'pend_t')


def sampler_row_bytes(capacity: int) -> int:
    """Bytes of one node's record: ALL and OLD (neighbour, edge id, time; ``capacity`` entries each), the two counts
    and the newest folded time."""
    return 48 * int(capacity) + 16


def sampler_record_dtype(capacity: int) -> np.dtype:
    """The row record of a ``.lists`` file as a numpy structured type (packed, little-endian)."""
    C = int(capacity)
    return np.dtype([(k, '<f8' if k.endswith('_t') else '<i8', (C,)) for k in _LIST_FIELDS]
                    + [('all_cnt', '<i4'), ('old_cnt', '<i4'), ('newest', '<f8')])


def lists_path(header_path: str) -> str:
    return header_path[:-3] + '.lists'


def _sampler_tables(sampler) -> List[torch.Tensor]:
    """The per-node tables in record order."""
    return [sampler._lists[k] for k in _LIST_FIELDS] + [sampler._all_cnt, sampler._old_cnt, sampler._newest]


def _record_fields(chunk: torch.Tensor, tables: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    """Views of a uint8 [m, 48 C + 16] block of records, one per table (the table's dtype and row shape)."""
    out, off = [], 0
    for t in tables:
        w = int(np.prod(t.shape[1:])) * t.element_size()
        out.append(chunk[:, off:off + w].view(t.dtype).reshape((chunk.shape[0],) + tuple(t.shape[1:])))
        off += w
    return out


def save_sampler(sampler, directory: str, tag: str = 'sampler', chunk_bytes: int = DEFAULT_CHUNK_BYTES) -> str:
    """Writes this rank's part of a streaming sampler: a header with the pending batch, and the records of the nodes
    the rank owns (every rank of a ``ShardedStreamingSampler`` calls it).  The pending batch is saved as it is, not
    folded, so the latest batch's queries stay answerable after a load.  Records stream to disk through two pinned
    host buffers of ``chunk_bytes``.  A sampler with a flagged device error raises (``check_errors``) before anything
    is written: its answers are unspecified.  Returns the header path."""
    sampler.check_errors()
    world, rank, rows = _shard_info(sampler, sampler.num_nodes)
    C = int(sampler.max_neighbors)
    rb = sampler_row_bytes(C)
    os.makedirs(directory, exist_ok=True)
    path = shard_path(directory, tag, rank, world)
    lpath = lists_path(path)
    tables = _sampler_tables(sampler)
    on_gpu = sampler.device.type == 'cuda'
    per = max(1, int(chunk_bytes) // rb)
    staging = torch.empty(min(per, max(rows, 1)), rb, dtype=torch.uint8, device=sampler.device)

    def fill(lo: int, hi: int, buf: torch.Tensor) -> None:
        for f, t in zip(_record_fields(staging[:hi - lo], tables), tables):
            f.copy_(t[lo:hi])
        buf.copy_(staging[:hi - lo], non_blocking=on_gpu)

    _write_rows(lpath + '.tmp', rows, per, (rb,), torch.uint8, on_gpu, fill)
    count = int(sampler._pend_count.item())
    header = {'format': SAMPLER_FORMAT, 'world': world, 'rank': rank, 'num_nodes': int(sampler.num_nodes),
              'capacity': C, 'rows': rows, 'last_time': float(sampler._last_time.item()), 'pend_count': count}
    header.update({k: sampler._pend[k][:count].cpu() for k in _PEND_FIELDS})
    torch.save(header, path + '.tmp')
    os.replace(lpath + '.tmp', lpath)
    os.replace(path + '.tmp', path)                         # the header appears last: a reader never sees half a shard
    return path


def sampler_shards(directory: str, tag: str, num_nodes: int, capacity: int) -> List[Tuple[str, dict]]:
    """(header path, header) of every shard of a sampler checkpoint, after every check a load makes before it writes:
    a complete set of shards, the format, the node count and capacity, each shard's row count and ``.lists`` size,
    and the same pending batch and last time in every shard."""
    shards = []
    for path in list_shards(directory, tag):
        h = torch.load(path, map_location='cpu', mmap=True, weights_only=True)
        if not isinstance(h, dict) or h.get('format') != SAMPLER_FORMAT:
            raise ValueError(f'{path}: not a {SAMPLER_FORMAT} file')
        if int(h['num_nodes']) != num_nodes or int(h['capacity']) != capacity:
            raise ValueError(f'{path}: checkpoint is for {h["num_nodes"]} nodes and capacity {h["capacity"]}; the '
                             f'sampler has {num_nodes} and {capacity}')
        want_rows = rows_on_rank(num_nodes, int(h['world']), int(h['rank']))
        if int(h['rows']) != want_rows:
            raise ValueError(f'{path}: {h["rows"]} rows, rank {h["rank"]} of {h["world"]} owns {want_rows}')
        size, want = os.path.getsize(lists_path(path)), want_rows * sampler_row_bytes(capacity)
        if size != want:
            raise ValueError(f'{lists_path(path)}: {size} bytes, expected {want}')
        shards.append((path, h))
    first = shards[0][1]
    for path, h in shards[1:]:
        if (int(h['pend_count']) != int(first['pend_count']) or float(h['last_time']) != float(first['last_time'])
                or not all(torch.equal(h[k], first[k]) for k in _PEND_FIELDS)):
            raise ValueError(f'{path}: its pending batch differs from the one of {shards[0][0]}')
    return shards


def _read_rows(path: str, rows: int, per: int, row_bytes: int, device: torch.device
               ) -> Iterator[Tuple[int, torch.Tensor]]:
    """(lo, uint8 [m, row_bytes] on ``device``) for the chunks of a raw file, read through two (pinned) host buffers:
    the read of chunk k+1 runs while chunk k is copied to the device."""
    on_gpu = device.type == 'cuda'
    bufs = [torch.empty(min(per, max(rows, 1)), row_bytes, dtype=torch.uint8, pin_memory=on_gpu) for _ in range(2)]
    events = [None, None]
    with open(path, 'rb') as fh:
        for k, lo in enumerate(range(0, rows, per)):
            buf = bufs[k & 1][:min(per, rows - lo)]
            if events[k & 1] is not None:
                events[k & 1].synchronize()                 # the copy that last read this buffer is done
            if fh.readinto(memoryview(buf.numpy()).cast('B')) != buf.numel():
                raise ValueError(f'{path}: shorter than its header says')
            chunk = buf.to(device, non_blocking=on_gpu)
            if on_gpu:
                events[k & 1] = torch.cuda.Event()
                events[k & 1].record()
            yield lo, chunk


def load_sampler(sampler, directory: str, tag: str = 'sampler', chunk_bytes: int = DEFAULT_CHUNK_BYTES) -> None:
    """Reads a sampler checkpoint written with ANY number of ranks into this sampler (re-sharding by node id; every
    rank of a ``ShardedStreamingSampler`` calls it).  Everything ``sampler_shards`` checks raises before anything is
    written.  Then the sampler is reset (a sharded one: a new cache generation, and its next query takes the rank
    barrier), its owned rows are filled from every shard and the pending batch and last pushed time are restored:
    the next push and queries answer exactly as the saved sampler's would.  The tables are written in place, so a
    CUDA graph captured on this sampler before the load stays valid, unless the pending batch exceeds
    ``2 * max_batch``: then the pending buffers grow, which is refused inside a capture."""
    world, rank, rows = _shard_info(sampler, sampler.num_nodes)
    C = int(sampler.max_neighbors)
    rb = sampler_row_bytes(C)
    shards = sampler_shards(directory, tag, int(sampler.num_nodes), C)
    first = shards[0][1]
    count = int(first['pend_count'])
    if count > 2 * sampler.max_batch:
        sampler._grow((count + 1) // 2)
    sampler.reset()
    tables = _sampler_tables(sampler)
    owned = [t[:rows] for t in tables]
    per = max(1, int(chunk_bytes) // rb)
    total = 0
    with torch.no_grad():
        for path, h in shards:
            for lo, chunk in _read_rows(lists_path(path), int(h['rows']), per, rb, sampler.device):
                total += scatter_rows(owned, world, rank, int(h['world']), int(h['rank']),
                                      _record_fields(chunk, tables), first_row=lo)
        if total != rows:
            raise ValueError(f'checkpoint covers {total} of the {rows} rows of rank {rank}')
        for k in _PEND_FIELDS:
            sampler._pend[k][:count].copy_(first[k])
        sampler._pend_count.fill_(count)
        sampler._last_time.fill_(float(first['last_time']))
    sampler._last_host = float(first['last_time'])
