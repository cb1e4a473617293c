"""Streaming-sampler checkpoints (tpnet_b200/checkpoint.py: save_sampler / load_sampler): host logic, runs on CPU.

The record format, the header checks, the re-sharding row scatter and the file sizes are host code.  ``HostSampler``
holds the attributes the two functions read and write, as CPU tensors, so a whole save -> load round trip runs here;
the CUDA classes themselves are covered by tests/test_gpu_sampler_checkpoint.py."""
import os

import numpy as np
import pytest
import torch

from tpnet_b200 import checkpoint as ck
from tpnet_b200.sharded import rows_on_rank

LISTS = ('all_nbr', 'all_eid', 'all_t', 'old_nbr', 'old_eid', 'old_t')
PEND = ('pend_node', 'pend_nbr', 'pend_eid', 'pend_t')


class HostSampler:
    """Rank ``rank`` of ``world`` of a streaming sampler, on CPU tensors: owned rows + ``cache`` cache rows."""

    def __init__(self, N, C, world=1, rank=0, max_batch=4, cache=3):
        self.num_nodes, self.max_neighbors, self.world, self.rank = N, C, world, rank
        self.n_local = rows_on_rank(N, world, rank)
        self.device = torch.device('cpu')
        rows = self.n_local + cache
        self._lists = {k: torch.full((rows, C), -7, dtype=torch.float64 if k.endswith('_t') else torch.int64)
                       for k in LISTS}
        self._all_cnt = torch.full((rows,), -7, dtype=torch.int32)
        self._old_cnt = torch.full((rows,), -7, dtype=torch.int32)
        self._newest = torch.full((rows,), -7.0, dtype=torch.float64)
        self._pend_count = torch.zeros(1, dtype=torch.int32)
        self._last_time = torch.full((1,), -np.inf, dtype=torch.float64)
        self.max_batch = 0
        self._grow(max_batch)
        self._last_host = -np.inf
        self.flag = None
        self.resets = 0

    def _grow(self, max_batch):
        pend = {'pend_node': torch.zeros(2 * max_batch, dtype=torch.int32),
                'pend_nbr': torch.zeros(2 * max_batch, dtype=torch.int64),
                'pend_eid': torch.zeros(2 * max_batch, dtype=torch.int64),
                'pend_t': torch.zeros(2 * max_batch, dtype=torch.float64)}
        for k, v in pend.items():
            if self.max_batch:
                v[:2 * self.max_batch] = self._pend[k]
        self._pend, self.max_batch = pend, max_batch

    def check_errors(self):
        if self.flag is not None:
            self.flag, e = None, self.flag
            raise e

    def reset(self):
        self.resets += 1
        self._all_cnt.zero_()
        self._old_cnt.zero_()
        self._newest.fill_(-np.inf)
        self._pend_count.zero_()
        self._last_time.fill_(-np.inf)
        self._last_host = -np.inf

    def fill(self, pend_count=6, last_time=41.5):
        """Every owned row holds values derived from its node id; a pending batch of ``pend_count`` entries."""
        C = self.max_neighbors
        u = torch.arange(self.n_local, dtype=torch.int64) * self.world + self.rank
        for i, k in enumerate(LISTS):
            v = u[:, None] * 1000 + 100 * i + torch.arange(C)[None, :]
            self._lists[k][:self.n_local] = v.double() + 0.25 if k.endswith('_t') else v
        self._all_cnt[:self.n_local] = (u % (C + 1)).int()
        self._old_cnt[:self.n_local] = (u % C).int()
        self._newest[:self.n_local] = u.double() + 0.5
        if pend_count > 2 * self.max_batch:
            self._grow((pend_count + 1) // 2)
        j = torch.arange(pend_count)
        self._pend['pend_node'][:pend_count] = (j // 2).int()
        self._pend['pend_nbr'][:pend_count] = j * 3
        self._pend['pend_eid'][:pend_count] = j + 10 ** 12
        self._pend['pend_t'][:pend_count] = last_time - (pend_count - 1 - j).double()
        self._pend_count.fill_(pend_count)
        self._last_time.fill_(last_time)
        return self

    def owned(self):
        return [t[:self.n_local] for t in ck._sampler_tables(self)]


def expected_rows(N, C, world, rank):
    return HostSampler(N, C, world, rank).fill().owned()


# ---------------------------------------------------------------- format and sizes
def test_record_layout_and_file_sizes():
    for C in (1, 20, 40):
        dt = ck.sampler_record_dtype(C)
        assert dt.itemsize == ck.sampler_row_bytes(C) == 48 * C + 16
        assert [dt.fields[k][1] for k in LISTS] == [i * 8 * C for i in range(6)]
        assert (dt.fields['all_cnt'][1], dt.fields['old_cnt'][1], dt.fields['newest'][1]) == (48 * C, 48 * C + 4,
                                                                                               48 * C + 8)
    # the 10M-node power-law sampler at C = 20: 9.76 GB of records in all, split by node id over the ranks
    N, rb = 10_000_001, ck.sampler_row_bytes(20)
    assert rb == 976 and N * rb == 9_760_000_976
    for G in (1, 2, 3, 8):
        rows = [rows_on_rank(N, G, r) for r in range(G)]
        assert sum(rows) == N and max(rows) - min(rows) <= 1
    per = ck.DEFAULT_CHUNK_BYTES // rb                       # rows per chunk: host memory is two chunks, not the table
    assert per == 68_759 and 2 * per * rb <= 2 * ck.DEFAULT_CHUNK_BYTES
    assert -(-N // per) == 146


def test_saved_files_hold_the_records_and_the_header(tmp_path):
    N, C = 29, 3
    s = HostSampler(N, C, world=2, rank=1).fill(pend_count=6)
    path = ck.save_sampler(s, str(tmp_path), chunk_bytes=4 * ck.sampler_row_bytes(C))   # 4 rows a chunk, ragged tail
    assert path.endswith('sampler.rank1-of-2.pt') and ck.lists_path(path).endswith('sampler.rank1-of-2.lists')
    h = torch.load(path, weights_only=True)
    assert h['format'] == ck.SAMPLER_FORMAT
    assert (h['world'], h['rank'], h['num_nodes'], h['capacity'], h['rows']) == (2, 1, N, C, 14)
    assert h['pend_count'] == 6 and h['last_time'] == 41.5
    for k in PEND:
        assert torch.equal(h[k], s._pend[k][:6])
    rec = np.fromfile(ck.lists_path(path), dtype=ck.sampler_record_dtype(C))
    assert rec.shape == (14,)
    for name, t in zip(LISTS + ('all_cnt', 'old_cnt', 'newest'), s.owned()):
        assert np.array_equal(rec[name], t.numpy()), name
    assert sorted(os.listdir(tmp_path)) == ['sampler.rank1-of-2.lists', 'sampler.rank1-of-2.pt']      # no .tmp left


# ---------------------------------------------------------------- the shared row scatter
@pytest.mark.parametrize('saved_world', [1, 2, 3, 4])
@pytest.mark.parametrize('load_world', [1, 2, 3, 4])
def test_scatter_rows_places_every_node_once(saved_world, load_world):
    """Tables of mixed shapes and dtypes, saved shards fed in chunks of 4 rows: each node lands exactly once, in its
    row (u // load_world on rank u % load_world)."""
    N, C = 23, 3
    landed = 0
    for r in range(load_world):
        dst = HostSampler(N, C, load_world, r).owned()
        for t in dst:
            t.fill_(-1)
        got = 0
        for q in range(saved_world):
            src = expected_rows(N, C, saved_world, q)
            for lo in range(0, src[0].shape[0], 4):
                got += ck.scatter_rows(dst, load_world, r, saved_world, q, [t[lo:lo + 4] for t in src], first_row=lo)
        assert got == rows_on_rank(N, load_world, r)
        for d, w in zip(dst, expected_rows(N, C, load_world, r)):
            assert torch.equal(d, w)
        landed += got
    assert landed == N


def test_scatter_rows_fills_the_leading_columns_of_wider_rows():
    src = torch.arange(12, dtype=torch.float32).view(4, 3)
    dst = torch.zeros(2, 5)
    assert ck.scatter_rows(dst, 2, 1, 1, 0, src) == 2                 # nodes 1 and 3 -> rows 0 and 1
    assert torch.equal(dst[:, :3], src[1::2]) and not dst[:, 3:].any()


# ---------------------------------------------------------------- round trips
@pytest.mark.parametrize('saved_world', [1, 2, 3])
@pytest.mark.parametrize('load_world', [1, 2, 3, 4])
@pytest.mark.parametrize('N', [3, 29])
def test_round_trip_reshards_by_node_id(tmp_path, saved_world, load_world, N):
    """N = 3 leaves a rank of world 4 with no rows.  Chunks of 2 rows on save and 3 on load (ragged tails); a loading
    rank whose pending buffers are too small grows them."""
    C = 4
    for q in range(saved_world):
        ck.save_sampler(HostSampler(N, C, saved_world, q).fill(pend_count=10), str(tmp_path),
                        chunk_bytes=2 * ck.sampler_row_bytes(C))
    for r in range(load_world):
        s = HostSampler(N, C, load_world, r, max_batch=2)
        cache = {k: v[s.n_local:].clone() for k, v in s._lists.items()}
        ck.load_sampler(s, str(tmp_path), chunk_bytes=3 * ck.sampler_row_bytes(C))
        assert s.resets == 1 and s.max_batch == 5
        for d, w in zip(s.owned(), expected_rows(N, C, load_world, r)):
            assert torch.equal(d, w)
        assert not s._all_cnt[s.n_local:].any() and not s._old_cnt[s.n_local:].any()      # cache rows: empty
        assert all(torch.equal(s._lists[k][s.n_local:], v) for k, v in cache.items())
        want = HostSampler(N, C, 1, 0).fill(pend_count=10)
        assert int(s._pend_count) == 10 and float(s._last_time) == 41.5 and s._last_host == 41.5
        for k in PEND:
            assert torch.equal(s._pend[k][:10], want._pend[k][:10])


# ---------------------------------------------------------------- refusals: raised before anything is written
def untouched(s):
    return (s.resets == 0 and int(s._pend_count) == 0 and bool((s._all_cnt == -7).all())
            and bool((s._lists['all_nbr'] == -7).all()))


def save_world(tmp_path, tag, N, C, world, **kw):
    for q in range(world):
        ck.save_sampler(HostSampler(N, C, world, q).fill(**kw), str(tmp_path), tag)


def test_refusals(tmp_path):
    N, C = 29, 4
    d = str(tmp_path)
    save_world(tmp_path, 'two', N, C, 2)
    # node count or capacity of another sampler
    for s in (HostSampler(N + 1, C), HostSampler(N, C + 1)):
        with pytest.raises(ValueError, match='checkpoint is for'):
            ck.load_sampler(s, d, 'two')
        assert untouched(s)
    # a missing shard; shards of two world sizes under one tag
    os.rename(ck.shard_path(d, 'two', 1, 2), os.path.join(d, 'moved'))
    s = HostSampler(N, C)
    with pytest.raises(FileNotFoundError, match='ranks \\[1\\]'):
        ck.load_sampler(s, d, 'two')
    os.rename(os.path.join(d, 'moved'), ck.shard_path(d, 'two', 1, 2))
    ck.save_sampler(HostSampler(N, C).fill(), d, 'two')
    with pytest.raises(ValueError, match='mixes world sizes'):
        ck.load_sampler(s, d, 'two')
    with pytest.raises(FileNotFoundError):
        ck.load_sampler(s, d, 'nothing')
    assert untouched(s)
    # a .lists file of the wrong size
    save_world(tmp_path, 'cut', N, C, 2)
    with open(ck.lists_path(ck.shard_path(d, 'cut', 1, 2)), 'r+b') as fh:
        fh.truncate(ck.sampler_row_bytes(C) * 5)
    with pytest.raises(ValueError, match='bytes, expected'):
        ck.load_sampler(s, d, 'cut')
    assert untouched(s)
    # a header that is not a sampler header (a state checkpoint under the same tag), or a wrong row count
    torch.save(ck.pack_shard(torch.zeros(N, 2, 3), 1, 0, N, 0.0, 0.0, {}), ck.shard_path(d, 'state', 0, 1))
    with pytest.raises(ValueError, match=ck.SAMPLER_FORMAT):
        ck.load_sampler(s, d, 'state')
    save_world(tmp_path, 'rows', N, C, 1)
    h = torch.load(ck.shard_path(d, 'rows', 0, 1), weights_only=True)
    h['rows'] -= 1
    torch.save(h, ck.shard_path(d, 'rows', 0, 1))
    with pytest.raises(ValueError, match='owns'):
        ck.load_sampler(s, d, 'rows')
    # ranks whose pending batches differ
    ck.save_sampler(HostSampler(N, C, 2, 0).fill(pend_count=6), d, 'pend')
    ck.save_sampler(HostSampler(N, C, 2, 1).fill(pend_count=4), d, 'pend')
    with pytest.raises(ValueError, match='pending batch differs'):
        ck.load_sampler(s, d, 'pend')
    assert untouched(s)
    # a sampler with a flagged device error is not saved
    bad = HostSampler(N, C).fill()
    bad.flag = ValueError('pushed times decreased')
    with pytest.raises(ValueError, match='decreased'):
        ck.save_sampler(bad, os.path.join(d, 'flagged'), 'x')
    assert not os.path.exists(os.path.join(d, 'flagged'))
