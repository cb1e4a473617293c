"""Multi-GPU check of a resumed stream job, launched by torchrun (one rank per GPU) twice, at two world sizes:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29547 \
        tests/dist_gpu_resume_check.py --phase save --dir D
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 1 --master-addr 127.0.0.1 --master-port 29547 \
        tests/dist_gpu_resume_check.py --phase resume --dir D

save: every rank runs ShardedStreamingSampler + ShardedRandomProjection (eager decay; symmetric peer memory, NVLink
pulls, flag barriers) over the first batches of a replicated stream, then writes save_checkpoint + save_sampler at
the batch boundary.  resume: the ranks of the new world size load both and run the remaining batches; rank 0 also
runs StreamingRecentSampler + RandomProjectionModule over the whole stream without a stop.  After every push the
slices of all ranks, all-gathered by position, must be bit-equal to rank 0's single-GPU answers, and at the end the
state rows must be bit-equal to the single-GPU state."""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import RandomProjectionModule  # noqa: E402
from tpnet_b200 import checkpoint as ck  # noqa: E402
from tpnet_b200.neighbor_sampler import ShardedStreamingSampler, StreamingRecentSampler  # noqa: E402
from tpnet_b200.sharded import ShardedRandomProjection  # noqa: E402

N, C, K = 20011, 20, 20
SIZES = (1, 5000, 30_000, 777, 40_000, 3, 12_000)
SAVE_AFTER = 3                                 # batches 0..3 before the stop, 4.. after it


def batches():
    rng = np.random.default_rng(5)
    t0 = 0.0
    for i, B in enumerate(SIZES):
        src = ((rng.zipf(1.3, B) - 1) % N).astype(np.int64)
        dst = ((rng.zipf(1.3, B) - 1) % N).astype(np.int64)
        t = t0 + np.sort(np.floor(rng.random(B) * 50.0))
        t0 = t[-1]
        eid = rng.integers(1, 1 << 40, B)
        qn = np.concatenate([src, dst, rng.integers(0, N, B + 64)]).astype(np.int64)
        qt = np.concatenate([t, t, t, t[-1] + np.floor(rng.random(64) * 3.0)])
        yield i, (src, dst, eid, t), qn, qt


def state_kw(dev):
    return dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=3, time_decay_weight=1e-4, device=str(dev),
                use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=64, decay_mode='eager')


def gather_slices(local: torch.Tensor, per: int, m: int) -> torch.Tensor:
    pad = local.new_zeros((per,) + tuple(local.shape[1:]))
    pad[:local.shape[0]] = local
    full = local.new_empty((dist.get_world_size() * per,) + tuple(local.shape[1:]))
    dist.all_gather_into_tensor(full, pad)
    return full[:m]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--phase', choices=('save', 'resume'), required=True)
    ap.add_argument('--dir', required=True)
    args = ap.parse_args()
    rank = int(os.environ['RANK']); local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    world = dist.get_world_size()
    torch.manual_seed(7)
    state = ShardedRandomProjection(ext_rows=2 * max(SIZES) + 64, state_device=dev, **state_kw(dev)).to(dev)
    sampler = ShardedStreamingSampler(N, C, dev, max_batch=max(SIZES), cache_rows=N)
    plain = ref = None
    if args.phase == 'resume':
        ck.load_checkpoint(state, args.dir, 'state')
        ck.load_sampler(sampler, args.dir, 'sampler')
        if rank == 0:
            torch.manual_seed(7)
            ref = RandomProjectionModule(**state_kw(dev)).to(dev)
            plain = StreamingRecentSampler(N, C, dev, max_batch=max(SIZES))
    ok = True
    with torch.no_grad():
        for i, (src, dst, eid, t), qn, qt in batches():
            if plain is not None:
                plain.push(src, dst, eid, t)
                ref.update(src, dst, t)
            if (args.phase == 'save') != (i <= SAVE_AFTER):
                continue
            sampler.push(src, dst, eid, t)
            keep, nbr, e_, t_ = sampler.get_historical_neighbors(qn, qt, K, as_tensors=True)
            state.update(src, dst, t)
            got = [gather_slices(x, sampler.row_split(len(qn))[0], len(qn)) for x in (nbr, e_, t_)]
            if plain is not None:
                want = plain.get_historical_neighbors(qn, qt, K, as_tensors=True)
                good = all(torch.equal(a, b) for a, b in zip(got, want))
                if not good:
                    print(f'SAMPLER MISMATCH at batch {i}: {[int((a != b).sum()) for a, b in zip(got, want)]}')
                ok &= good
        if args.phase == 'save':
            ck.save_checkpoint(state, args.dir, 'state')
            ck.save_sampler(sampler, args.dir, 'sampler')
        else:
            full = state.gather_global()
            if ref is not None:
                for layer, (a, b) in enumerate(zip(full, ref.random_projections)):
                    if not torch.equal(a, b.data):
                        print(f'STATE MISMATCH in layer {layer}: max abs err {(a - b.data).abs().max().item()}')
                        ok = False
    sampler.check_errors()
    state.check_errors()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, 0)
    ok = bool(flag.item())
    sampler.close()
    state.close()
    dist.barrier()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)
    if rank == 0:
        print(f'{args.phase} at world {world}: ' + ('saved' if args.phase == 'save' else
                                                    'resumed job == single GPU without a stop: PASS'))


if __name__ == '__main__':
    main()
