"""Multi-GPU check of the sharded streaming sampler, launched by torchrun (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29543 \
        tests/dist_gpu_sampler_check.py

Every rank runs ShardedStreamingSampler (symmetric peer memory, NVLink pulls, flag barriers on the device) on the same
replicated stream; rank 0 also runs the single-GPU StreamingRecentSampler.  After every push the slices of all ranks,
all-gathered by position, must be bit-equal to rank 0's single-GPU answers in all three arrays."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200.neighbor_sampler import ShardedStreamingSampler, StreamingRecentSampler  # noqa: E402


def gather_slices(local: torch.Tensor, per: int, m: int) -> torch.Tensor:
    pad = local.new_zeros((per,) + tuple(local.shape[1:]))
    pad[:local.shape[0]] = local
    full = local.new_empty((dist.get_world_size() * per,) + tuple(local.shape[1:]))
    dist.all_gather_into_tensor(full, pad)
    return full[:m]


def main():
    rank = int(os.environ['RANK']); local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    N, C, K = 20011, 20, 20
    s = ShardedStreamingSampler(N, C, dev, max_batch=40_000, cache_rows=N)
    plain = StreamingRecentSampler(N, C, dev, max_batch=40_000) if rank == 0 else None
    rng = np.random.default_rng(5)
    ok, t0 = True, 0.0
    for B in (1, 5000, 30_000, 777, 40_000, 3):
        src = ((rng.zipf(1.3, B) - 1) % N).astype(np.int64)
        dst = ((rng.zipf(1.3, B) - 1) % N).astype(np.int64)
        t = t0 + np.sort(np.floor(rng.random(B) * 50.0))
        t0 = t[-1]
        eid = rng.integers(1, 1 << 40, B)
        s.push(src, dst, eid, t)
        qn = np.concatenate([src, dst, rng.integers(0, N, B + 64)]).astype(np.int64)
        qt = np.concatenate([t, t, t, t[-1] + np.floor(rng.random(64) * 3.0)])
        keep, nbr, e_, t_ = s.get_historical_neighbors(qn, qt, K, as_tensors=True)
        per = s.row_split(len(qn))[0]
        got = [gather_slices(x, per, len(qn)) for x in (nbr, e_, t_)]
        if plain is not None:
            plain.push(src, dst, eid, t)
            want = plain.get_historical_neighbors(qn, qt, K, as_tensors=True)
            good = all(torch.equal(a, b) for a, b in zip(got, want))
            if not good:
                print(f'MISMATCH after a push of {B} edges: {[int((a != b).sum()) for a, b in zip(got, want)]}')
            ok &= good
    s.check_errors()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, 0)
    ok = bool(flag.item())
    s.close()
    dist.barrier()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)
    if rank == 0:
        print(f'sharded streaming sampler (world {int(os.environ["WORLD_SIZE"])}) == single GPU: PASS')


if __name__ == '__main__':
    main()
