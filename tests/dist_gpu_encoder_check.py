"""Multi-GPU check of the sharded encoder call and get_random_projections, launched by torchrun (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        tests/dist_gpu_encoder_check.py

Every rank runs ShardedRandomProjection (peer data plane: device-side routing, NVLink pulls, flag barriers) on the
same replicated stream; rank 0 also runs the single-GPU module.  With gather=True every rank must hold the reference's
tensors: the encoder features (head included, tensor-core head: bit-equal) and the rows of get_random_projections
(bit-equal), and every rank must hold the same ones."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import RandomProjectionModule  # noqa: E402
from tpnet_b200.sharded import ShardedRandomProjection  # noqa: E402


def same_everywhere(x: torch.Tensor) -> bool:
    y = x.clone()
    dist.broadcast(y, 0)
    flag = torch.tensor([1 if torch.equal(x, y) else 0], device=x.device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item())


def main():
    rank = int(os.environ['RANK']); local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    ok = True
    N, dim, L = 2003, 140, 3
    for mode in ('eager', 'lazy'):
        kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=L, time_decay_weight=1e-4, device=str(dev),
                  use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=dim)
        torch.manual_seed(7)
        sh = ShardedRandomProjection(decay_mode=mode, ext_rows=2 * N + 64, exchange='peer', state_device=dev,
                                     **kw).to(dev)
        ref = None
        if rank == 0:
            torch.manual_seed(7)
            ref = RandomProjectionModule(decay_mode=mode, **kw).to(dev)
            ref.mlp.load_state_dict(sh.mlp.state_dict())
        rng = np.random.default_rng(3)
        t = 0.0
        for B, m, K in ((3000, 401, 20), (500, 57, 7), (9000, 1, 20)):
            s = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
            d = (1 + (rng.zipf(1.3, B) - 1) % (N - 1)).astype(np.int64)
            ts = np.sort(t + rng.random(B) * 500.0)
            t = ts[-1]
            nbr = rng.integers(0, N, (m, K)).astype(np.int64)
            src = rng.integers(1, N, m).astype(np.int64)
            dst = rng.integers(1, N, m).astype(np.int64)
            ids = rng.integers(0, N, 777).astype(np.int64)
            with torch.no_grad():
                feat = sh.get_neighbor_pair_wise_feature(nbr, src, dst, gather=True)
            rows = sh.get_random_projections(ids, gather=True)
            ok &= same_everywhere(feat) and all(same_everywhere(r) for r in rows)
            if rank == 0:
                with torch.no_grad():
                    want = ref.get_neighbor_pair_wise_feature(nbr, src, dst)
                good = torch.equal(feat, want) and all(torch.equal(a, b) for a, b in zip(rows, ref.get_random_projections(ids)))
                if not good:
                    print(f'MISMATCH mode={mode} m={m} K={K}: max abs err {(feat - want).abs().max().item()}')
                ok &= good
            sh.update(s, d, ts)
            if ref is not None:
                ref.update(s, d, ts)
        sh.check_errors()
        sh.close()
        del sh
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.broadcast(flag, 0)
        ok = bool(flag.item())
        if rank == 0:
            print(f'mode={mode} world={dist.get_world_size()}: {"ok" if ok else "FAILED"}')
    dist.barrier()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)
    if rank == 0:
        print('sharded encoder calls == single GPU: PASS')


if __name__ == '__main__':
    main()
