"""Multi-GPU check of the counter-based P_0, launched by torchrun (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29575 \
        tests/dist_gpu_p0_check.py

Every rank builds a ShardedRandomProjection with p0_seed (symmetric peer memory, eager and lazy decay), the ranks
all-gather P_0, and rank 0 compares it with a one-GPU RandomProjectionModule of the same p0_seed, bit for bit: after
construction and after each of two resets (the ranks run a routed update in between)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200 import RandomProjectionModule  # noqa: E402
from tpnet_b200.sharded import ShardedRandomProjection  # noqa: E402

N, DIM, SEED = 20011, 140, (1 << 63) + 12345


def main():
    rank = int(os.environ['RANK'])
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    torch.manual_seed(7)
    for mode in ('eager', 'lazy'):
        kw = dict(node_num=N, edge_num=10 * N, dim_factor=1, num_layer=3, time_decay_weight=1e-4, device=str(dev),
                  use_matrix=False, beginning_time=np.float64(0.0), not_scale=False, enforce_dim=DIM, decay_mode=mode)
        state = ShardedRandomProjection(ext_rows=2 * N, state_device=dev, p0_seed=SEED, **kw).to(dev)
        plain = RandomProjectionModule(state_device=dev, p0_seed=SEED, **kw).to(dev) if rank == 0 else None
        rng = np.random.default_rng(3)
        for k in range(3):
            if k:
                s, d = rng.integers(0, N, 5000), rng.integers(0, N, 5000)
                state.update(s, d, np.sort(rng.random(5000)) + k)
                state.reset_random_projections()
                if plain is not None:
                    plain.reset_random_projections()
            full = state.gather_global()[0]
            if rank == 0:
                assert torch.equal(full, plain.random_projections[0].data), (mode, k)
                assert state.p0_draw == plain.p0_draw == k
        dist.barrier()
    if rank == 0:
        print(f'PASS world {dist.get_world_size()}: P_0 equals the one-GPU module after construction and two resets')
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
