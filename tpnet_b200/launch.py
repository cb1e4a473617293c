"""Runs an UNMODIFIED reference script on the B200 drop-in:

    python -m tpnet_b200.launch /path/to/TPNet train_link_prediction.py --dataset_name wikipedia \
        --model_name TPNet --use_random_projection --gpu 0 ...

What it does before handing control to the script (``runpy``, ``__name__ == '__main__'``):
  * puts the reference checkout first on ``sys.path`` and makes it the working directory (the
    scripts read ``./processed_data`` and write ``./logs``, ``./saved_models``);
  * replaces ``models.TPNet.RandomProjectionModule`` by ``tpnet_b200.RandomProjectionModule``, so
    ``from models.TPNet import TPNet, RandomProjectionModule`` (``train_link_prediction.py:36``,
    ``evaluate_link_prediction.py:33``) binds the CUDA-backed class;
  * Python >= 3.11 only: lets ``random.sample`` accept a set again (``utils/DataLoader.py:156``
    relies on the pre-3.11 behaviour, which converted the set with ``tuple()``).
  * with ``--tpn-gpu-sampler`` (an option of the launcher, removed before the script sees its arguments):
    ``utils.utils.get_neighbor_sampler`` returns ``tpnet_b200.neighbor_sampler.RecentNeighborSampler`` for
    the `recent` strategy (the one TPNet uses; any other strategy still gets the reference's sampler).
  * with ``--tpn-gpu-neg-sampler`` (also consumed here): ``utils.utils.NegativeEdgeSampler`` is
    ``tpnet_b200.NegativeEdgeSampler`` on the script's device, for every strategy.  Same sets, sizes and ordering
    rule, different draws (a counter-based generator instead of numpy's MT19937): not a parity arm.
  * with ``--tpn-stock`` (also consumed here): NOTHING is swapped — the reference's own class runs, with only the
    Python >= 3.11 ``random.sample`` shim applied.  This is the comparison arm of ``scripts/apauc_parity.py``.
  * ``--gpu G``: ``torch.cuda.set_device(G)`` before the script starts (the scripts only build the string
    ``cuda:G``; the library launches on the current device).
Nothing of the reference is copied or edited.
"""
from __future__ import annotations

import os
import random
import runpy
import sys
from typing import List


def allow_sampling_from_sets() -> None:
    """``random.sample(set, k)`` as CPython <= 3.10 did it: ``population = tuple(population)``."""
    if getattr(random.sample, '_tpn_set_shim', False):
        return
    original = random.sample

    def sample(population, k, *args, **kwargs):
        if isinstance(population, (set, frozenset)):
            population = tuple(population)
        return original(population, k, *args, **kwargs)

    sample._tpn_set_shim = True
    random.sample = sample


def use_gpu_sampler(device: str = 'cuda:0') -> None:
    """``utils.utils.get_neighbor_sampler`` (utils/utils.py:239-262) -> the GPU sampler for 'recent'."""
    import utils.utils as ref_utils                         # the reference's module, unmodified

    from .neighbor_sampler import RecentNeighborSampler
    if getattr(ref_utils.get_neighbor_sampler, '_tpn_gpu_sampler', False):
        return
    original = ref_utils.get_neighbor_sampler

    def get_neighbor_sampler(data, sample_neighbor_strategy: str = 'uniform', time_scaling_factor: float = 0.0,
                             seed: int = None):
        if sample_neighbor_strategy != 'recent':
            return original(data=data, sample_neighbor_strategy=sample_neighbor_strategy,
                            time_scaling_factor=time_scaling_factor, seed=seed)
        return RecentNeighborSampler(data.src_node_ids, data.dst_node_ids, data.edge_ids, data.node_interact_times,
                                     device)

    get_neighbor_sampler._tpn_gpu_sampler = True
    ref_utils.get_neighbor_sampler = get_neighbor_sampler


def use_gpu_neg_sampler(device: str = 'cuda:0') -> None:
    """``utils.utils.NegativeEdgeSampler`` (utils/utils.py:315-505) -> the GPU negative sampler."""
    import utils.utils as ref_utils                         # the reference's module, unmodified

    from .negative_sampler import NegativeEdgeSampler
    if getattr(ref_utils.NegativeEdgeSampler, '_tpn_gpu_neg_sampler', False):
        return

    class GpuNegativeEdgeSampler(NegativeEdgeSampler):
        _tpn_gpu_neg_sampler = True

        def __init__(self, src_node_ids, dst_node_ids, interact_times=None, last_observed_time=None,
                     negative_sample_strategy: str = 'random', seed: int = None):
            super().__init__(src_node_ids, dst_node_ids, interact_times, last_observed_time,
                             negative_sample_strategy, seed, device=device)

    ref_utils.NegativeEdgeSampler = GpuNegativeEdgeSampler


def install(reference_dir: str, gpu_sampler: bool = False, device: str = 'cuda:0', gpu_neg_sampler: bool = False):
    """Makes the reference importable and swaps in the drop-in class.  Returns ``models.TPNet``."""
    reference_dir = os.path.abspath(reference_dir)
    if not os.path.isfile(os.path.join(reference_dir, 'models', 'TPNet.py')):
        raise FileNotFoundError(f'{reference_dir} is not a TPNet checkout (models/TPNet.py not found)')
    if reference_dir not in sys.path:
        sys.path.insert(0, reference_dir)
    import models.TPNet as ref_tpnet                        # the reference's module, unmodified

    import tpnet_b200
    ref_tpnet.RandomProjectionModule = tpnet_b200.RandomProjectionModule
    if sys.version_info >= (3, 11):
        allow_sampling_from_sets()
    if gpu_sampler:
        use_gpu_sampler(device)
    if gpu_neg_sampler:
        use_gpu_neg_sampler(device)
    return ref_tpnet


def main(argv: List[str]) -> None:
    if len(argv) < 2:
        raise SystemExit('usage: python -m tpnet_b200.launch <TPNet checkout> <script.py> [script arguments ...]')
    reference_dir, script = os.path.abspath(argv[0]), argv[1]
    own = ('--tpn-gpu-sampler', '--tpn-gpu-neg-sampler', '--tpn-stock')
    rest = [a for a in argv[2:] if a not in own]
    gpu = 0
    if '--gpu' in rest and rest.index('--gpu') + 1 < len(rest):      # the scripts' own device option (load_configs.py)
        gpu = int(rest[rest.index('--gpu') + 1])
    if gpu >= 0:
        import torch
        if torch.cuda.is_available():
            torch.cuda.set_device(gpu)                      # the library launches on the CURRENT device
    if '--tpn-stock' in argv[2:]:
        # comparison arm: the reference's own RandomProjectionModule, untouched
        if reference_dir not in sys.path:
            sys.path.insert(0, reference_dir)
        if sys.version_info >= (3, 11):
            allow_sampling_from_sets()
    else:
        install(reference_dir, gpu_sampler='--tpn-gpu-sampler' in argv[2:], device=f'cuda:{gpu}',
                gpu_neg_sampler='--tpn-gpu-neg-sampler' in argv[2:])
    os.chdir(reference_dir)
    for d in ('logs', 'saved_models', 'saved_results'):     # the scripts expect these to exist or create them lazily
        os.makedirs(os.path.join(reference_dir, d), exist_ok=True)
    sys.argv = [script] + rest
    runpy.run_path(os.path.join(reference_dir, script), run_name='__main__')


if __name__ == '__main__':
    main(sys.argv[1:])
