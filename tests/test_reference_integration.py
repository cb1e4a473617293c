"""Drop-in wiring against the unmodified reference, as ``oracle/make_ref.py`` installs it into
``oracle/_ref/TPNet`` (skipped where it is not installed).  No compute: the module has no CPU path; what is
checked is that the reference's own loader accepts the synthetic datasets, that the launcher binds
the CUDA-backed class under the reference's import, and that the reference assembles its model around it."""
import dataclasses
import logging
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

import tpnet_b200
from oracle.make_ref import ref_dir
from tpnet_b200 import launch
from tpnet_b200.synth import SHAPES, write_processed_dataset

REF = ref_dir()
needs_reference = pytest.mark.skipif(not REF, reason='reference not installed (oracle/make_ref.py copies it from a '
                                                     'TPNet checkout)')


@pytest.fixture()
def in_tmp(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    return tmp_path


@needs_reference
def test_reference_loader_accepts_synthetic_datasets(in_tmp):
    ref = launch.install(REF)
    assert ref.RandomProjectionModule is tpnet_b200.RandomProjectionModule
    from utils.DataLoader import get_link_prediction_data           # the reference's loader
    wiki = dataclasses.replace(SHAPES['wikipedia'], num_src=60, num_dst=15, num_edges=900)
    write_processed_dataset(wiki, str(in_tmp), seed=0)
    node_f, edge_f, full, train, val, test, nn_val, nn_test = get_link_prediction_data(
        'wikipedia', 0.15, 0.15, logging.getLogger())
    assert node_f.shape == (76, 172) and edge_f.shape == (901, 172) and not edge_f[0].any()
    assert full.num_interactions == 900 and full.num_unique_nodes == 75
    assert full.src_node_ids.min() == 1 and full.src_node_ids.max() == 60
    assert full.dst_node_ids.min() == 61 and full.dst_node_ids.max() == 75
    assert np.all(np.diff(full.node_interact_times) >= 0)
    assert 0 < train.num_interactions < 900 and val.num_interactions > 0 and test.num_interactions > 0
    # Flights-shaped: one id space, day stamps that the loader converts to seconds
    fl = dataclasses.replace(SHAPES['flights'], name='Flights', num_src=50, num_edges=800)
    write_processed_dataset(fl, str(in_tmp), seed=2, edge_feat_dim=1)
    _, edge_f, full, *_ = get_link_prediction_data('Flights', 0.15, 0.15, logging.getLogger(), convert_time=True)
    assert edge_f.shape == (801, 172) and full.num_unique_nodes == 50
    assert np.all(full.node_interact_times % 86400.0 == 0) and len(np.unique(full.node_interact_times)) > 3


@needs_reference
def test_reference_assembles_its_model_around_the_drop_in(in_tmp):
    ref = launch.install(REF)
    from models.modules import LinkPredictor_v1
    from utils.DataLoader import get_link_prediction_data
    from utils.utils import get_neighbor_sampler
    wiki = dataclasses.replace(SHAPES['wikipedia'], num_src=40, num_dst=10, num_edges=600)
    write_processed_dataset(wiki, str(in_tmp), seed=1)
    node_f, edge_f, full, train, *_ = get_link_prediction_data('wikipedia', 0.15, 0.15, logging.getLogger())
    sampler = get_neighbor_sampler(data=train, sample_neighbor_strategy='recent', seed=0)
    # the constructor call of train_link_prediction.py:126-133
    rp = ref.RandomProjectionModule(node_num=node_f.shape[0], edge_num=edge_f.shape[0], dim_factor=10, num_layer=2,
                                    time_decay_weight=1e-6, device='cpu', use_matrix=False,
                                    beginning_time=train.node_interact_times[0], not_scale=False, enforce_dim=-1)
    assert isinstance(rp, tpnet_b200.RandomProjectionModule)
    backbone = ref.TPNet(node_raw_features=node_f, edge_raw_features=edge_f, neighbor_sampler=sampler, time_feat_dim=100,
                         random_projections=rp, num_neighbors=20, num_layers=2, dropout=0.1, device='cpu')
    head = LinkPredictor_v1(input_dim1=172, input_dim2=172, hidden_dim=172, output_dim=1, random_projections=rp,
                            not_encode=False)
    model = torch.nn.Sequential(backbone, head)
    assert backbone.random_projections is rp and head.random_projections is rp
    trainable = [n for n, p in model.named_parameters() if p.requires_grad]
    assert any('random_projections.mlp' in n for n in trainable)              # the head of the drop-in is trained
    assert not any(n.endswith(('random_projections.random_projections.0', 'now_time')) for n in trainable)
    keys = [k for k in model.state_dict().keys() if 'random_projections' in k]
    assert any(k.endswith('random_projections.random_projections.2') for k in keys)
    assert any(k.endswith('random_projections.begging_time') for k in keys)
    # compute needs CUDA: loud failure, not a silent CPU path
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        rp.update(train.src_node_ids[:5], train.dst_node_ids[:5], train.node_interact_times[:5])


def test_launcher_runs_a_reference_style_script(in_tmp):
    """`python -m tpnet_b200.launch <checkout> <script>`: the script sees the drop-in under the reference's import
    path, its own argv, the checkout as working directory, and `random.sample` on a set (DataLoader.py:156)."""
    fake = in_tmp / 'checkout'
    (fake / 'models').mkdir(parents=True)
    (fake / 'models' / '__init__.py').write_text('')
    (fake / 'models' / 'TPNet.py').write_text('class RandomProjectionModule:\n    pass\nclass TPNet:\n    pass\n')
    (fake / 'probe.py').write_text(
        'import os, random, sys\n'
        'from models.TPNet import TPNet, RandomProjectionModule\n'
        'random.seed(2020)\n'
        'picked = random.sample({3, 1, 2, 5, 8}, 2)\n'
        'print(RandomProjectionModule.__module__, sys.argv[1:], os.path.basename(os.getcwd()), len(picked))\n')
    repo = os.path.dirname(os.path.dirname(os.path.abspath(tpnet_b200.__file__)))
    r = subprocess.run([sys.executable, '-m', 'tpnet_b200.launch', str(fake), 'probe.py', '--dataset_name', 'wikipedia'],
                       capture_output=True, text=True, cwd=repo, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip().splitlines()[-1] == "tpnet_b200.random_projection ['--dataset_name', 'wikipedia'] checkout 2"


def test_launcher_gpu_sampler_option(in_tmp):
    """`--tpn-gpu-sampler`: consumed by the launcher; `utils.utils.get_neighbor_sampler` keeps the reference's
    sampler for every strategy but 'recent'."""
    fake = in_tmp / 'checkout2'
    (fake / 'models').mkdir(parents=True)
    (fake / 'utils').mkdir()
    (fake / 'models' / '__init__.py').write_text('')
    (fake / 'utils' / '__init__.py').write_text('')
    (fake / 'models' / 'TPNet.py').write_text('class RandomProjectionModule:\n    pass\n')
    (fake / 'utils' / 'utils.py').write_text(
        'def get_neighbor_sampler(data, sample_neighbor_strategy="uniform", time_scaling_factor=0.0, seed=None):\n'
        '    return ("reference sampler", sample_neighbor_strategy, seed)\n')
    (fake / 'probe.py').write_text(
        'import sys\n'
        'from utils.utils import get_neighbor_sampler\n'
        'print(get_neighbor_sampler(data=None, sample_neighbor_strategy="uniform", seed=3), '
        'getattr(get_neighbor_sampler, "_tpn_gpu_sampler", False), sys.argv[1:])\n')
    repo = os.path.dirname(os.path.dirname(os.path.abspath(tpnet_b200.__file__)))
    # --gpu 0: where CUDA is present the launcher selects that device, so it must exist on a one-GPU machine
    for extra, patched in (([], False), (['--tpn-gpu-sampler'], True)):
        r = subprocess.run([sys.executable, '-m', 'tpnet_b200.launch', str(fake), 'probe.py', '--gpu', '0'] + extra,
                           capture_output=True, text=True, cwd=repo, timeout=300)
        assert r.returncode == 0, r.stderr
        assert r.stdout.strip().splitlines()[-1] == f"('reference sampler', 'uniform', 3) {patched} ['--gpu', '0']"


def test_launcher_selects_the_device_named_by_gpu(in_tmp, monkeypatch):
    """`--gpu G` is parsed by the launcher and made the current CUDA device before the script runs (the reference
    scripts only build the string 'cuda:G'); torch.cuda.set_device is recorded, so any G works on any machine."""
    fake = in_tmp / 'checkout3'
    (fake / 'models').mkdir(parents=True)
    (fake / 'models' / 'TPNet.py').write_text('')
    (fake / 'probe.py').write_text('import sys\nopen("argv.txt", "w").write(repr(sys.argv[1:]))\n')
    chosen = []
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: True)
    monkeypatch.setattr(torch.cuda, 'set_device', chosen.append)
    monkeypatch.setattr(sys, 'argv', list(sys.argv))
    monkeypatch.setattr(sys, 'path', list(sys.path))
    monkeypatch.setattr(random, 'sample', random.sample)
    launch.main([str(fake), 'probe.py', '--tpn-stock', '--gpu', '3'])       # --tpn-stock: nothing is imported or swapped
    assert chosen == [3]
    assert (fake / 'argv.txt').read_text() == repr(['--gpu', '3'])
