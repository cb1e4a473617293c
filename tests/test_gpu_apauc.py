"""GPU suite: the UNMODIFIED reference scripts (``oracle/_ref/TPNet``, installed by ``oracle/make_ref.py``)
on the drop-in — north_star's third parity criterion, AP/AUC within 0.1 points.

Down-scaled Wikipedia-shaped dataset (bipartite, 2 projection layers, batch 200, K=20), 2 epochs.
``scripts/apauc_parity.py`` runs ``train_link_prediction.py`` with the reference's own class and with
``tpnet_b200.launch`` swapping in the CUDA class, then evaluates the stock arm's checkpoint with
``evaluate_link_prediction.py`` under both classes.  Full-shape results: ``profiles/r02_apauc_*.json``.
Those two tests need the reference scripts and skip where they are not installed; the last test keeps the
module-level part of the same run (the calls the training makes on the module) as a comparison with the oracle.
"""
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

TOL = 0.001          # 0.1 points of AP / AUC (north_star)


@pytest.fixture(scope='module')
def parity():
    import apauc_parity
    if not os.path.isfile(os.path.join(apauc_parity.REF, 'models', 'TPNet.py')):
        pytest.skip('oracle/_ref/TPNet not installed (oracle/make_ref.py copies it from a TPNet checkout)')
    return apauc_parity.parity_run('wikipedia', epochs=2, edges=12000, src=400, dst=60, timeout=1500)


def test_same_checkpoint_same_ap_auc_under_both_classes(parity):
    """One checkpoint, evaluate_link_prediction.py under the reference class and under the drop-in: test and
    new-node test AP / AUC agree within 0.1 points (same weights and negatives: the hot path is the only difference)."""
    assert set(parity['eval_stock']) == {'test metrics', 'new node test metrics'}
    for split, metrics in parity['eval_stock'].items():
        for name, value in metrics.items():
            assert abs(value - parity['eval_dropin'][split][name]) <= TOL, (split, name, parity)
    assert all(0.0 < v <= 1.0 for m in parity['eval_dropin'].values() for v in m.values())


def test_training_on_the_drop_in_reaches_the_reference_ap_auc(parity):
    """train_link_prediction.py end to end on each class (reset per epoch, update per batch, backup / reload around
    validation, early-stopping checkpoints through state_dict): validate / test / new-node AP and AUC within 0.1 points."""
    for split in ('validate metrics', 'new node validate metrics', 'test metrics', 'new node test metrics'):
        for name, value in parity['train_stock'][split].items():
            assert abs(value - parity['train_dropin'][split][name]) <= TOL, (split, name, parity)


@pytest.mark.parametrize('mode', ['eager', 'lazy'])
def test_training_choreography_on_the_same_dataset_matches_the_oracle(mode):
    """The module-level half of the two tests above, which runs without the reference scripts: the calls their
    training makes on the random-projection module, on the same down-scaled Wikipedia shape (400 + 60 nodes, 12,000
    edges, batches of 200, 70 / 15 / 15 split).  Two epochs of: reset, then per training batch the decoder features
    of (src, dst) and (src, neg) followed by the update; backup, the validation batches the same way, reload.  Then
    state_dict / load_state_dict into a new module, which runs the test batches.  Every feature call and the layers
    after every phase are compared with the oracle, which the committed reference fixtures pin to the reference
    class bit for bit (tests/test_oracle.py)."""
    import dataclasses

    import numpy as np
    import torch

    from oracle.walk_projection import WalkProjectionOracle
    from test_gpu_parity import assert_layers, layers, module_from_cfg, pair_tol
    from tpnet_b200 import RandomProjectionModule
    from tpnet_b200.synth import SHAPES, edge_stream

    full = SHAPES['wikipedia']
    shape = dataclasses.replace(full, num_edges=12000, num_src=400, num_dst=60,
                                time_span=full.time_span * 12000 / full.num_edges)       # as apauc_parity.make_dataset
    batches = list(edge_stream(shape, 200, shape.num_edges // 200, seed=0))
    rng = np.random.default_rng(1)
    negs = [rng.integers(shape.num_src + 1, shape.node_num, 200).astype(np.int64) for _ in batches]
    n_train, n_val = 42, 9
    kw = dict(node_num=shape.node_num, edge_num=shape.edge_num, dim_factor=shape.dim_factor, num_layer=shape.num_layer,
              time_decay_weight=shape.time_decay_weight, use_matrix=False, beginning_time=float(batches[0][2][0]),
              not_scale=False, enforce_dim=-1)

    def run(m, o, lo, hi):
        for j in range(lo, hi):
            s, d, t = batches[j]
            for b in (d, negs[j]):
                got = m.pair_wise_gram(s, b).cpu().numpy()
                ref = o.pair_wise_gram(s, b, exact=True)
                tol = 1e-5 * np.abs(ref) + 2e-6 * pair_tol(o, s, b, np.expm1(ref.astype(np.float64))) + 1e-7
                assert np.all(np.abs(got - ref) <= tol), (mode, j, float(np.max(np.abs(got - ref) - tol)))
            m.update(s, d, t)
            o.update(s, d, t)

    o = WalkProjectionOracle(**kw)
    m = module_from_cfg(kw, o.P[0], mode)
    for epoch in range(2):
        torch.manual_seed(epoch)
        m.reset_random_projections()
        o.reset(m.random_projections[0].data.cpu().numpy())
        run(m, o, 0, n_train)
        assert_layers(layers(m), o.P, mode)
        saved, o_saved = m.backup_random_projections(), o.backup()
        run(m, o, n_train, n_train + n_val)
        m.reload_random_projections(saved)
        o.reload(o_saved)
        assert float(m.now_time.item()) == float(o.now_time)
        assert_layers(layers(m), o.P, mode)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    torch.manual_seed(99)                                       # another P_0: the state_dict must bring the real one
    m2 = RandomProjectionModule(device='cuda:0', decay_mode=mode, **dict(kw, beginning_time=np.float64(0.0))).to('cuda:0')
    m2.load_state_dict(sd)
    assert float(m2.now_time.item()) == float(o.now_time)
    assert_layers(layers(m2), o.P, mode)
    run(m2, o, n_train + n_val, len(batches))
    assert_layers(layers(m2), o.P, mode)
    m.check_errors()
    m2.check_errors()
