"""GPU suite of the negative edge sampler (tpn_neg_sampler_*): bit equality with the numpy restatement of the device
algorithm (oracle/negative_sampler.py) for all three strategies, repeatability, CUDA-graph capture, error flags and
refusals."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.negative_sampler import DeviceRestatement  # noqa: E402
from tpnet_b200 import NegativeEdgeSampler, RandomProjectionModule  # noqa: E402
from tpnet_b200.pipeline import StepGraphs  # noqa: E402
from tpnet_b200.synth import SHAPES, GraphShape, edge_stream  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def stream(shape, edges, batch=1000, seed=0):
    parts = list(edge_stream(shape, batch, edges // batch, seed=seed))
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


def eval_batches(t, first, B):
    for i in range(first, len(t), B):
        yield i, min(i + B, len(t))


def assert_same(got, want):
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.parametrize('shape_name, edges', [('wikipedia', 157_000), ('reddit', 200_000), ('flights', 400_000)])
@pytest.mark.parametrize('strategy', ['random', 'historical', 'inductive'])
def test_bit_equal_to_the_restatement_over_a_split(shape_name, edges, strategy):
    src, dst, t = stream(SHAPES[shape_name], edges)
    val = int(0.70 * len(t))
    first = int(0.85 * len(t))
    lot = float(t[val])
    seed = 0 if strategy != 'random' else 17
    gpu = NegativeEdgeSampler(src, dst, t, lot, strategy, seed=seed, device=DEV)
    ref = DeviceRestatement(src, dst, t if strategy != 'random' else None, lot, seed=seed)
    assert np.array_equal(gpu.unique_src_node_ids, ref.S) and np.array_equal(gpu.unique_dst_node_ids, ref.D)
    src_d, dst_d, t_d = (torch.from_numpy(a).to(DEV) for a in (src, dst, t))
    for call, (i, j) in enumerate(eval_batches(t, first, 200)):
        want = ref.sample(strategy, call, j - i, src[i:j], dst[i:j], t[i], t[j - 1])
        if call % 2:
            got = gpu.sample(j - i, src[i:j], dst[i:j], t[i], t[j - 1])
        else:
            s, d = gpu.sample(j - i, src_d[i:j], dst_d[i:j], t_d[i], t_d[j - 1], as_tensors=True)
            got = (s.cpu().numpy(), d.cpu().numpy())
        assert_same(got, want)
    gpu.check_errors()


@pytest.mark.parametrize('strategy', ['historical', 'inductive'])
def test_bit_equal_on_a_power_law_replica_with_batches_of_100000(strategy):
    shape = GraphShape('powerlaw-replica', 1_000_000, 0, 2_000_000, 3, 1e-7, 6.0e4, False, 1.2)
    src, dst, t = stream(shape, 2_000_000, batch=100_000, seed=3)
    lot = float(t[1_000_000])
    gpu = NegativeEdgeSampler(src, dst, t, lot, strategy, seed=11, device=DEV)
    ref = DeviceRestatement(src, dst, t, lot, seed=11)
    for call, i in enumerate((1_500_000, 1_700_000, 1_900_000)):
        j = i + 100_000
        assert_same(gpu.sample(j - i, src[i:j], dst[i:j], t[i], t[j - 1]),
                    ref.sample(strategy, call, j - i, src[i:j], dst[i:j], t[i], t[j - 1]))


def small_graph(seed, E=300, n=12, ties=4):
    rng = np.random.default_rng(seed)
    src = rng.integers(1, n + 1, E)
    dst = rng.integers(1, n + 1, E)
    t = np.floor(rng.random(E) * E / ties)
    return src.astype(np.int64), dst.astype(np.int64), t


@pytest.mark.parametrize('strategy', ['historical', 'inductive'])
@pytest.mark.parametrize('size', [1, 7, 60, 400])
def test_bit_equal_in_the_fill_and_with_replacement_cases(strategy, size):
    src, dst, t = small_graph(size)
    lot = float(np.quantile(t, 0.3))
    gpu = NegativeEdgeSampler(src, dst, t, lot, strategy, seed=5, device=DEV)
    ref = DeviceRestatement(src, dst, t, lot, seed=5)
    order = np.argsort(t, kind='stable')
    for call, i in enumerate(range(0, len(t), 23)):
        idx = order[i:i + 23]
        s, e = t[idx[0]], t[idx[-1]]
        assert_same(gpu.sample(size, src[idx], dst[idx], s, e), ref.sample(strategy, call, size, src[idx], dst[idx], s, e))
    # a batch naming ids outside S / D and an empty batch exclude nothing extra
    bs = np.array([0, 10 ** 9, 3], dtype=np.int64)
    bd = np.array([2, 5, 10 ** 9], dtype=np.int64)
    call = gpu.call_index
    assert_same(gpu.sample(size, bs, bd, 10.0, 20.0), ref.sample(strategy, call, size, bs, bd, 10.0, 20.0))
    assert_same(gpu.sample(size, bs[:0], bd[:0], 10.0, 20.0), ref.sample(strategy, call + 1, size, bs[:0], bd[:0], 10.0, 20.0))


def test_reset_random_state_repeats_the_draws():
    src, dst, t = small_graph(1, E=2000, n=60)
    for strategy in ('random', 'historical'):
        gpu = NegativeEdgeSampler(src, dst, t, None, strategy, seed=3, device=DEV)
        first = [gpu.sample(50, src[:50], dst[:50], 100.0, 120.0) for _ in range(4)]
        gpu.reset_random_state()
        again = [gpu.sample(50, src[:50], dst[:50], 100.0, 120.0) for _ in range(4)]
        for a, b in zip(first, again):
            assert_same(a, b)
        assert not np.array_equal(first[0][1], first[1][1])


def test_seed_none_draws_the_key_from_numpys_global_generator():
    src, dst, t = small_graph(2)
    np.random.seed(4)
    a = NegativeEdgeSampler(src, dst, device=DEV)
    np.random.seed(4)
    b = NegativeEdgeSampler(src, dst, device=DEV)
    assert_same(a.sample(100), b.sample(100))
    with pytest.raises(ValueError):
        NegativeEdgeSampler(src, dst, t, None, 'historical', device=DEV).sample(5, src[:5], dst[:5], 0.0, 1.0)


def test_cuda_graphs_per_batch_replay_the_eager_calls():
    src, dst, t = stream(SHAPES['wikipedia'], 60_000)
    src_d, dst_d, t_d = (torch.from_numpy(a).to(DEV) for a in (src, dst, t))
    gpu = NegativeEdgeSampler(src, dst, t, None, 'historical', seed=2, device=DEV)
    spans = list(eval_batches(t, 50_000, 200))[:20]
    eager = [gpu.sample(j - i, src[i:j], dst[i:j], t[i], t[j - 1]) for i, j in spans]
    gpu.reset_random_state()
    graphs, outs = [], []
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for i, j in spans:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                outs.append(gpu.sample(j - i, src_d[i:j], dst_d[i:j], t_d[i], t_d[j - 1], as_tensors=True))
            graphs.append(g)
    torch.cuda.synchronize()
    for g, (s, d), want in zip(graphs, outs, eager):
        g.replay()
        torch.cuda.synchronize()
        assert_same((s.cpu().numpy(), d.cpu().numpy()), want)


def test_step_graphs_custom_step_samples_inside_the_graph():
    src, dst, t = stream(SHAPES['wikipedia'], 30_000)
    gpu = NegativeEdgeSampler(src, dst, t, None, 'historical', seed=8, device=DEV)
    spans = list(eval_batches(t, 25_000, 200))[:10]
    gpu.sample(200, src[:200], dst[:200], t[0], t[199])               # sizes the workspace before any capture
    gpu.reset_random_state()
    eager = [gpu.sample(j - i, src[i:j], dst[i:j], t[i], t[j - 1]) for i, j in spans]
    gpu.reset_random_state()
    sh = SHAPES['wikipedia']
    module = RandomProjectionModule(node_num=sh.node_num, edge_num=sh.edge_num, dim_factor=10, num_layer=2,
                                    time_decay_weight=1e-6, use_matrix=False, beginning_time=0.0, not_scale=False,
                                    enforce_dim=-1, device=DEV).to(DEV)
    batches = [tuple(torch.from_numpy(a[i:j]).to(DEV) for a in (src, dst, t)) + (float(t[j - 1]),) for i, j in spans]
    out = {'neg_src': torch.empty(200, dtype=torch.int64, device=DEV),
           'neg_dst': torch.empty(200, dtype=torch.int64, device=DEV)}

    def step(m, b, o):
        s, d = gpu.sample(len(b[0]), b[0], b[1], b[2][0], b[2][-1], as_tensors=True)
        o['neg_src'][:len(s)].copy_(s)
        o['neg_dst'][:len(d)].copy_(d)
        m.update(b[0], b[1], b[2], next_time=b[3])

    graphs = StepGraphs(module, batches, step=step, out=out, max_batch=200)
    for k, want in enumerate(eager):
        o = graphs.replay(k)
        n = len(want[0])
        assert_same((o['neg_src'][:n].cpu().numpy(), o['neg_dst'][:n].cpu().numpy()), want)


def test_empty_fill_domain_sets_the_device_flag():
    src = np.array([1, 1, 2, 2], dtype=np.int64)
    dst = np.array([3, 4, 3, 4], dtype=np.int64)
    t = np.array([0.0, 1.0, 2.0, 3.0])
    gpu = NegativeEdgeSampler(src, dst, t, None, 'historical', seed=1, device=DEV)
    with pytest.raises(ValueError):
        gpu.sample(3, src, dst, 0.0, 3.0)
    s, d = gpu.sample(3, torch.from_numpy(src).to(DEV), torch.from_numpy(dst).to(DEV), 0.0, 3.0, as_tensors=True)
    assert (s.cpu().numpy() == -1).all()
    with pytest.raises(ValueError):
        gpu.check_errors()
    gpu.check_errors()                                                  # cleared


def test_sample_refusals():
    src, dst, t = small_graph(0)
    gpu = NegativeEdgeSampler(src, dst, t, None, 'historical', seed=1, device=DEV)
    for args, exc in [((-1, src, dst, 0.0, 1.0), ValueError), ((2.5, src, dst, 0.0, 1.0), ValueError),
                      ((5, None, dst, 0.0, 1.0), ValueError), ((5, src, dst[:-1], 0.0, 1.0), ValueError),
                      ((5, src, dst, float('nan'), 1.0), ValueError),
                      ((5, src, dst, torch.zeros(2, dtype=torch.float64, device=DEV), 1.0), ValueError),
                      ((5, src, dst, torch.zeros((), dtype=torch.float32, device=DEV), 1.0), ValueError)]:
        with pytest.raises(exc):
            gpu.sample(*args)
    assert gpu.call_index == 0
    assert len(gpu.sample(0, src, dst, 0.0, 1.0)[0]) == 0


# Different negatives move AP / AUC by sampling noise only.  A bound, not a parity claim: 2 points.
TOL_NEG_ARM = 0.02


def test_reference_scripts_run_with_the_gpu_negative_sampler():
    """evaluate_link_prediction.py, unmodified, with --tpn-gpu-sampler --tpn-gpu-neg-sampler under `historical`
    negatives on a down-scaled Flights replica: it completes, and test / new-node test AP and AUC lie within
    TOL_NEG_ARM of the stock arm on the same checkpoint (the draws differ, so this is not a parity test)."""
    sys.path.insert(0, os.path.join(ROOT, 'scripts'))
    import apauc_parity
    if not os.path.isfile(os.path.join(apauc_parity.REF, 'models', 'TPNet.py')):
        pytest.skip('oracle/_ref/TPNet not installed (oracle/make_ref.py copies it from a TPNet checkout)')
    res = apauc_parity.parity_run('flights', epochs=1, edges=20000, src=500, negative='historical', timeout=1500,
                                  train_both=False, gpu_neg_arm=True)
    for split, metrics in res['eval_stock'].items():
        for name, value in metrics.items():
            assert abs(value - res['eval_xevalneg'][split][name]) <= TOL_NEG_ARM, (split, name, res)
