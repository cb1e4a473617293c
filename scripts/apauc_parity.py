#!/usr/bin/env python
"""AP / AUC parity of the UNMODIFIED reference scripts on the B200 drop-in (north_star's third parity
criterion: "AP/AUC within 0.1 points").  Test / measurement infrastructure, not product code.

    python scripts/apauc_parity.py --shape wikipedia --epochs 2 --out profiles/r02_apauc_wikipedia.json
    python scripts/apauc_parity.py --shape flights --edges 400000 --negative historical ...

Needs the reference installed by ``oracle/make_ref.py`` into ``oracle/_ref/TPNet`` (git-ignored; it travels
to the GPU box with the snapshot) and a CUDA device.  What it runs, all through ``tpnet_b200.launch`` and
all with the reference's own ``train_link_prediction.py`` / ``evaluate_link_prediction.py``, unedited:

  arm "stock"   ``--tpn-stock``: the reference's own ``RandomProjectionModule`` (stock ATen ops on the same
                GPU, ``torch.use_deterministic_algorithms(True)`` as ``utils/utils.py:18-32`` sets it);
  arm "dropin"  ``tpnet_b200.RandomProjectionModule`` swapped in (the product path);
  cross-eval    the checkpoint TRAINED BY THE STOCK ARM is evaluated by ``evaluate_link_prediction.py`` twice,
                once with each class.  Same weights, same negatives (seeded samplers), so any AP/AUC difference
                is the hot path's alone — this is the sharp test; the two training runs additionally show that
                the choreography (.to(), reset, backup/reload, state_dict, early stopping) works end to end.

Synthetic datasets of the BASELINE shapes are written in the reference's on-disk format by
``tpnet_b200.synth.write_processed_dataset`` (the real datasets are not available offline).
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import re
import shutil
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tpnet_b200.synth import SHAPES, write_processed_dataset  # noqa: E402

REF = os.path.join(ROOT, 'oracle', '_ref', 'TPNet')
DATASET_NAME = {'wikipedia': 'wikipedia', 'reddit': 'reddit', 'flights': 'Flights'}


def make_dataset(shape_name: str, edges: int = 0, src: int = 0, dst: int = 0, seed: int = 0) -> str:
    shape = SHAPES[shape_name]
    shape = dataclasses.replace(shape, name=DATASET_NAME[shape_name])
    if edges:
        # a prefix-sized replica: same endpoint distribution and per-edge time step, fewer edges
        shape = dataclasses.replace(shape, num_edges=int(edges),
                                    time_span=shape.time_span * edges / SHAPES[shape_name].num_edges)
    if src:
        shape = dataclasses.replace(shape, num_src=int(src), num_dst=int(dst) if shape.num_dst else 0)
    feat = 1 if shape_name == 'flights' else 172       # Flights has 1-d edge features, padded by the loader
    marker = os.path.join(REF, 'processed_data', shape.name, 'SHAPE.json')
    want = dataclasses.asdict(shape)
    if os.path.isfile(marker) and json.load(open(marker)) == want:
        return shape.name
    write_processed_dataset(shape, REF, seed=seed, edge_feat_dim=feat, dtype='float32')
    json.dump(want, open(marker, 'w'))
    return shape.name


def run_script(script: str, prefix: str, dataset: str, shape_name: str, stock: bool, gpu: int, extra, log_dir: str,
               timeout: int):
    shape = SHAPES[shape_name]
    cmd = [sys.executable, '-m', 'tpnet_b200.launch', REF, script, '--prefix', prefix, '--dataset_name', dataset,
           '--model_name', 'TPNet', '--use_random_projection', '--rp_num_layer', str(shape.num_layer),
           '--rp_time_decay_weight', repr(shape.time_decay_weight), '--num_runs', '1', '--gpu', str(gpu)] + list(extra)
    if stock:
        cmd.append('--tpn-stock')
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get('PYTHONPATH', ''), TQDM_DISABLE='1')
    t0 = time.time()
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    dt = time.time() - t0
    os.makedirs(log_dir, exist_ok=True)
    with open(os.path.join(log_dir, f'{prefix}_{os.path.basename(script)}.log'), 'w') as fh:
        fh.write(' '.join(cmd) + '\n' + r.stdout[-20000:] + '\n--- stderr ---\n' + r.stderr[-20000:])
    if r.returncode != 0:
        raise RuntimeError(f'{" ".join(cmd)} failed ({r.returncode}):\n{r.stderr[-4000:]}')
    return dt


def read_metrics(path: str):
    d = json.load(open(path))
    return {k: {m: float(v) for m, v in d[k].items()} for k in d}


def read_validate_from_log(path: str):
    """Last epoch's validate / new node validate AP and AUC from the reference's log file (4 decimals)."""
    out = {}
    pat = re.compile(r'INFO - (validate|new node validate) (average_precision|roc_auc), ([0-9.]+)')
    for line in open(path):
        m = pat.search(line)
        if m:
            out.setdefault(m.group(1) + ' metrics', {})[m.group(2)] = float(m.group(3))
    return out


def diff(a, b):
    worst = 0.0
    for k in a:
        for m in a[k]:
            if k in b and m in b[k]:
                worst = max(worst, abs(a[k][m] - b[k][m]))
    return worst


def parity_run(shape_name: str, epochs: int, gpu: int = 0, edges: int = 0, src: int = 0, dst: int = 0,
               negative: str = 'random', log_dir: str = os.path.join(ROOT, 'gpurun_out', 'apauc'), timeout: int = 3000,
               train_both: bool = True, gpu_neg_arm: bool = False):
    if not os.path.isfile(os.path.join(REF, 'models', 'TPNet.py')):
        raise FileNotFoundError('oracle/_ref/TPNet missing: run `python oracle/make_ref.py` where /root/reference exists')
    dataset = make_dataset(shape_name, edges, src, dst)
    train_args = ['--num_epochs', str(epochs), '--patience', str(max(epochs, 1))]
    res = {'shape': shape_name, 'dataset': dataset, 'edges': edges or SHAPES[shape_name].num_edges, 'epochs': epochs,
           'negative_sample_strategy_eval': negative, 'seconds': {}}
    results = os.path.join(REF, 'saved_results')
    models = os.path.join(REF, 'saved_models')
    logs = os.path.join(REF, 'logs')

    res['seconds']['train_stock'] = run_script('train_link_prediction.py', 'stock', dataset, shape_name, True, gpu,
                                               train_args, log_dir, timeout)
    res['train_stock'] = read_metrics(os.path.join(results, f'stock_link_{dataset}_TPNet_seed0.json'))
    res['train_stock'].update(read_validate_from_log(os.path.join(logs, f'stock_link_{dataset}_TPNet.log')))
    if train_both:
        res['seconds']['train_dropin'] = run_script('train_link_prediction.py', 'dropin', dataset, shape_name, False,
                                                    gpu, train_args, log_dir, timeout)
        res['train_dropin'] = read_metrics(os.path.join(results, f'dropin_link_{dataset}_TPNet_seed0.json'))
        res['train_dropin'].update(read_validate_from_log(os.path.join(logs, f'dropin_link_{dataset}_TPNet.log')))
        res['train_max_abs_diff'] = diff(res['train_stock'], res['train_dropin'])

    # cross-evaluation of ONE checkpoint (the stock arm's) by both classes
    shutil.copyfile(os.path.join(models, f'stock_link_{dataset}_TPNet_seed0.pkl'),
                    os.path.join(models, f'xeval_link_{dataset}_TPNet_seed0.pkl'))
    ev = ['--negative_sample_strategy', negative]
    res['seconds']['eval_stock'] = run_script('evaluate_link_prediction.py', 'stock', dataset, shape_name, True, gpu, ev,
                                              log_dir, timeout)
    res['seconds']['eval_dropin'] = run_script('evaluate_link_prediction.py', 'xeval', dataset, shape_name, False, gpu,
                                               ev, log_dir, timeout)
    res['eval_stock'] = read_metrics(os.path.join(results, f'stock_link_{negative}_{dataset}_TPNet_seed0.json'))
    res['eval_dropin'] = read_metrics(os.path.join(results, f'xeval_link_{negative}_{dataset}_TPNet_seed0.json'))
    res['eval_max_abs_diff'] = diff(res['eval_stock'], res['eval_dropin'])
    res['tolerance'] = 0.001
    res['pass_eval'] = res['eval_max_abs_diff'] <= 0.001
    if gpu_neg_arm:
        # the same checkpoint with the GPU neighbour sampler, without and then with the GPU negative sampler; the
        # negative sampler draws other negatives from the same sets, so this arm is compared, not held to parity
        for prefix, flags in (('xevalnbr', ['--tpn-gpu-sampler']),
                              ('xevalneg', ['--tpn-gpu-sampler', '--tpn-gpu-neg-sampler'])):
            shutil.copyfile(os.path.join(models, f'stock_link_{dataset}_TPNet_seed0.pkl'),
                            os.path.join(models, f'{prefix}_link_{dataset}_TPNet_seed0.pkl'))
            res['seconds'][f'eval_{prefix}'] = run_script('evaluate_link_prediction.py', prefix, dataset, shape_name,
                                                          False, gpu, ev + flags, log_dir, timeout)
            res[f'eval_{prefix}'] = read_metrics(os.path.join(results, f'{prefix}_link_{negative}_{dataset}_TPNet_seed0.json'))
        res['eval_neg_sampler_max_abs_diff'] = diff(res['eval_stock'], res['eval_xevalneg'])
    if train_both:
        res['pass_train'] = res['train_max_abs_diff'] <= 0.001
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--shape', default='wikipedia', choices=list(DATASET_NAME))
    ap.add_argument('--epochs', type=int, default=1)
    ap.add_argument('--edges', type=int, default=0, help='0 = the full BASELINE edge count')
    ap.add_argument('--src', type=int, default=0)
    ap.add_argument('--dst', type=int, default=0)
    ap.add_argument('--gpu', type=int, default=0)
    ap.add_argument('--negative', default='random', choices=['random', 'historical', 'inductive'])
    ap.add_argument('--no-train-dropin', action='store_true')
    ap.add_argument('--gpu-neg-arm', action='store_true',
                    help='also evaluate the stock checkpoint with --tpn-gpu-sampler, then adding --tpn-gpu-neg-sampler')
    ap.add_argument('--timeout', type=int, default=3000)
    ap.add_argument('--out', default='')
    a = ap.parse_args()
    res = parity_run(a.shape, a.epochs, a.gpu, a.edges, a.src, a.dst, a.negative, timeout=a.timeout,
                     train_both=not a.no_train_dropin, gpu_neg_arm=a.gpu_neg_arm)
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, 'w').write(line + '\n')


if __name__ == '__main__':
    main()
