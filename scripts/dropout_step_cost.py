"""Cost of dropout in the training step: TrainEngine forward + backward, and one whole DataParallelTrainer.step, on the
`train` workload of bench.py (32 synthetic DIPS-shaped ragged pairs, 5-layer shared IEGMN, DB5 checkpoint weights), with
p = 0 and p = 0.25 alternated in the same process.  Each timing is the median of 5 repetitions of `--steps` steps, CUDA
events around the repetition; the card's name and power limit are printed with the numbers.  Writes one JSON line to
stdout (and to --out if given)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, 'tests')):
    sys.path.insert(0, _p)

import numpy as np
import torch

import bench
import bench_train
import golden_io as gio
from equidock_public_b200 import hetero_graph as hg
from equidock_public_b200 import synthetic
from equidock_public_b200.losses import PocketBatch
from equidock_public_b200.training import DataParallelTrainer, TrainEngine


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = f'{torch.cuda.get_device_name(0)}, power limit unknown'
    return q


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument('--pairs', type=int, default=32)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--p', type=float, default=0.25)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    ns = argparse.Namespace(workload='train', pairs_per_gpu=a.pairs, seed=0)
    triples, _, sizes = bench_train.make_train_pairs(ns, 0, 1, bench)
    batch = hg.batch_pairs(synthetic.to_torch_pairs([(t[0], t[1]) for t in triples])).to(dev)
    tl = lambda key: [torch.from_numpy(t[2][key]) for t in triples]
    tgt = PocketBatch(tl('bound_lig'), tl('bound_rec'), tl('pocket_lig'), tl('pocket_rec'), dev)
    ckpt = bench.WORKLOADS['train']['ckpt']
    arms = {}
    for p in (0.0, a.p):
        margs = dict(gio.load_args(ckpt))
        margs['dropout'] = p
        model = gio.build_model(ckpt, dev, args=margs).train()
        eng = TrainEngine(model)
        trainer = DataParallelTrainer(gio.build_model(ckpt, dev, args=margs), lr=1e-4, weight_decay=1e-4, clip=100.0)
        arms[p] = (eng, trainer)

    def fwd_bwd(eng):
        fwd = eng.forward(batch)
        eng.backward(fwd, torch.ones_like(fwd['ligand_coors']), torch.full_like(fwd['keypts'], 1e-2))

    bodies = {('train_engine_fwd_bwd', p): (lambda e=arms[p][0]: fwd_bwd(e)) for p in arms}
    bodies.update({('trainer_step', p): (lambda t=arms[p][1]: t.step(batch, tgt)) for p in arms})
    for body in bodies.values():          # warm-up of every shape / module of both arms
        for _ in range(3):
            body()
    torch.cuda.synchronize()
    times = {k: [] for k in bodies}
    for _ in range(a.reps):               # the two arms alternate inside every repetition
        for k, body in bodies.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                body()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.steps)
    res = {'card': card(), 'workload': f'bench.py train workload, {a.pairs} pairs, {sum(x + y for x, y in sizes)} residues',
           'steps_per_rep': a.steps, 'reps': a.reps, 'p': a.p, 'ms_per_step_median': {}, 'ms_per_step_all': {}}
    for (what, p), v in times.items():
        res['ms_per_step_median'][f'{what} p={p:g}'] = float(np.median(v))
        res['ms_per_step_all'][f'{what} p={p:g}'] = [round(x, 4) for x in v]
    for what in ('train_engine_fwd_bwd', 'trainer_step'):
        t0, t1 = float(np.median(times[(what, 0.0)])), float(np.median(times[(what, a.p)]))
        res[f'{what}_dropout_overhead_pct'] = 100.0 * (t1 - t0) / t0
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
