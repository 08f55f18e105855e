"""bench.py --dump-outputs: the arrays written for the last timed step (CPU: layout, dtypes, the seeded sample under the
size limit, argument checks; GPU: a real run's files against a direct forward of the same seeded batch)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _result(n_lig, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s, dt=torch.float32: torch.randn(*s, generator=g, dtype=dt)
    return ([r(n, 3) for n in n_lig], [r(50, 3) for _ in n_lig], [r(50, 3) for _ in n_lig],
            [r(3, 3, dt=torch.float64) for _ in n_lig], [r(1, 3, dt=torch.float64) for _ in n_lig])


def _load(d):
    return {k: np.load(os.path.join(d, f'{k}.npy')) for k in bench.OUTPUT_NAMES}


def test_dump_writes_every_output_in_pair_order(tmp_path):
    n_lig = [7, 3, 12]
    res = _result(n_lig)
    keep = bench.dump_outputs(str(tmp_path / 'out'), res)
    got = _load(tmp_path / 'out')
    assert list(keep) == [0, 1, 2]
    assert got['ligand_coors'].dtype == np.float32 and got['ligand_coors'].shape == (sum(n_lig), 3)
    assert np.array_equal(got['ligand_coors'], torch.cat(res[0]).numpy())
    for k, v in zip(bench.OUTPUT_NAMES[1:], res[1:]):
        assert np.array_equal(got[k], torch.stack(v).numpy()), k
    assert got['rotation'].dtype == np.float64 and got['translation'].shape == (3, 1, 3)


def test_dump_over_the_limit_writes_a_fixed_sample_of_whole_pairs(tmp_path):
    n_lig = [5, 40, 9, 200, 17, 60, 3, 33]
    res = _result(n_lig, seed=1)
    per_pair = [12 * n + 2 * 600 + 72 + 24 for n in n_lig]
    limit = sum(per_pair) // 2
    keep = bench.dump_outputs(str(tmp_path / 'a'), res, limit=limit)
    assert 0 < len(keep) < len(n_lig) and list(keep) == sorted(keep)
    assert sum(per_pair[i] for i in keep) <= limit
    assert list(bench.dump_outputs(str(tmp_path / 'b'), res, limit=limit)) == list(keep)
    got = _load(tmp_path / 'a')
    assert sum(v.nbytes for v in got.values()) <= limit
    assert np.array_equal(got['ligand_coors'], torch.cat([res[0][i] for i in keep]).numpy())
    for k, v in zip(bench.OUTPUT_NAMES[1:], res[1:]):
        assert np.array_equal(got[k], torch.stack([v[i] for i in keep]).numpy()), k


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--workload', 'train', '--dump-outputs', 'x'],
                                  ['--impl', 'reference', '--dump-outputs', 'x']])
def test_bench_refuses_arguments_it_cannot_honour(argv, tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv, cwd=tmp_path, capture_output=True,
                       text=True, timeout=120)
    assert p.returncode == 2 and 'error:' in p.stderr, p.stderr
    assert not (tmp_path / 'x').exists()


@pytest.mark.gpu
def test_bench_dump_is_the_forward_of_the_bench_batch(tmp_path, cuda_device):
    import argparse
    import golden_io as gio
    from equidock_public_b200 import hetero_graph as hg
    from equidock_public_b200 import synthetic
    out = tmp_path / 'dump'
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '3', '--warmup', '1', '--reps', '1',
                        '--pairs-per-gpu', '5', '--no-cpu-baseline', '--no-residue-e2e', '--dump-outputs', str(out)],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    got = _load(out)
    pairs, _, _ = bench.make_pairs(argparse.Namespace(workload='db5-shaped', pairs_per_gpu=5, seed=0), 0, 1)
    model = gio.build_model('dips', cuda_device)
    ref = model(hg.batch_pairs(synthetic.to_torch_pairs(pairs)).to(cuda_device), 0)
    assert got['ligand_coors'].shape == (5 * 200, 3) and got['keypts_ligand'].shape == (5, 50, 3)
    assert np.abs(got['ligand_coors'] - torch.cat(ref[0]).cpu().numpy()).max() < 1e-4
    for k, v in zip(bench.OUTPUT_NAMES[1:], ref[1:]):
        want = torch.stack(v).cpu().numpy()
        assert got[k].shape == want.shape and np.abs(got[k] - want).max() < 1e-4 * max(1.0, np.abs(want).max()), k
