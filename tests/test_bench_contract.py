"""bench.py's reference arm (the CPU legs, runnable without a GPU): one JSON line with the keys the contract names, for the
headline workload and for the training step; the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _run(*args, timeout=300):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + list(args), capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    return r


def test_reference_arm_training_line():
    r = _run('--impl', 'reference', '--workload', 'train', '--steps', '1', '--warmup', '0')
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d['impl'] == 'reference' and d['metric'] == 'train_samples_per_s'
    assert d['value'] > 0 and d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {"value": d['value'], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d['gpu_launches'] == 0 and d['config']['cpu_sample_only'] is True


def test_steps_and_warmup_are_what_was_asked_for():
    """--steps / --warmup set the steps the arm runs, also above the reference training arm's defaults."""
    r = _run('--impl', 'reference', '--workload', 'train', '--steps', '6', '--warmup', '2')
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][0])
    assert (d['steps'], d['warmup']) == (6, 2)
    for bad in (['--steps', '0'], ['--warmup', '-1'], ['--impl', 'reference', '--dump-outputs', 'x']):
        r = _run(*bad, timeout=60)
        assert r.returncode != 0 and 'error' in r.stderr


def _dumped(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


@pytest.mark.gpu
def test_dump_outputs_of_the_tile_workload(tmp_path):
    """--dump-outputs writes the last timed step's super-resolved tile (a seeded pixel sample and the top-left corner) as
    float32 .npy files under 64 MB, the same on a second run with the same arguments."""
    runs = []
    for i in range(2):
        d = str(tmp_path / ('run%d' % i))
        r = _run('--tile', '660', '--steps', '2', '--warmup', '1', '--no-cpu-baseline', '--no-facade', '--dump-outputs', d)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][0])
        assert line['steps'] == 2 and line['warmup'] == 1
        runs.append(_dumped(d))
    got = runs[0]
    assert set(got) == {'sr_pixel_sample', 'sr_corner'}
    assert all(a.dtype == np.float32 for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got['sr_pixel_sample'].shape == (660 * 660, 6) and got['sr_corner'].shape == (512, 512, 6)
    assert np.array_equal(got['sr_pixel_sample'].reshape(660, 660, 6)[:512, :512], got['sr_corner'])    # whole tile sampled
    assert np.isfinite(got['sr_corner']).all() and got['sr_corner'].std() > 0
    assert all(np.array_equal(got[k], runs[1][k]) for k in got)


@pytest.mark.gpu
def test_dump_outputs_of_the_training_step(tmp_path):
    d = str(tmp_path / 'train')
    r = _run('--workload', 'train', '--train-batch', '8', '--steps', '3', '--warmup', '1', '--no-cpu-baseline', '--dump-outputs', d)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][0])
    assert line['steps'] == 3 and line['warmup'] == 1
    got = _dumped(d)
    assert set(got) == {'loss', 'mse', 'params_sample'}
    assert got['loss'].shape == (1,) and np.isfinite(got['loss']).all() and got['loss'][0] > 0
    assert got['params_sample'].dtype == np.float32 and got['params_sample'].shape == (1789574,)        # all of DSen2's


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'train', '--gpus', '2'],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith('{')]


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    for extra in ([], ['--workload', 'train']):
        r = _run('--steps', '1', '--warmup', '0', *extra, timeout=120)
        assert r.returncode != 0 and 'no CPU fallback' in (r.stderr + r.stdout)
