"""bench.py's reference arm on CPU (tiny preset): one JSON line with the result keys (the GPU arm prints the same keys
plus roofline / clocks / gpu_launches).  --dump-outputs: the writer on CPU, the GPU arm's dump on a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--preset', 'tiny',
                        '--steps', '2', '--warmup', '3'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.strip()]
    assert len(lines) == 1                                       # ONE JSON line
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'train_samples_per_s' and d['unit'] == 'samples/s'
    assert d['higher_is_better'] is True and d['scaling'] == 'weak' and d['vs_baseline'] is None
    assert d['dtype'] == 'f32' and d['data'] == 'synthetic' and d['n_gpus'] == 1
    assert d['value'] > 0 and d['ms_per_step'] > 0 and d['steps'] >= 1 and d['warmup'] >= 1
    assert 'workload' in d['config'] and 'model' not in d['config']
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == d['value'] and cb['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_gpu_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--preset', 'tiny', '--steps', '2'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and 'no CPU fallback' in (r.stderr + r.stdout)


def test_dump_outputs_writes_float_arrays_within_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, 'DUMP_ARRAY_BYTES', 4096)
    big = np.random.RandomState(0).standard_normal((100, 16)).astype(np.float32)        # 6400 B: rows sampled
    bench.dump_outputs(str(tmp_path / 'out'), {'ids': np.arange(5), 'sums': np.ones(3), 'big': big})
    got = {f[:-4]: np.load(str(tmp_path / 'out' / f)) for f in os.listdir(str(tmp_path / 'out'))}
    assert sorted(got) == ['big', 'ids', 'sums']
    assert got['ids'].dtype == np.float32 and np.array_equal(got['ids'], np.arange(5))
    assert got['sums'].dtype == np.float64
    rows = np.sort(np.random.RandomState(bench.SEED).choice(100, 64, replace=False))
    assert got['big'].nbytes <= 4096 and np.array_equal(got['big'], big[rows])


def test_dump_outputs_needs_the_gpu_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--preset', 'tiny',
                        '--dump-outputs', str(tmp_path / 'out')], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and '--dump-outputs' in r.stderr and not os.path.exists(str(tmp_path / 'out'))


@pytest.mark.gpu
def test_gpu_arm_dumps_what_the_timed_steps_computed(tmp_path):
    """Two runs with the same arguments: the same arrays, and the same inputs behind them (the parameters the
    timed steps started from are seeded, so the last step's outputs agree to rounding)."""
    runs = []
    for name in ('a', 'b'):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--preset', 'tiny', '--steps', '5',
                            '--warmup', '3', '--eval-users', '64', '--no-extra-legs', '--no-cpu-baseline',
                            '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line['steps'] == 5 and line['warmup'] == 3
        runs.append({f[:-4]: np.load(str(out / f)) for f in os.listdir(str(out))})
    a, b = runs
    U, I = 2000, 5000
    shapes = {'train_prediction': (256,), 'train_loss': (), 'param_uid_embeddings_weight': (U, 64),
              'param_iid_embeddings_weight': (I, 64), 'param_mlp_0_weight': (64, 64 + 768), 'param_mlp_0_bias': (64,),
              'eval_prediction': (64 * 1001,), 'eval_metrics': (5,)}
    assert {k: v.shape for k, v in a.items()} == shapes
    assert sum(v.nbytes for v in a.values()) <= 64 * 10 ** 6
    assert a['eval_metrics'].dtype == np.float64 and all(a[k].dtype == np.float32 for k in shapes if k != 'eval_metrics')
    for k in shapes:
        assert np.isfinite(a[k]).all(), k
        assert np.allclose(a[k], b[k], rtol=1e-5, atol=1e-6), k
