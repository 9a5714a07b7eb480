"""bench.py's JSON contract, exercised on the CPU through the reference arm (the only arm that runs without a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + list(args), cwd=ROOT, env=e,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout


def _dumped(out_dir):
    got = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}
    assert set(got) == {'boxes', 'scores', 'labels', 'counts'}
    assert got['boxes'].dtype == got['scores'].dtype == np.float32
    assert got['labels'].dtype == got['counts'].dtype == np.float64
    n, k = got['scores'].shape
    assert got['boxes'].shape == (n, k, 4) and got['labels'].shape == (n, k) and got['counts'].shape == (n,)
    assert got['counts'].sum() > 0, 'the dump must not be vacuous'
    return got


def test_reference_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    lines = [l for l in _run('--impl', 'reference', '--workload', 'tiny', '--steps', '2', '--warmup', '1',
                             '--dump-outputs', str(tmp_path)).splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'images/sec' and d['unit'] == 'images/s'
    assert d['higher_is_better'] is True and d['n_gpus'] == 1 and d['steps'] == 2 and d['value'] > 0
    assert d['e2e'] == {'value': d['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['value'] == d['value'] and 1 <= cb['cores'] <= (os.cpu_count() or 1)
    assert 'workload' in d['config']
    assert _dumped(tmp_path)['counts'].shape == (1,)


def test_reference_arm_non_zero_ranks_exit_silently():
    out = _run('--impl', 'reference', '--workload', 'tiny', '--gpus', '2', '--steps', '1', '--warmup', '0',
               env={'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2'})
    assert out.strip() == ''


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'tiny', '--steps', '1'], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode != 0 and p.stdout.strip() == ''


@pytest.mark.gpu
def test_product_arm_dumps_the_same_outputs_for_the_same_arguments(tmp_path):
    """--dump-outputs: the last timed step's detections of the whole batch; the seeded inputs make two runs with the
    same arguments give identical files."""
    runs = []
    for name in ('a', 'b'):
        out = _run('--workload', 'tiny', '--steps', '2', '--warmup', '1', '--no-cpu-baseline',
                   '--dump-outputs', str(tmp_path / name))
        assert len([l for l in out.splitlines() if l.strip()]) == 1
        runs.append(_dumped(tmp_path / name))
    assert runs[0]['counts'].shape == (2,)
    for k in runs[0]:
        np.testing.assert_array_equal(runs[0][k], runs[1][k], err_msg=k)
