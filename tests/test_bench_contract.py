"""bench.py contract checks that need no GPU: the reference arm prints ONE JSON line with the driver's keys, and the b200 arm
fails loudly (no CPU fallback) when there is no CUDA device."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
REQUIRED = ['impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
            'dtype', 'data', 'config', 'cpu_baseline', 'e2e']


def run(*flags, env=None):
    return subprocess.run([sys.executable, str(ROOT / 'bench.py'), *flags], capture_output=True, text=True, timeout=600,
                          env=dict(os.environ, **(env or {})))


def test_reference_arm_prints_the_contract_line():
    r = run('--impl', 'reference', '--steps', '1', '--warmup', '1')
    assert r.returncode == 0, r.stderr[-400:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith('{')]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for k in REQUIRED:
        assert k in j, k
    assert j['impl'] == 'reference' and j['metric'] == 'building_env_steps_per_sec' and j['higher_is_better'] is True
    assert j['vs_baseline'] is None and j['value'] > 0
    # the UNMODIFIED reference when oracle/_ref was built here (oracle/build_ref.py), else the oracle port
    expected = 'reference' if (ROOT / 'oracle' / '_ref' / 'site' / 'citylearn' / 'citylearn.py').is_file() else 'port'
    assert j['cpu_baseline']['kind'] == expected and j['cpu_baseline']['cores'] >= 1 and j['cpu_baseline']['value'] == j['value']
    assert j['e2e'] == {'value': j['value'], 'unit': j['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in j['config'] and '17 buildings x 4096 envs' in j['config']['workload']


def test_reference_arm_other_ranks_exit_quietly():
    r = run('--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '1', env={'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_b200_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('needs a machine without a CUDA device')
    r = run('--steps', '1', '--warmup', '1', '--no-cpu-baseline')
    assert r.returncode != 0
    assert 'CUDA' in (r.stderr + r.stdout)


def test_dump_outputs_samples_the_same_envs_of_every_array(tmp_path):
    import numpy as np
    from bench import dump_outputs
    E = 1000
    arrays = {'a': np.arange(E * 6, dtype='float32').reshape(E, 6), 'b': np.arange(E, dtype='float64')}
    dump_outputs(tmp_path / 'full', arrays)
    for k, v in arrays.items():
        assert np.array_equal(np.load(tmp_path / 'full' / f'{k}.npy'), v)
    dump_outputs(tmp_path / 'cut', arrays, budget=100 * 32)            # 32 bytes per env: 100 envs fit
    a, b = np.load(tmp_path / 'cut' / 'a.npy'), np.load(tmp_path / 'cut' / 'b.npy')
    assert a.shape == (100, 6) and a.dtype == np.float32 and b.dtype == np.float64
    assert np.array_equal(a[:, 0] / 6, b) and np.all(np.diff(b) > 0)
    dump_outputs(tmp_path / 'again', arrays, budget=100 * 32)
    assert np.array_equal(np.load(tmp_path / 'again' / 'b.npy'), b)


@pytest.mark.gpu
def test_b200_arm_times_exactly_the_requested_steps_and_dumps_them(tmp_path):
    """Two runs with the same arguments dump the same last-step outputs of the one timed K-step launch."""
    import numpy as np
    E, K = 64, 7
    flags = ['--steps', str(K), '--warmup', '3', '--envs', str(E), '--extras', 'none', '--no-cpu-baseline']
    dumps = []
    for i in range(2):
        r = run(*flags, '--dump-outputs', str(tmp_path / str(i)))
        assert r.returncode == 0, r.stderr[-400:]
        j = json.loads([ln for ln in r.stdout.splitlines() if ln.strip().startswith('{')][0])
        assert j['steps'] == K and j['gpu_launches'] == 1 and j['roofline']['steps_per_launch'] == K
        dumps.append({n: np.load(tmp_path / str(i) / f'{n}.npy') for n in ('observations', 'rewards', 'district')})
    obs, rew, dst = dumps[0]['observations'], dumps[0]['rewards'], dumps[0]['district']
    assert obs.dtype == rew.dtype == dst.dtype == np.float32
    assert obs.shape == (E, 476) and rew.shape == (E, 17) and dst.shape == (E, 3)
    assert np.isfinite(rew).all() and np.isfinite(dst).all()
    for n in dumps[0]:
        assert np.array_equal(dumps[0][n], dumps[1][n], equal_nan=True), n
