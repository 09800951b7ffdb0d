"""bench.py keeps the driver's contract: one JSON line with the required keys, for both arms."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import conftest as cf

BENCH = os.path.join(cf.ROOT, 'bench.py')
COMMON = ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
          'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e', 'gpu_launches')


def _run(args, env=None):
  proc = subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, timeout=900,
                        env=dict(os.environ, **(env or {})))
  assert proc.returncode == 0, proc.stderr[-2000:]
  lines = [l for l in proc.stdout.strip().splitlines() if l.startswith('{')]
  assert len(lines) == 1, proc.stdout
  return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
  line = _run(['--impl', 'reference', '--steps', '3', '--warmup', '3'], env={'BSB_BENCH_BUDGET_S': '0.5'})
  for key in COMMON:
    assert key in line, key
  assert line['impl'] == 'reference' and line['metric'] == 'env-steps/sec' and line['higher_is_better'] is True
  assert line['value'] > 0 and line['vs_baseline'] is None and line['gpu_launches'] == 0
  assert line['cpu_baseline']['kind'] in ('reference', 'port') and line['cpu_baseline']['cores'] >= 1
  assert line['cpu_baseline']['value'] == line['value'] == line['e2e']['value']
  assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
  assert 'workload' in line['config']


def test_reference_arm_is_silent_on_other_ranks():
  proc = subprocess.run([sys.executable, BENCH, '--impl', 'reference', '--gpus', '2', '--steps', '3', '--warmup', '3'],
                        capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK='1', WORLD_SIZE='2'))
  assert proc.returncode == 0 and proc.stdout.strip() == ''


@pytest.mark.gpu
def test_engine_arm_prints_the_contract_line(tmp_path):
  line = _run(['--steps', '40', '--warmup', '3', '--skip-cpu-baseline', '--skip-host-obs', '--skip-fused', '--skip-traffic',
               '--legs', 'catch_131072', '--dump-outputs', str(tmp_path)])
  dumped = {name: np.load(tmp_path / name) for name in os.listdir(tmp_path)}
  assert set(dumped) == {'observation_sample.npy', 'reward.npy', 'discount.npy', 'step_type.npy', 'log_point.npy'}
  assert all(a.dtype in (np.float32, np.float64) for a in dumped.values())
  assert sum(a.nbytes for a in dumped.values()) <= 64 << 20
  assert dumped['reward.npy'].shape == (65536,) and dumped['observation_sample.npy'].shape[1:] == (32, 32)
  for key in COMMON + ('roofline', 'clocks'):
    assert key in line, key
  assert line['n_gpus'] == 1 and line['steps'] == 40 and line['scaling'] == 'weak' and line['data'] == 'synthetic'
  assert line['gpu_launches'] >= 40 and line['value'] > 1e8
  roof = line['roofline']
  assert roof['bound'] == 'hbm' and roof['unit'] == 'GB/s' and abs(roof['frac'] - roof['achieved'] / roof['peak']) < 1e-9
  assert line['e2e']['h2d_bytes_per_step'] == 4 * 65536 and line['e2e']['d2h_bytes_per_step'] == 12 * 65536
  assert line['e2e']['value'] > 0 and line['e2e']['value'] != line['value']
  assert len(line['windows_ms']) == 5 and roof['frac_from_ms_per_step'] <= roof['frac'] + 1e-9
  leg = line['configs']['catch_131072']
  assert leg['parity_sampled'] is True and leg['global_lanes'] == 131072 and leg['step_us'] > 0 and leg['rollout_us'] > 0
