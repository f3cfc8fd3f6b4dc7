"""
CPU check of bench.py's reference arm (the driver runs `bench.py --impl reference` beside the GPU arm): exactly one
JSON line on stdout with the contract's keys, the same metric / unit / config as the GPU arm would print, and a
cpu_baseline block describing the run.  Small sizes so it takes seconds; the GPU arm itself needs the B200.
"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_reference(extra_env=None):
  env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
  env.update(extra_env or {})
  out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '1', '--n-train', '300', '--cpu-sample', '2000', '--gpus', '1'],
                       capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
  assert out.returncode == 0, out.stderr
  lines = [l for l in out.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, out.stdout
  return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
  line = run_reference()
  assert line['impl'] == 'reference' and line['higher_is_better'] is True and line['scaling'] == 'weak'
  assert line['metric'].startswith('posterior+acq candidates/sec') and line['unit'] == 'candidates/s'
  assert line['dtype'] == 'f64' and line['data'] == 'synthetic' and line['vs_baseline'] is None
  assert line['steps'] == 1 and line['warmup'] == 1 and line['n_gpus'] == 1 and line['gpu_launches'] == 0
  cb = line['cpu_baseline']
  assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == line['value'] and '2000 candidates' in cb['sample']
  # a step = posterior build + scoring of the bounded sample; value projects both measured parts to the full step
  assert line['value'] > 0 and cb['posterior_build_s'] > 0 and cb['scoring_only_value'] >= line['value']
  full_m = line['config']['candidates_per_gpu']
  want = full_m / (cb['posterior_build_s'] + full_m / cb['scoring_only_value'])
  assert abs(want - line['value']) <= 1e-9 * want
  assert line['e2e'] == {'value': line['value'], 'unit': 'candidates/s', 'h2d_bytes_per_step': 0,
                         'd2h_bytes_per_step': 0}
  cfg = line['config']
  assert 'workload' in cfg and cfg['n_train'] == 300 and cfg['kernel'] == 'matern-2.5' and cfg['acquisition'] == 'ei'
  assert 'model' not in cfg


def test_reference_arm_other_ranks_print_nothing():
  """ Under torchrun only rank 0 runs the CPU arm; the other ranks exit 0 without output. """
  env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1', PYTHONDONTWRITEBYTECODE='1')
  out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                        '--steps', '1', '--warmup', '1'], capture_output=True, text=True, env=env, timeout=300,
                       cwd=ROOT)
  assert out.returncode == 0 and out.stdout.strip() == ''


def test_reference_arm_of_every_config():
  """ `bench.py --impl reference --config c2..c5`: one JSON line each, strong-scaling label, a port-kind cpu_baseline. """
  import pytest
  for cfg in ('c2', 'c3', 'c4', 'c5'):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--config', cfg, '--steps', '1',
                          '--warmup', '0', '--n-train', '200', '--cpu-sample', '700', '--gpus', '1'],
                         capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 0, (cfg, out.stderr[-2000:])
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, (cfg, out.stdout)
    line = json.loads(lines[0])
    assert line['impl'] == 'reference' and line['scaling'] == 'strong' and line['value'] > 0, cfg
    assert line['config']['n_train'] == 200 and 'workload' in line['config'] and 'model' not in line['config']
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['value'] == line['value']
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['gpu_launches'] == 0


@pytest.mark.gpu
def test_dump_outputs_repeat_under_the_same_arguments(tmp_path):
  """ `bench.py --dump-outputs DIR` on the GPU arm, twice with the same arguments: float64 .npy files of the last timed
      step of every leg, the same values both times, and --steps timed steps in every leg. """
  import numpy as np
  dumps = []
  for run in ('a', 'b'):
    out_dir = str(tmp_path / run)
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '3', '--warmup', '1',
                          '--n-train', '1100', '--cands-per-gpu', '30000', '--no-extras', '--no-cpu-baseline',
                          '--dump-outputs', out_dir],
                         capture_output=True, text=True, env=dict(os.environ, PYTHONDONTWRITEBYTECODE='1'), timeout=900,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    assert line['steps'] == 3 and len(line['step_ms_each']['device']) == 3 and len(line['step_ms_each']['e2e']) == 3
    dumps.append(dict((f[:-4], np.load(os.path.join(out_dir, f))) for f in sorted(os.listdir(out_dir))))
  a, b = dumps
  assert sorted(a) == sorted(b) == sorted(
      ['device_best_score', 'device_best_index', 'e2e_point', 'e2e_device_candidates_point', 'posterior_lml',
       'posterior_alpha', 'posterior_L_sample'])
  assert a['posterior_alpha'].shape == (1100,) and a['e2e_point'].shape == (6,)
  for name in a:
    assert a[name].dtype == np.float64, name
    np.testing.assert_allclose(a[name], b[name], rtol=1e-12, atol=0, err_msg=name)
