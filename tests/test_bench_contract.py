"""bench.py contract checks that need no GPU: the reference arm (CPU port of
the reference's op sequence) runs, prints exactly one JSON line on stdout with
the keys the driver reads, and a non-zero rank under torchrun prints nothing."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
  env = dict(os.environ, PYTHONPATH=REPO)
  env.update(env_extra or {})
  return subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--impl', 'reference',
                         '--steps', '1', '--warmup', '0', '--walkers', '64'],
                        capture_output=True, text=True, timeout=600, env=env)


def test_reference_arm_prints_one_json_line():
  out = _run()
  assert out.returncode == 0, out.stderr[-2000:]
  lines = [l for l in out.stdout.splitlines() if l.strip()]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d['impl'] == 'reference' and d['metric'] == 'walker_steps_per_sec'
  assert d['unit'] == 'walker-steps/s' and d['higher_is_better'] is True
  assert d['value'] > 0 and d['ms_per_step'] > 0 and d['vs_baseline'] is None
  assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
  assert d['cpu_baseline']['value'] == d['value'] and 'sample' in d['cpu_baseline']
  assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0,
                      'd2h_bytes_per_step': 0}
  assert 'workload' in d['config'] and 'C2' in d['config']['workload']


def test_reference_arm_other_ranks_do_nothing():
  out = _run({'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
  assert out.returncode == 0 and out.stdout.strip() == ''


def test_bad_arguments_are_refused():
  env = dict(os.environ, PYTHONPATH=REPO)
  for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']):
    out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py')] + extra,
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 2 and out.stdout.strip() == '', extra
