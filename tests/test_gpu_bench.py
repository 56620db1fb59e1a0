"""-m gpu checks of bench.py --dump-outputs: the files, their types and size,
that equal arguments give equal outputs, and that --steps sets the number of
timed batch iterations (visible in the walker count of the last epoch)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WALKERS, N_SITES = 1024, 36


def _bench(out_dir, steps):
  env = dict(os.environ, PYTHONPATH=REPO)
  out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--steps', str(steps), '--warmup', '0',
                        '--walkers', str(WALKERS), '--configs', '', '--no-cpu-baseline',
                        '--dump-outputs', str(out_dir)],
                       capture_output=True, text=True, timeout=900, env=env)
  assert out.returncode == 0, out.stderr[-2000:]
  lines = [l for l in out.stdout.splitlines() if l.strip()]
  assert len(lines) == 1
  arrays = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}
  return json.loads(lines[0]), arrays


@pytest.mark.gpu
def test_dump_outputs_repeatable_and_steps_honoured(tmp_path):
  line, a = _bench(tmp_path / 'a', 3)
  _, b = _bench(tmp_path / 'b', 3)
  assert line['steps'] == 3
  assert sorted(a) == ['accepted_moves', 'configs', 'energy_stats', 'epoch_energies', 'params']
  assert all(x.dtype in (np.float32, np.float64) for x in a.values())
  assert sum(x.nbytes for x in a.values()) <= 64 << 20
  assert a['configs'].shape == (WALKERS, N_SITES) and set(np.unique(a['configs'])) == {-1.0, 1.0}
  assert np.all(a['configs'].sum(axis=1) == 0)                        # Sz = 0 is kept by exchange moves
  assert a['epoch_energies'].shape == (1,) and np.all(np.isfinite(a['params']))
  assert a['energy_stats'][2] == 3 * WALKERS                          # the timed epoch ran 3 batch iterations
  np.testing.assert_allclose(a['epoch_energies'][-1], a['energy_stats'][0] / a['energy_stats'][2], rtol=1e-12)
  for name in a:
    np.testing.assert_array_equal(a[name], b[name], err_msg=name)

  line, c = _bench(tmp_path / 'c', 60)                                 # one epoch of 50 and one of 10
  assert line['steps'] == 60
  assert c['epoch_energies'].shape == (2,) and c['energy_stats'][2] == 10 * WALKERS
