"""Cost of stochastic reconfiguration at C2 (6x6 Heisenberg, rbm H = 144, 8192
walkers, 20 batches per epoch = 163,840 stored walkers) next to the
EnergyGradient epoch, and the energy trajectories of both optimizers over the
same number of epochs from the same seeded start.

Reports, with CUDA events on the launching stream and the card's name and
power limit read in the same run:
  - one cgsvmc_log_amp_jvp launch over all stored walkers,
  - one S v (training.sr_matvec: JVP + weighted gradient sum + vector ops),
  - the conjugate-gradient solve of one epoch (iterations, residual, time),
  - the wall time of a whole epoch (run_optimization_epoch returns a host
    float, so each epoch ends synchronised) for SR and for EnergyGradient.
The stored walkers (1.3 MB) and parameters stay in L2 across repetitions: the
figures are for the warm working set a training run sees.

  python profiles/run_sr_epoch.py [--epochs 30] [--out profiles/sr_epoch_c2.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from cgs_vmc_b200 import graph_builders, lattices, operators, training, utils, wavefunctions  # noqa: E402
from cgs_vmc_b200.session import Session  # noqa: E402


def card():
  out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
  name, _, limit = out.stdout.strip().partition(',')
  return {'name': name.strip() or torch.cuda.get_device_name(0), 'power_limit': limit.strip()}


def build(optimizer_name, hp, seed):
  graph_builders.reset_num_epochs()
  wf = wavefunctions.build_wavefunction(hp).seed(seed)
  ham = operators.HeisenbergHamiltonian(lattices.square_nn_bonds(6), -1.0, 1.0)
  opt = training.ground_state_optimizer(optimizer_name)()
  ops = opt.build_opt_ops(wavefunction=wf, hamiltonian=ham, hparams=hp, shared_resources={})
  return wf, opt, ops


def event_ms(fn, reps):
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  fn()
  torch.cuda.synchronize()
  a.record()
  for _ in range(reps):
    fn()
  b.record()
  b.synchronize()
  return a.elapsed_time(b) / reps


def trajectory(optimizer_name, hp, epochs, seed):
  wf, opt, ops = build(optimizer_name, hp, seed)
  s = Session()
  energies, wall = [], []
  for _ in range(epochs):
    t0 = time.perf_counter()
    energies.append(opt.run_optimization_epoch(ops, s, hp))
    wall.append(time.perf_counter() - t0)
  return opt, ops, energies, wall


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--epochs', type=int, default=30)
  ap.add_argument('--sr-lr', type=float, default=0.05)
  ap.add_argument('--sr-shift', type=float, default=0.01)
  ap.add_argument('--adam-lr', type=float, default=0.01)
  ap.add_argument('--out', default='')
  args = ap.parse_args()
  common = dict(wavefunction_type='rbm', num_sites=36, size_x=6, size_y=6, num_fc_layers=0, fc_layer_size=144,
                batch_size=8192, num_batches_per_epoch=20, num_equilibration_sweeps=5)
  hp_sr = utils.create_hparams(optimizer='gradient', learning_rates=[args.sr_lr] * 4, sr_diag_shift=args.sr_shift,
                               **common)
  hp_eg = utils.create_hparams(optimizer='adam', learning_rates=[args.adam_lr] * 4, **common)
  result = {'workload': 'C2: 6x6 Heisenberg (72 NN bonds, jx=-1, jz=1), rbm H=144, 8192 walkers, '
                        '20 batches per epoch, 5 equilibration sweeps per epoch',
            'card': card(), 'epochs': args.epochs,
            'sr': {'optimizer': 'gradient', 'lr': args.sr_lr, 'sr_diag_shift': args.sr_shift,
                   'sr_cg_tolerance': hp_sr.sr_cg_tolerance, 'sr_cg_max_iterations': hp_sr.sr_cg_max_iterations},
            'energy_gradient': {'optimizer': 'adam', 'lr': args.adam_lr}}

  # trajectories (the first epochs also capture the graphs)
  opt, ops, e_sr, wall_sr = trajectory('StochasticReconfiguration', hp_sr, args.epochs, seed=2)
  _, _, e_eg, wall_eg = trajectory('EnergyGradient', hp_eg, args.epochs, seed=2)
  result['sr']['energies'] = e_sr
  result['energy_gradient']['energies'] = e_eg
  skip = min(3, args.epochs - 1)      # graph capture and first-launch set-up
  result['sr']['epoch_ms_median'] = 1e3 * float(np.median(wall_sr[skip:]))
  result['energy_gradient']['epoch_ms_median'] = 1e3 * float(np.median(wall_eg[skip:]))

  # the pieces of one SR update, on a filled sample store
  s = Session()
  s.run(ops.mc_step, n_steps=hp_sr.num_equilibration_sweeps * hp_sr.num_sites)
  s.run(ops.reset_gradients)
  for _ in range(hp_sr.num_batches_per_epoch):
    s.run(opt._batch_step)
  packed = opt.stored_configs()
  ansatz = opt.sums.ansatz
  m = packed.shape[0]
  v = torch.randn(ansatz.num_params, dtype=torch.float64, generator=torch.Generator().manual_seed(0)).cuda()
  v32 = v.float()
  o_mean = opt.sums.sums[0].double() / m
  result['stored_walkers'] = m
  result['jvp_ms'] = event_ms(lambda: ansatz.log_amp_jvp(packed, v32), 50)
  result['jvp_gflop'] = 2.0 * 36 * 144 * m / 1e9
  result['matvec_ms'] = event_ms(lambda: training.sr_matvec(ansatz, packed, o_mean, v, float(m), args.sr_shift), 20)
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  s.run(ops.apply_gradients)
  b.record()
  b.synchronize()
  result['solve_ms'] = a.elapsed_time(b)
  result['cg_iterations'] = opt.cg_iterations
  result['cg_residual'] = opt.cg_residual
  s.run(ops.reset_gradients)
  line = json.dumps(result)
  print(line)
  if args.out:
    with open(args.out, 'w') as f:
      f.write(line + '\n')


if __name__ == '__main__':
  main()
