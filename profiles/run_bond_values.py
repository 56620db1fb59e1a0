"""Per-bond local values (spin-spin correlations): the fused pure-RBM kernel
(cgsvmc_bond_values) against the amplitude route (cgsvmc_flip_enum +
cgsvmc_log_amp of every flipped configuration + cgsvmc_bond_values_from_amps,
in walker chunks of at most 2^25 values like operators.HeisenbergBonds).

Workloads (Heisenberg couplings jx = -1 on NN bonds, Marshall-signed jx on all
pairs, jz = 1; walkers after 2 sweeps from random Sz = 0 configurations):
  C2: 6x6, rbm H = 144, 8,192 walkers, the 72 NN bonds and all 630 pairs;
  C5: 16x16, rbm H = 256, the 512 NN bonds at 131,072 walkers and all
      32,640 pairs at 8,192 walkers.
Reports per route the time of one call (CUDA events over `reps` calls after a
warm-up call), the bond values and ratio evaluations (antiparallel bonds with
jx != 0, the ones that need psi(flip) / psi) per second, and the largest
difference between the routes.  The card's name and power limit are read in
the same run.  Inputs are not flushed from L2 between calls (the 16x16
all-pairs output alone is 1 GB; the others fit the 126 MB L2).

  python profiles/run_bond_values.py [--out profiles/bond_values.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from cgs_vmc_b200 import _native, lattices, operators, utils, wavefunctions  # noqa: E402


def card():
  out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
  name, _, limit = out.stdout.strip().partition(',')
  return {'name': name.strip() or torch.cuda.get_device_name(0), 'power_limit': limit.strip()}


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


def amplitude_route(ansatz, ham, packed, out):
  b, k = packed.shape[0], ham.n_bonds
  chunk = max(1, operators._BOND_VALUES_CHUNK // k)
  for c0 in range(0, b, chunk):
    pc = packed[c0:c0 + chunk]
    bc = pc.shape[0]
    z = ansatz.log_amp(pc)
    _, flipped = ham.flip_enum(pc)
    fl = ansatz.log_amp(flipped.reshape(bc * k, -1)).reshape(bc, k)
    _native.bond_values_from_amps(ham, pc, z, None, fl, None, out=out[c0:c0 + chunk])
  return out


def ratio_count(packed, n_sites, ij, jx):
  cfg = _native.unpack_configs(packed, n_sites)
  ij_t = torch.from_numpy(ij.astype(np.int64)).cuda()
  live = torch.from_numpy(jx != 0).cuda()
  total = 0
  for k0 in range(0, len(ij), 4096):
    i, j = ij_t[k0:k0 + 4096, 0], ij_t[k0:k0 + 4096, 1]
    total += int(((cfg[:, i] != cfg[:, j]) & live[k0:k0 + 4096]).sum())
  return total


def workload(name, side, hidden, walkers, bonds_kind, reps):
  n = side * side
  hp = utils.create_hparams(wavefunction_type='rbm', num_sites=n, num_fc_layers=0, fc_layer_size=hidden)
  ansatz = wavefunctions.build_wavefunction(hp).seed(1).native(n)
  packed = _native.random_configs(walkers, n, seed=7)
  ansatz.mc_steps(packed, 2 * n, seed=11)
  if bonds_kind == 'nn':
    ij = np.asarray(lattices.square_nn_bonds(side), np.int32)
    jx = np.full(len(ij), -1.0, np.float32)
  else:
    ij = np.asarray(lattices.all_pairs(n), np.int32)
    signs = lattices.marshall_signs(n, lattices.square_nn_bonds(side), -1.0, 1.0)
    jx = (signs[ij[:, 0]] * signs[ij[:, 1]]).astype(np.float32)
  ham = _native.Hamiltonian(ij, jx, 1.0, n)
  fused_out = torch.empty(walkers, len(ij), dtype=torch.float32, device='cuda')
  amp_out = torch.empty_like(fused_out)
  fused_ms = event_ms(lambda: ansatz.bond_values(ham, packed, out=fused_out), reps)
  amp_ms = event_ms(lambda: amplitude_route(ansatz, ham, packed, amp_out), max(1, reps // 5))
  ratios = ratio_count(packed, n, ij, jx)
  values = walkers * len(ij)
  diff = float(((fused_out - amp_out).abs() / (amp_out.abs() + 0.25)).max())
  return {'workload': name, 'n_sites': n, 'hidden': hidden, 'walkers': walkers, 'bonds': len(ij),
          'ratio_evaluations': ratios,
          'fused': {'ms': fused_ms, 'values_per_s': values / fused_ms * 1e3,
                    'ratio_evaluations_per_s': ratios / fused_ms * 1e3},
          'amplitude_route': {'ms': amp_ms, 'values_per_s': values / amp_ms * 1e3,
                              'ratio_evaluations_per_s': ratios / amp_ms * 1e3},
          'speedup': amp_ms / fused_ms, 'max_rel_diff': diff}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', default='')
  args = ap.parse_args()
  _native.require_cuda()
  rows = [workload('C2 NN', 6, 144, 8192, 'nn', 50),
          workload('C2 all pairs', 6, 144, 8192, 'all', 20),
          workload('C5 NN', 16, 256, 131072, 'nn', 10),
          workload('C5 all pairs', 16, 256, 8192, 'all', 5)]
  result = {'card': card(), 'rows': rows}
  line = json.dumps(result)
  print(line)
  if args.out:
    with open(args.out, 'w') as f:
      f.write(line + '\n')


if __name__ == '__main__':
  main()
