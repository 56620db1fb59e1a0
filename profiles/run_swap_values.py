"""Replica-swap values of the second Renyi entropy: the fused pure-RBM kernel
(cgsvmc_swap_values) against the amplitude route (cgsvmc_swap_configs +
cgsvmc_log_amp of every swapped configuration + cgsvmc_swap_values_from_amps,
in pair chunks of at most 2^25 swapped configurations like
operators.RenyiSwap).

Workloads (the prefix regions of lattices.prefix_regions, walkers after 2
sweeps from random Sz = 0 configurations, paired row p with row P + p):
  C2: 6x6, rbm H = 144, 8,192 walkers (4,096 pairs), 18 regions;
  C5: 16x16, rbm H = 256, 131,072 walkers (65,536 pairs), 128 regions.
Reports per route the time of one call (CUDA events over `reps` calls after a
warm-up call), the pair-regions per second, and the largest difference
between the routes relative to the amplitude route's value (+ 1e-3).  The
card's name and power limit are read in the same run.  Inputs are not flushed
from L2 between calls (the C5 swapped configurations of the amplitude route
are 537 MB; everything else fits the 126 MB L2).

  python profiles/run_swap_values.py [--out profiles/swap_values.json]
"""
import argparse
import json
import os
import subprocess
import sys

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


def amplitude_route(ansatz, packed, n, masks, out):
  p, r = packed.shape[0] // 2, masks.shape[0]
  chunk = max(1, operators._BOND_VALUES_CHUNK // (2 * r))
  for c0 in range(0, p, chunk):
    c1 = min(p, c0 + chunk)
    pc = packed if c1 - c0 == p else torch.cat([packed[c0:c1], packed[p + c0:p + c1]])
    z = ansatz.log_amp(pc)
    swapped = _native.swap_configs(pc, n, masks)
    sl = ansatz.log_amp(swapped.reshape((c1 - c0) * r * 2, -1)).reshape(c1 - c0, r, 2)
    _native.swap_values_from_amps(pc, n, masks, z, None, sl, None, out=out[c0:c1])
  return out


def workload(name, side, hidden, walkers, reps):
  n = side * side
  hp = utils.create_hparams(wavefunction_type='rbm', num_sites=n, num_fc_layers=0, fc_layer_size=hidden)
  ansatz = wavefunctions.build_wavefunction(hp).seed(1).native(n)
  packed = _native.random_configs(walkers, n, seed=7)
  ansatz.mc_steps(packed, 2 * n, seed=11)
  regions = lattices.prefix_regions(n)
  masks = operators.RenyiSwap(regions).masks(packed.device)
  p, r = walkers // 2, len(regions)
  fused_out = torch.empty(p, r, dtype=torch.float32, device='cuda')
  amp_out = torch.empty_like(fused_out)
  fused_ms = event_ms(lambda: ansatz.swap_values(packed, masks, out=fused_out), reps)
  amp_ms = event_ms(lambda: amplitude_route(ansatz, packed, n, masks, amp_out), max(1, reps // 5))
  computed = int(((amp_out != 0) & (amp_out != 1)).sum())
  diff = float(((fused_out - amp_out).abs() / (amp_out.abs() + 1e-3)).max())
  pair_regions = p * r
  return {'workload': name, 'n_sites': n, 'hidden': hidden, 'walkers': walkers, 'pairs': p, 'regions': r,
          'ratio_evaluations': computed,
          'fused': {'ms': fused_ms, 'pair_regions_per_s': pair_regions / fused_ms * 1e3},
          'amplitude_route': {'ms': amp_ms, 'pair_regions_per_s': pair_regions / amp_ms * 1e3},
          'speedup': amp_ms / fused_ms, 'max_rel_diff': diff}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', default='')
  args = ap.parse_args()
  _native.require_cuda()
  rows = [workload('C2', 6, 144, 8192, 2000),
          workload('C5', 16, 256, 131072, 50)]
  result = {'card': card(), 'rows': rows}
  line = json.dumps(result)
  print(line)
  if args.out:
    with open(args.out, 'w') as f:
      f.write(line + '\n')


if __name__ == '__main__':
  main()
