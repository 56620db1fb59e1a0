#!/usr/bin/env python
"""Where a conv_tc forward spends its cycles: MMA phase (issue -> commit
barrier) against epilogue, per tensor layer, from the counters of the timing
build (`python __graft_entry__.py --timing` -> libcgsvmc_timing.so).

  CGSVMC_LIBRARY=cgs_vmc_b200/libcgsvmc_timing.so python profiles/run_conv_tc_phases.py
"""
import argparse
import ctypes
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--walkers', type=int, default=8192)
  args = ap.parse_args()
  os.environ.setdefault('CGSVMC_LIBRARY', os.path.join(REPO, 'cgs_vmc_b200', 'libcgsvmc_timing.so'))
  import numpy as np
  import torch
  from cgs_vmc_b200 import _native, engine, lattices
  lib = _native.load()
  a = _native.Ansatz('conv_2d', 100, num_layers=5, num_filters=16, kernel_size=5, size_x=10, size_y=10)
  gen = torch.Generator().manual_seed(1234)
  a.set_params(torch.randn(a.num_params, generator=gen) * 0.05)
  ij, jx, jz = lattices.j1j2_couplings(10, 0.5)
  ham = _native.Hamiltonian(ij, jx, jz, 100)
  state = engine.WalkerState(args.walkers, 100, seed=0xC65)
  out = (ctypes.c_ulonglong * 4)()

  def measure(name, fn):
    fn()
    lib.cgsvmc_debug_conv_tc_phases(out)          # clear
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    lib.cgsvmc_debug_conv_tc_phases(out)
    mma, epi, layers, fwd = [int(v) for v in out]
    print(json.dumps({'kernel': name, 'ms': e0.elapsed_time(e1),
                      'tensor_layers': layers, 'forwards': fwd,
                      'mma_phase_cycles_per_layer': mma / max(1, layers),
                      'epilogue_cycles_per_layer': epi / max(1, layers),
                      'mma_share': mma / max(1, mma + epi)}))

  measure('tc_mc_kernel (20 steps)', lambda: state.mc_steps(a, 20))
  measure('tc_eloc_kernel', lambda: a.local_energy(ham, state.packed))


if __name__ == '__main__':
  main()
