"""Diagnostic: precision of the tensor-core gradient sums (rbm2 pair-table kernel,
conv_tc_grad.cu) against the FP32 register-tile kernels and the float64 oracle,
per parameter tensor."""
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))
from cgs_vmc_b200 import _native, engine  # noqa: E402
from oracle import ansatz as oansatz  # noqa: E402
from oracle import bits, estimators, lattices  # noqa: E402
from gpu_util import make_native, packed_cuda  # noqa: E402

F64 = torch.float64


def blocks(spec):
  out, off = [], 0
  for name, shape in oansatz.param_shapes(spec):
    n = int(np.prod(shape))
    out.append((name, off, off + n))
    off += n
  return out


def report(tag, got, ref, spec):
  for k in range(got.shape[0]):
    for name, a, b in blocks(spec):
      d = got[k, a:b] - ref[k, a:b]
      print('%-34s k=%d %-12s |ref| max %.3e  norm %.3e   err max %.3e  norm-rel %.3e' % (
          tag, k, name, np.abs(ref[k, a:b]).max(), np.linalg.norm(ref[k, a:b]), np.abs(d).max(),
          np.linalg.norm(d) / (np.linalg.norm(ref[k, a:b]) + 1e-30)))
    d = got[k] - ref[k]
    print('%-34s k=%d %-12s norm-rel %.3e' % (tag, k, 'ALL', np.linalg.norm(d) / np.linalg.norm(ref[k])))


def rbm():
  spec = oansatz.AnsatzSpec('rbm', 36, num_layers=0, layer_size=144, size_x=6, size_y=6)
  params = oansatz.init_params(spec, seed=1234, bias_scale=0.1, dtype=F64)
  a = make_native(spec, oansatz.flatten(params).numpy())
  ij, jx, jz = lattices.heisenberg_couplings(lattices.square_nn_bonds(6))
  ham = _native.Hamiltonian(ij, jx, jz, 36)
  for B, iters in ((256, 1), (8192, 1), (8192, 2), (8192, 5), (8192, 50)):
    res = {}
    for flag in ('1', '0'):
      os.environ['CGSVMC_RBM2_TC_GRAD'] = flag
      st = engine.WalkerState(B, 36, seed=9)
      sums = engine.EnergyGradientSums(a, B)
      e_all = torch.empty(iters, B, dtype=torch.float32, device='cuda')
      cfgs = []
      for i in range(iters):
        cfgs.append(st.packed.clone())
        sums.batch_steps(ham, st, 36, 1, e_loc_out=e_all[i:i + 1]) if False else None
        if iters == 1:
          e_all[0] = sums.batch_step(ham, st, 36)
      if iters > 1:
        st = engine.WalkerState(B, 36, seed=9)
        sums = engine.EnergyGradientSums(a, B)
        sums.batch_steps(ham, st, 36, iters, e_loc_out=e_all)
      res[flag] = (sums.sums.cpu().numpy().astype(np.float64), e_all.double().cpu())
    os.environ.pop('CGSVMC_RBM2_TC_GRAD')
    print('--- rbm C2, B = %d, %d iteration(s): tensor cores vs register tiles' % (B, iters))
    report('rbm tc vs simt', res['1'][0], res['0'][0], spec)
    print('e_loc equal:', bool(torch.equal(res['1'][1], res['0'][1])), ' mean E', float(res['0'][1].mean()))
    if iters == 1:
      # float64 reference of the same sums
      st = engine.WalkerState(B, 36, seed=9)
      cfg = bits.unpack(st.packed.cpu().numpy().view(np.uint64), 36)
      w = torch.stack([torch.ones(B, dtype=F64), res['0'][1][0]])
      ref = estimators.weighted_grad_sum(spec, params, torch.from_numpy(cfg).to(F64), w).numpy()
      report('rbm tc vs float64', res['1'][0], ref, spec)
      report('rbm simt vs float64', res['0'][0], ref, spec)


def conv():
  spec = oansatz.AnsatzSpec('conv_2d', 100, num_layers=5, num_filters=16, kernel_size=5, size_x=10, size_y=10)
  batch = 70
  params = oansatz.init_params(spec, seed=17, bias_scale=0.1, dtype=F64)
  cfg = bits.random_sz0_configs(spec.n_sites, batch, np.random.default_rng(17))
  a = make_native(spec, oansatz.flatten(params).numpy())
  rng = np.random.default_rng(3)
  w = rng.normal(size=(2, batch)).astype(np.float32)
  w[0] = 1.0
  ref = estimators.weighted_grad_sum(spec, params, torch.from_numpy(cfg).to(F64), torch.from_numpy(w).to(F64)).numpy()
  for flag, tag in (('1', 'conv tc vs float64'), ('0', 'conv simt vs float64')):
    os.environ['CGSVMC_CONV_TC_GRAD'] = flag
    out = a.weighted_grad_sum(packed_cuda(cfg), torch.from_numpy(w).cuda()).cpu().numpy().astype(np.float64)
    print('--- ' + tag)
    report(tag, out, ref, spec)
  os.environ.pop('CGSVMC_CONV_TC_GRAD')


if __name__ == '__main__':
  rbm()
  if '--conv' in sys.argv:
    conv()
