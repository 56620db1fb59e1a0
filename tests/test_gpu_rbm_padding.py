"""-m gpu: the pure-RBM kernels pad H up to a multiple of 32 with units of
W = 0 and c = 0, so an RBM with H = 144 must sample, evaluate and differentiate
exactly like an RBM with H = 160 whose 16 extra units have W = 0 and c = 0.
The two take different paths through the epoch kernel: H = 144 sums its
gradient on the tensor cores and re-parks the 2W rows in shared memory every
iteration (behind an mbarrier, with the empty walker slots zeroed again), while
H = 160 has no spare column for the tensor-core path and uses the FP32 register
tiles with the 2W rows read from global memory.  Run at several walker counts:
one batch per CTA, a ragged last batch, several batches per CTA."""
import numpy as np
import pytest
import torch

from oracle import ansatz as oansatz
from oracle import lattices

pytestmark = pytest.mark.gpu

N_SIDE, N, H, HP = 6, 36, 144, 160


@pytest.fixture(scope='module')
def native():
  from cgs_vmc_b200 import _native
  _native.load()
  return _native


@pytest.fixture(scope='module')
def rbm_pair(native):
  """(H = 144 RBM, H = 160 RBM with 16 zero units) with the same real parameters."""
  from gpu_util import make_native
  spec = oansatz.AnsatzSpec('rbm', N, num_layers=0, layer_size=H, size_x=N_SIDE, size_y=N_SIDE)
  spec_p = oansatz.AnsatzSpec('rbm', N, num_layers=0, layer_size=HP, size_x=N_SIDE, size_y=N_SIDE)
  a, a0, w, c = oansatz.init_params(spec, seed=11, bias_scale=0.1, dtype=torch.float64)
  w_p = torch.cat([w, torch.zeros(N, HP - H, dtype=w.dtype)], dim=1)
  c_p = torch.cat([c, torch.zeros(HP - H, dtype=c.dtype)])
  return (make_native(spec, oansatz.flatten([a, a0, w, c]).numpy()),
          make_native(spec_p, oansatz.flatten([a, a0, w_p, c_p]).numpy()))


def _run(native, ansatz, ham, batch, n_batches):
  from cgs_vmc_b200 import engine
  st = engine.WalkerState(batch, N, seed=9, walker_id0=3)
  sums = torch.zeros(2, ansatz.num_params, dtype=torch.float32, device='cuda')
  stats = torch.zeros(4, dtype=torch.float64, device='cuda')
  e_loc = torch.empty(n_batches, batch, dtype=torch.float32, device='cuda')
  log_amp = torch.empty(n_batches, batch, dtype=torch.float32, device='cuda')
  ansatz.batch_steps(ham, st.packed, n_batches, sums, stats, N, st.seed, st.walker_id0,
                     accept_count=st.accept_count, e_loc_out=e_loc, log_amp_out=log_amp)
  return e_loc, log_amp, st.packed, st.accept_count, sums, stats


def _split(sums, h):
  """[2, P] sums -> (a and a0 columns, W [2, N, h], c [2, h])."""
  s = sums.cpu().numpy()
  return s[:, :N + 1], s[:, N + 1:N + 1 + N * h].reshape(2, N, h), s[:, N + 1 + N * h:]


# 8192: C2, one batch per CTA, the walkers stay in registers across iterations;
# 8190: a ragged last batch; 20000: more batches than CTAs (walkers read back)
@pytest.mark.parametrize('batch', [8192, 8190, 20000])
def test_padded_units_are_neutral(native, rbm_pair, batch):
  """20 iterations of cgsvmc_batch_steps at C2 (6x6 Heisenberg): local
  energies, log-amplitudes, configurations and acceptance counts bit for bit;
  the gradient columns of the shared parameters within 2e-6 x sqrt(walker
  passes) of the largest entry (tensor cores against FP32 tiles), the zero
  units' columns exactly 0."""
  n_batches = 20
  ij, jx, jz = lattices.heisenberg_couplings(lattices.square_nn_bonds(N_SIDE))
  ham = native.Hamiltonian(ij, jx, jz, N)
  e1, l1, s1, acc1, sums1, stats1 = _run(native, rbm_pair[0], ham, batch, n_batches)
  e2, l2, s2, acc2, sums2, stats2 = _run(native, rbm_pair[1], ham, batch, n_batches)
  assert torch.equal(e1, e2)
  assert torch.equal(l1, l2)
  assert torch.equal(s1, s2)
  assert torch.equal(acc1, acc2) and int(acc1) > 0
  np.testing.assert_allclose(stats1.cpu().numpy(), stats2.cpu().numpy(), rtol=1e-12)
  side1, w1, c1 = _split(sums1, H)
  side2, w2, c2 = _split(sums2, HP)
  assert np.all(w2[:, :, H:] == 0) and np.all(c2[:, H:] == 0)
  ref = np.concatenate([side2.ravel(), w2[:, :, :H].ravel(), c2[:, :H].ravel()])
  got = np.concatenate([side1.ravel(), w1.ravel(), c1.ravel()])
  assert np.all(np.isfinite(ref))
  tol = 2e-6 * (np.abs(ref).max() + 1.0) * (n_batches * batch) ** 0.5
  np.testing.assert_allclose(got, ref, rtol=0, atol=tol)
