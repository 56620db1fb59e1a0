"""-m gpu tests of stochastic reconfiguration: cgsvmc_log_amp_jvp against the
float64 oracle and, through the adjoint identity, against the golden-pinned
cgsvmc_weighted_grad_sum; the matrix-free S v and one epoch's SR direction
against dense oracle solves; the sharded reduction; unsupported and empty
calls; training to the exact energy; the driver.  Tolerances are stated per
test."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_util import make_native, oracle_params, packed_cuda
from oracle import ansatz as oansatz
from oracle import bits, ed, hamiltonian, lattices, sr

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = torch.float64
SR_LR, SR_SHIFT = 0.1, 0.01      # chosen from one run of lr in {0.02, 0.05, 0.1} x shift 0.01

JVP_SHAPES = {
    'chain12_h8': oansatz.AnsatzSpec('rbm', 12, num_layers=0, layer_size=8),             # 1 word
    'c2_6x6_h144': oansatz.AnsatzSpec('rbm', 36, num_layers=0, layer_size=144),          # 1 word, C2
    'n100_h64': oansatz.AnsatzSpec('rbm', 100, num_layers=0, layer_size=64),             # 2 words
    '16x16_h256': oansatz.AnsatzSpec('rbm', 256, num_layers=0, layer_size=256),          # 4 words
}


def _rbm(spec, seed, n_walkers, bias=0.3):
  """Native ansatz, float64 oracle parameters (the float32 values) and random
  Sz = 0 walkers (numpy +-1 and packed on the device)."""
  flat = oansatz.flatten(oansatz.init_params(spec, seed=seed, bias_scale=bias, dtype=F64)).float()
  native = make_native(spec, flat.numpy())
  cfg = bits.random_sz0_configs(spec.n_sites, n_walkers, np.random.default_rng(seed))
  return native, oracle_params(spec, flat.numpy()), cfg, packed_cuda(cfg)


def _tangent(spec, seed, zero_w=False):
  v = torch.from_numpy(np.random.default_rng(seed + 100).standard_normal(oansatz.num_params(spec)))
  if zero_w:      # V = 0: only the visible and hidden biases move
    n, h = spec.n_sites, spec.layer_size
    v[n + 1:n + 1 + n * h] = 0.0
  return v


@pytest.mark.parametrize('batch', [1, 33, 1000])
@pytest.mark.parametrize('name', sorted(JVP_SHAPES))
def test_jvp_matches_float64_oracle(name, batch):
  """|y - y_ref| <= 1e-5 sum_p |O_bp v_p| + 1e-6 per walker, for a dense
  random tangent and one with a zero W block."""
  spec = JVP_SHAPES[name]
  native, params, cfg, packed = _rbm(spec, 11, batch)
  cfg64 = torch.from_numpy(cfg).to(F64)
  for zero_w in (False, True):
    v = _tangent(spec, 11, zero_w)
    y = native.log_amp_jvp(packed, v.float().cuda()).cpu().double()
    v32 = v.float().double()          # the tangent the kernel received
    ref = sr.log_amp_jvp(spec, params, cfg64, v32)
    scale = torch.cat([(sr.per_sample_grads(spec, params, chunk) * v32).abs().sum(dim=1)
                       for chunk in cfg64.split(50)])
    err = (y - ref).abs()
    assert bool((err <= 1e-5 * scale + 1e-6).all()), (zero_w, float((err / scale).max()))


def test_jvp_adjoint_of_weighted_grad_sum_c2():
  """w . jvp(v) == v . weighted_grad_sum(w) at C2 (6x6, H = 144, B = 8192),
  to 1e-5 relative to sum_b |w_b jvp(v)_b|: ties the new kernel to the
  golden-pinned gradient."""
  spec = JVP_SHAPES['c2_6x6_h144']
  native, _, _, packed = _rbm(spec, 12, 8192)
  rng = np.random.default_rng(13)
  w = torch.from_numpy(rng.standard_normal(8192)).float().cuda()
  v = torch.from_numpy(rng.standard_normal(native.num_params)).float().cuda()
  y = native.log_amp_jvp(packed, v).double()
  g = native.weighted_grad_sum(packed, w.reshape(1, -1))[0].double()
  lhs, rhs = float(torch.dot(w.double(), y)), float(torch.dot(v.double(), g))
  assert abs(lhs - rhs) <= 1e-5 * float((w.double() * y).abs().sum()), (lhs, rhs)


def test_unsupported_and_empty_calls():
  from cgs_vmc_b200 import _native, operators, training, utils, wavefunctions
  unsupported = [
      oansatz.AnsatzSpec('fully_connected', 16, num_layers=1, layer_size=8),
      oansatz.AnsatzSpec('conv_2d', 16, num_layers=1, num_filters=2, kernel_size=3, size_x=4, size_y=4),
      oansatz.AnsatzSpec('rbm', 16, num_layers=1, layer_size=8),
  ]
  for spec in unsupported:
    native = make_native(spec, np.zeros(oansatz.num_params(spec), np.float32))
    tangent = torch.zeros(native.num_params, device='cuda')
    for batch in (0, 4):      # UNSUPPORTED also without walkers: a call with none probes for support
      packed = torch.zeros(batch, 1, dtype=torch.int64, device='cuda')
      with pytest.raises(NotImplementedError):
        native.log_amp_jvp(packed, tangent)
  # the optimizer refuses the same three and a sum of two RBMs
  for kind, over in [('fully_connected', dict(num_fc_layers=1)), ('conv_2d', dict(num_conv_layers=1)),
                     ('rbm', dict(num_fc_layers=1)),
                     ('sum', dict(num_fc_layers=0, composite_wavefunction_types=('rbm', 'rbm'),
                                  composite_output_activations=('exp', 'exp')))]:
    hp = utils.create_hparams(wavefunction_type=kind, num_sites=16, size_x=4, size_y=4, fc_layer_size=8,
                              num_conv_filters=2, kernel_size=3, batch_size=64, **over)
    wf = wavefunctions.build_wavefunction(hp)
    ham = operators.HeisenbergHamiltonian(lattices.square_nn_bonds(4), -1.0, 1.0)
    with pytest.raises(NotImplementedError, match='pure RBM'):
      training.ground_state_optimizer('StochasticReconfiguration')().build_opt_ops(
          wavefunction=wf, hamiltonian=ham, hparams=hp, shared_resources={})
  # a supported ansatz: no walkers is a no-op, a NULL buffer is INVALID
  native, _, _, packed = _rbm(JVP_SHAPES['chain12_h8'], 14, 4)
  tangent = torch.ones(native.num_params, device='cuda')
  assert native.log_amp_jvp(packed[:0], tangent).shape == (0,)
  lib = _native.load()
  assert lib.cgsvmc_log_amp_jvp(native._handle, ctypes.c_void_p(packed.data_ptr()), 4, None,
                                None, None) == _native.ERR_INVALID
  assert lib.cgsvmc_log_amp_jvp(native._handle, None, 0, None, None, None) == _native.OK
  torch.cuda.synchronize()


def _sv_setup(n_walkers=4096):
  """4x4, H = 16 (P = 289) and M random walkers; <O> from the device sums."""
  spec = oansatz.AnsatzSpec('rbm', 16, num_layers=0, layer_size=16)
  native, params, cfg, packed = _rbm(spec, 21, n_walkers)
  ones = torch.ones(1, n_walkers, device='cuda')
  o_mean = native.weighted_grad_sum(packed, ones)[0].double() / n_walkers
  v = _tangent(spec, 21).cuda()
  return spec, native, params, cfg, packed, o_mean, v


def test_device_sv_matches_dense_oracle():
  """training.sr_matvec against the oracle's dense (S + shift I) v, 1e-4
  relative in norm."""
  from cgs_vmc_b200 import training
  spec, native, params, cfg, packed, o_mean, v = _sv_setup()
  shift = 0.01
  dev = training.sr_matvec(native, packed, o_mean, v, float(cfg.shape[0]), shift, allreduce=lambda t: t)
  s = sr.sr_matrix(spec, params, torch.from_numpy(cfg).to(F64))
  ref = s @ v.cpu() + shift * v.cpu()
  err = torch.linalg.vector_norm(dev.cpu() - ref) / torch.linalg.vector_norm(ref)
  assert float(err) <= 1e-4, float(err)


def test_virtual_shards_reduce_to_the_whole_store():
  """Two halves of the store, each with the reduction injected (rank 0's view:
  its own partial plus the other's), give the matvec over the whole store to
  float32 rounding."""
  from cgs_vmc_b200 import training
  _, native, _, cfg, packed, o_mean, v = _sv_setup()
  m, shift = float(cfg.shape[0]), 0.01
  halves = packed.split(cfg.shape[0] // 2)
  partials = []

  def record(t):
    partials.append(t.clone())
    return t
  for half in halves:
    training.sr_matvec(native, half, o_mean, v, m, shift, allreduce=record)
  sharded = [training.sr_matvec(native, halves[k], o_mean, v, m, shift,
                                allreduce=lambda t, k=k: t + partials[1 - k]) for k in (0, 1)]
  whole = training.sr_matvec(native, packed, o_mean, v, m, shift, allreduce=lambda t: t)
  norm = float(torch.linalg.vector_norm(whole))
  for part in sharded:
    assert float(torch.linalg.vector_norm(part - whole)) <= 1e-5 * norm
  assert torch.equal(sharded[0], sharded[1])


def _sr_hparams(**over):
  from cgs_vmc_b200 import utils
  base = dict(wavefunction_type='rbm', num_sites=16, size_x=4, size_y=4, num_fc_layers=0, fc_layer_size=16,
              batch_size=1024, num_batches_per_epoch=4, num_equilibration_sweeps=5, optimizer='gradient')
  base.update(over)
  return utils.create_hparams(**base)


def test_one_epoch_direction_matches_oracle_solve():
  """The SR direction of one epoch (4 captured batch steps of 1024 walkers on
  4x4, H = 16) against numpy.linalg.solve(S + shift I, F) of the float64
  oracle on the stored configurations with oracle local energies: 1e-3
  relative in norm.  The recorded CG residual is within the tolerance."""
  from cgs_vmc_b200 import graph_builders, operators, training, wavefunctions
  from cgs_vmc_b200.session import Session
  graph_builders.reset_num_epochs()
  hp = _sr_hparams(sr_diag_shift=0.05, sr_cg_tolerance=1e-6, sr_cg_max_iterations=500,
                   learning_rates=[0.05] * 4)
  wf = wavefunctions.build_wavefunction(hp).seed(3)
  bonds = lattices.square_nn_bonds(4)
  ham = operators.HeisenbergHamiltonian(bonds, -1.0, 1.0)
  opt = training.ground_state_optimizer('StochasticReconfiguration')()
  ops = opt.build_opt_ops(wavefunction=wf, hamiltonian=ham, hparams=hp, shared_resources={})
  s = Session()
  s.run(ops.mc_step, n_steps=hp.num_equilibration_sweeps * hp.num_sites)
  s.run(ops.reset_gradients)
  for _ in range(hp.num_batches_per_epoch):
    s.run(opt._batch_step)
  flat = wf.native().params.detach().cpu().numpy().copy()
  s.run(ops.apply_gradients)
  assert opt.cg_residual <= hp.sr_cg_tolerance and 0 < opt.cg_iterations <= hp.sr_cg_max_iterations
  packed = opt.stored_configs()
  assert packed.shape == (4096, 1)
  spec = oansatz.AnsatzSpec('rbm', 16, num_layers=0, layer_size=16)
  params = oracle_params(spec, flat)
  cfg = torch.from_numpy(bits.unpack(packed.cpu().numpy().view(np.uint64), 16)).to(F64)
  ij, jx, jz = lattices.heisenberg_couplings(bonds)
  e_loc = hamiltonian.local_energy(cfg, ij, jx, jz, lambda c: oansatz.log_amp(spec, params, c))
  ref = sr.sr_direction(spec, params, cfg, e_loc, hp.sr_diag_shift)
  dev = opt.direction.cpu().numpy()
  assert np.linalg.norm(dev - ref) <= 1e-3 * np.linalg.norm(ref), np.linalg.norm(dev - ref) / np.linalg.norm(ref)
  # the update is params -= lr delta
  np.testing.assert_allclose(wf.native().params.cpu().numpy(), flat - 0.05 * dev.astype(np.float32),
                             rtol=0, atol=1e-6)


def test_sr_training_reaches_exact_energy():
  """4x4 Heisenberg (E0 = -11.2284832084), H = 16, optimizer=gradient, seeded:
  the mean of the last 10 of 100 epochs is within 1 % of E0 and not below it
  by more than the Monte-Carlo noise.  Measured on a B200: the 10-epoch
  running mean is first within 1 % after 32 epochs and 0.53 % off after 100."""
  from cgs_vmc_b200 import graph_builders, operators, training, wavefunctions
  from cgs_vmc_b200.session import Session
  graph_builders.reset_num_epochs()
  hp = _sr_hparams(learning_rates=[SR_LR] * 4, sr_diag_shift=SR_SHIFT)
  wf = wavefunctions.build_wavefunction(hp).seed(2)
  ham = operators.HeisenbergHamiltonian(lattices.square_nn_bonds(4), -1.0, 1.0)
  opt = training.ground_state_optimizer('StochasticReconfiguration')()
  ops = opt.build_opt_ops(wavefunction=wf, hamiltonian=ham, hparams=hp, shared_resources={})
  s = Session()
  energies = [opt.run_optimization_epoch(ops, s, hp) for _ in range(100)]
  e0, _, _ = ed.ground_state(16, *lattices.heisenberg_couplings(lattices.square_nn_bonds(4)))
  assert abs(e0 - (-11.2284832084)) < 1e-6
  tail = np.mean(energies[-10:])
  assert energies[0] > tail
  assert abs(tail - e0) < 0.01 * abs(e0), (energies[0], energies[-10:], e0)
  assert tail > e0 - 0.05          # variational within MC noise


def test_driver_end_to_end(tmp_path):
  """run_training.py --optimizer StochasticReconfiguration on the 8-site chain."""
  ckpt = str(tmp_path / 'sr')
  env = dict(os.environ, PYTHONPATH=REPO)
  subprocess.run([sys.executable, os.path.join(REPO, 'run_training.py'), '--checkpoint_dir', ckpt,
                  '--num_sites', '8', '--num_epochs', '3', '--wavefunction_type', 'rbm',
                  '--heisenberg_jx', '-1.0', '--optimizer', 'StochasticReconfiguration', '--hparams',
                  'batch_size=256,num_batches_per_epoch=3,num_equilibration_sweeps=2,fc_layer_size=8,'
                  'num_fc_layers=0,optimizer=gradient,learning_rates=[0.05,0.05,0.05,0.05],sr_diag_shift=0.01'],
                 check=True, env=env, timeout=300)
  metrics = open(os.path.join(ckpt, 'metrics.txt')).read().split()
  assert len(metrics) == 3 and all(np.isfinite(float(m)) for m in metrics)
  assert os.path.exists(os.path.join(ckpt, 'model_prior_2_epochs.pt'))
  assert os.path.exists(os.path.join(ckpt, 'hparams.pbtxt'))
