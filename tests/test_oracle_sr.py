"""CPU checks of stochastic reconfiguration: the float64 oracle's JVP, dense S
and matrix-free S v agree with each other, the library's conjugate-gradient
solver reproduces a direct solve, and the optimizer refuses wavefunctions it
has no JVP kernel for before touching the device."""
import numpy as np
import pytest
import torch

from oracle import ansatz as oansatz
from oracle import bits, sr

CASES = [
    oansatz.AnsatzSpec('rbm', 12, num_layers=0, layer_size=8),
    oansatz.AnsatzSpec('rbm', 16, num_layers=0, layer_size=16),
]


def _setup(spec, n_walkers, seed):
  params = oansatz.init_params(spec, seed=seed, bias_scale=0.3, dtype=torch.float64)
  rng = np.random.default_rng(seed)
  cfg = torch.from_numpy(bits.random_sz0_configs(spec.n_sites, n_walkers, rng)).to(torch.float64)
  v = torch.from_numpy(rng.standard_normal(oansatz.num_params(spec)))
  return params, cfg, v


@pytest.mark.parametrize('spec', CASES, ids=lambda s: 'n%d_h%d' % (s.n_sites, s.layer_size))
def test_jvp_equals_per_sample_gradients_times_tangent(spec):
  params, cfg, v = _setup(spec, 64, 3)
  o = sr.per_sample_grads(spec, params, cfg)
  assert o.shape == (64, oansatz.num_params(spec))
  np.testing.assert_allclose(sr.log_amp_jvp(spec, params, cfg, v).numpy(), (o @ v).numpy(),
                             rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('spec', CASES, ids=lambda s: 'n%d_h%d' % (s.n_sites, s.layer_size))
def test_dense_matvec_equals_matrix_free(spec):
  params, cfg, v = _setup(spec, 200, 4)
  dense = sr.sr_matrix(spec, params, cfg) @ v + 0.01 * v
  np.testing.assert_allclose(sr.sr_matvec(spec, params, cfg, v, 0.01).numpy(), dense.numpy(),
                             rtol=1e-10, atol=1e-12)


def test_conjugate_gradient_reproduces_direct_solve():
  """training.conjugate_gradient (the solver the optimizer runs on the device)
  on the oracle's dense S + shift I against numpy.linalg.solve."""
  from cgs_vmc_b200 import training
  spec = CASES[1]
  params, cfg, _ = _setup(spec, 400, 5)
  e_loc = torch.from_numpy(np.random.default_rng(6).standard_normal(400)) - 8.0
  shift = 0.01
  s = sr.sr_matrix(spec, params, cfg)
  a = s + shift * torch.eye(s.shape[0], dtype=s.dtype)
  f = sr.sr_forces(spec, params, cfg, e_loc)
  x, iterations, residual = training.conjugate_gradient(lambda p: a @ p, f, 1e-12, 2000)
  ref = sr.sr_direction(spec, params, cfg, e_loc, shift)
  assert residual <= 1e-12 and 0 < iterations < 2000
  assert np.linalg.norm(x.numpy() - ref) <= 1e-8 * np.linalg.norm(ref)


def test_conjugate_gradient_zero_right_hand_side_and_cap():
  from cgs_vmc_b200 import training
  a = torch.diag(torch.arange(1.0, 11.0, dtype=torch.float64))
  x, iterations, residual = training.conjugate_gradient(lambda p: a @ p, torch.zeros(10, dtype=torch.float64),
                                                        1e-6, 50)
  assert iterations == 0 and residual == 0.0 and not x.any()
  _, iterations, residual = training.conjugate_gradient(lambda p: a @ p, torch.ones(10, dtype=torch.float64),
                                                        1e-30, 3)
  assert iterations == 3 and residual > 0.0


@pytest.mark.parametrize('kind,overrides', [
    ('fully_connected', dict(num_fc_layers=1, fc_layer_size=8)),
    ('rbm', dict(num_fc_layers=1, fc_layer_size=8)),
    ('rbm', dict(num_fc_layers=0, fc_layer_size=300)),
    ('rbm', dict(num_fc_layers=0, fc_layer_size=8, num_sites=150)),
])
def test_sr_rejects_unsupported_wavefunctions_before_allocating(kind, overrides):
  """build_opt_ops refuses before it creates walkers or parameters, so the
  refusal does not need a device."""
  from cgs_vmc_b200 import operators, training, utils, wavefunctions
  hp = utils.create_hparams(wavefunction_type=kind, num_sites=overrides.pop('num_sites', 8), **overrides)
  wf = wavefunctions.build_wavefunction(hp)
  ham = operators.HeisenbergHamiltonian([(i, (i + 1) % hp.num_sites) for i in range(hp.num_sites)], -1.0, 1.0)
  with pytest.raises(NotImplementedError, match='pure RBM'):
    training.ground_state_optimizer('StochasticReconfiguration')().build_opt_ops(
        wavefunction=wf, hamiltonian=ham, hparams=hp, shared_resources={})
  assert wf._native is None


def test_sr_hparams_parse():
  from cgs_vmc_b200 import utils
  hp = utils.create_hparams()
  assert (hp.sr_diag_shift, hp.sr_cg_max_iterations, hp.sr_cg_tolerance) == (0.01, 100, 1e-4)
  hp.parse('sr_diag_shift=0.05,sr_cg_max_iterations=20,sr_cg_tolerance=1e-6,optimizer=gradient')
  assert (hp.sr_diag_shift, hp.sr_cg_max_iterations, hp.sr_cg_tolerance) == (0.05, 20, 1e-6)
