"""-m gpu tests of the per-bond local values (cgsvmc_bond_values,
cgsvmc_bond_values_from_amps, operators.HeisenbergBonds) and of the spin-spin
correlations built on them: the fused pure-RBM kernel against the float64
reference on fixed configurations for every KJ and both W placements; a large
all-pairs table against the amplitude route; the sum over bonds against the
local energy of every ansatz kind; exact expectations over the whole Sz = 0
basis; the C-ABI's argument handling; the evaluator and the driver.
Deterministic unless a test says otherwise; tolerances are stated per test."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from bond_oracle import bond_values as oracle_bond_values
from bond_oracle import exact_bond_expectations
from gpu_util import make_native, oracle_params, packed_cuda
from oracle import ansatz as oansatz
from oracle import bits

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = torch.float64

# every KJ (2, 4, 5, 8), 1, 2 and 4 spin words, W in shared memory and not (16x16)
SHAPES = {
    'n12_h24': oansatz.AnsatzSpec('rbm', 12, num_layers=0, layer_size=24),
    'c2_6x6_h144': oansatz.AnsatzSpec('rbm', 36, num_layers=0, layer_size=144),
    '10x10_h100': oansatz.AnsatzSpec('rbm', 100, num_layers=0, layer_size=100),
    '16x16_h256': oansatz.AnsatzSpec('rbm', 256, num_layers=0, layer_size=256),
}


def _lat():
  from cgs_vmc_b200 import lattices
  return lattices


def _rbm(spec, seed, n_walkers, bias=0.3):
  flat = oansatz.flatten(oansatz.init_params(spec, seed=seed, bias_scale=bias, dtype=F64)).float()
  native = make_native(spec, flat.numpy())
  cfg = bits.random_sz0_configs(spec.n_sites, n_walkers, np.random.default_rng(seed))
  return native, oracle_params(spec, flat.numpy()), cfg, packed_cuda(cfg)


def _pair_lists(n, rng):
  """name -> (ij int32 [K, 2], jx float32 [K], jz float32 [K])."""
  lat = _lat()
  side = int(round(n ** 0.5))
  nn = lat.square_nn_bonds(side) if side * side == n and n > 12 else lat.chain_bonds(n)
  out = {'nn': (np.asarray(nn, np.int32), np.full(len(nn), -1.0, np.float32), np.ones(len(nn), np.float32))}
  if n <= 100:
    ap = np.asarray(lat.all_pairs(n), np.int32)
    out['all_pairs'] = (ap, rng.choice([-1.0, 1.0], len(ap)).astype(np.float32), np.ones(len(ap), np.float32))
  i = rng.integers(0, n, 300)
  j = (i + rng.integers(1, n, 300)) % n                      # i != j, either order, repeats
  rnd = np.stack([i, j], 1).astype(np.int32)
  out['random'] = (rnd, rng.uniform(-1.5, 1.5, 300).astype(np.float32), rng.uniform(-1, 1, 300).astype(np.float32))
  if n > 64:                                                 # one site in each of two different words
    a = rng.integers(0, 64, 100)
    b = rng.integers(64, n, 100)
    span = np.stack([np.where(np.arange(100) % 2 == 0, a, b), np.where(np.arange(100) % 2 == 0, b, a)], 1)
    out['span_words'] = (span.astype(np.int32), np.full(100, 1.0, np.float32), np.full(100, 1.0, np.float32))
  jx0 = rnd[:64].copy()
  jx = np.where(np.arange(64) % 2 == 0, 0.0, 1.0).astype(np.float32)
  out['jx_zero'] = (jx0, jx, rng.uniform(-1, 1, 64).astype(np.float32))
  return out


def _check_against_oracle(v, cfg, spec, params, ij, jx, jz, cols=None):
  """|v - ref| <= 1e-4 |off-diagonal part| + 1e-6 per entry, the diagonal-only
  entries (parallel spins or jx = 0) bit-exact: float32 ratios from a sum of H
  log-cosh differences."""
  cols = np.arange(len(ij)) if cols is None else cols
  cfg64 = torch.from_numpy(cfg).to(F64)
  fn = lambda c: oansatz.log_amp(spec, params, c)
  ref = oracle_bond_values(cfg64, ij[cols], jx[cols].astype(np.float64), jz[cols].astype(np.float64), fn).numpy()
  got = v[:, cols]
  s = cfg[:, ij[cols, 0]] * cfg[:, ij[cols, 1]]
  diag = (0.25 * jz[cols]).astype(np.float32) * s.astype(np.float32)
  off = ref - diag
  err = np.abs(got - ref)
  assert np.all(err <= 1e-4 * np.abs(off) + 1e-6), float(err.max())
  only_diag = (s > 0) | (jx[cols] == 0)[None, :]
  np.testing.assert_array_equal(got[only_diag], diag[only_diag])


@pytest.mark.parametrize('name', sorted(SHAPES))
def test_fused_kernel_matches_float64_oracle(name):
  from cgs_vmc_b200 import _native
  spec = SHAPES[name]
  native, params, cfg, packed = _rbm(spec, 21, 67)
  rng = np.random.default_rng(5)
  for lname, (ij, jx, jz) in _pair_lists(spec.n_sites, rng).items():
    ham = _native.Hamiltonian(ij, jx, jz, spec.n_sites)
    v = native.bond_values(ham, packed).cpu().numpy()
    assert v.shape == (67, len(ij)), lname
    _check_against_oracle(v, cfg, spec, params, ij, jx, jz)


def _amplitude_route(native, ham, packed):
  """flip_enum + log_amp + cgsvmc_bond_values_from_amps, called directly."""
  from cgs_vmc_b200 import _native
  b = packed.shape[0]
  z = native.log_amp(packed)
  _, flipped = ham.flip_enum(packed)
  fl = native.log_amp(flipped.reshape(b * ham.n_bonds, -1)).reshape(b, ham.n_bonds)
  return _native.bond_values_from_amps(ham, packed, z, None, fl, None)


def test_all_pairs_at_256_sites():
  """All 32,640 pairs at N = 256 (most of the table read from global memory):
  every entry against the amplitude route, a sample of 400 bonds against the
  float64 reference."""
  from cgs_vmc_b200 import _native
  spec = SHAPES['16x16_h256']
  native, params, cfg, packed = _rbm(spec, 22, 64)
  lat = _lat()
  ij = np.asarray(lat.all_pairs(256), np.int32)
  assert len(ij) == 32640
  st = np.where((np.arange(256) // 16 + np.arange(256) % 16) % 2 == 0, 1.0, -1.0)
  jx = (st[ij[:, 0]] * st[ij[:, 1]]).astype(np.float32)
  jz = np.ones(len(ij), np.float32)
  ham = _native.Hamiltonian(ij, jx, jz, 256)
  v = native.bond_values(ham, packed)
  amp = _amplitude_route(native, ham, packed)
  assert bool(torch.isfinite(v).all())
  err = (v - amp).abs()
  assert bool((err <= 3e-4 * (amp.abs() + 0.25)).all()), float(err.max())   # amp: z' - z of two full passes
  cols = np.sort(np.random.default_rng(3).choice(len(ij), 400, replace=False))
  cols = np.concatenate([cols, [0, 7103, 7104, 7105, len(ij) - 1]])   # around the end of the staged part
  _check_against_oracle(v.cpu().numpy(), cfg, spec, params, ij, jx, jz, cols=cols)


SUM_KINDS = [
    ('rbm', dict(num_sites=16, num_fc_layers=0, fc_layer_size=12)),
    ('fully_connected', dict(num_sites=16, num_fc_layers=1, fc_layer_size=8)),
    ('rbm', dict(num_sites=16, num_fc_layers=1, fc_layer_size=8)),
    ('conv_1d', dict(num_sites=12, num_conv_layers=2, num_conv_filters=4, kernel_size=3)),
    ('conv_2d', dict(num_sites=16, size_x=4, size_y=4, num_conv_layers=2, num_conv_filters=4, kernel_size=3)),
    ('res_net_1d', dict(num_sites=12, num_resnet_blocks=1, num_conv_filters=4, kernel_size=3)),
    ('fully_connected', dict(num_sites=16, num_fc_layers=1, fc_layer_size=8, output_activation='tanh')),
    ('sum', dict(num_sites=16, num_fc_layers=1, fc_layer_size=8,
                 composite_wavefunction_types=('rbm', 'fully_connected'),
                 composite_output_activations=('exp', 'tanh'))),
    ('prod', dict(num_sites=16, num_fc_layers=0, fc_layer_size=8,
                  composite_wavefunction_types=('rbm', 'rbm'), composite_output_activations=('exp', 'exp'))),
]


@pytest.mark.parametrize('kind,overrides', SUM_KINDS,
                         ids=['rbm', 'fc', 'rbm_hidden', 'conv_1d', 'conv_2d', 'resnet_1d', 'fc_tanh', 'sum',
                              'prod'])
def test_bond_values_sum_to_local_energy(kind, overrides):
  """sum_k values[b, k] == E_loc[b] of HeisenbergHamiltonian.local_value to
  2e-5 (sum_k |values[b, k]| + 1): the same terms, summed in another order (and
  for the pure RBM by another kernel)."""
  from cgs_vmc_b200 import operators, utils, wavefunctions
  hp = utils.create_hparams(wavefunction_type=kind, **overrides)
  wf = wavefunctions.build_wavefunction(hp).seed(7) if kind not in ('sum', 'prod') else \
      wavefunctions.build_wavefunction(hp)
  n = hp.num_sites
  lat = _lat()
  bonds = lat.chain_bonds(n) + [(i, (i + 2) % n) for i in range(n)]
  jx = np.array([-1.0] * n + [0.5] * n, np.float32)
  jz = np.array([1.0] * n + [0.5] * n, np.float32)
  inputs = torch.from_numpy(bits.random_sz0_configs(n, 64, np.random.default_rng(8))).cuda()
  e = operators.HeisenbergHamiltonian(bonds, jx, jz).local_value(wf, inputs).double()
  v = operators.HeisenbergBonds(bonds, jx, jz).local_value(wf, inputs).double()
  assert tuple(v.shape) == (64, 2 * n) and v.dtype == F64
  assert bool(torch.isfinite(v).all())
  err = (v.sum(dim=1) - e).abs()
  assert bool((err <= 2e-5 * (v.abs().sum(dim=1) + 1.0)).all()), float(err.max())


def test_fused_route_matches_amplitude_route():
  """N = 12: the fused kernel and the amplitude route through the C-ABI give
  the same values to float32 accuracy, on NN bonds and all pairs."""
  from cgs_vmc_b200 import _native
  spec = SHAPES['n12_h24']
  native, _, _, packed = _rbm(spec, 23, 200)
  lat = _lat()
  for bonds in (lat.chain_bonds(12), lat.all_pairs(12)):
    ham = _native.Hamiltonian(bonds, 1.0, 1.0, 12)
    fused = native.bond_values(ham, packed)
    amp = _amplitude_route(native, ham, packed)
    torch.testing.assert_close(fused, amp, rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize('kind', ['rbm', 'fully_connected'])
def test_exact_expectations_over_the_sz0_basis(kind):
  """All 924 Sz = 0 configurations of the 12-site chain as walkers, weighted
  by |psi|^2 / Z from the device amplitudes: the weighted bond values equal
  <psi|S_i . S_j|psi> / <psi|psi> of all 66 pairs to 1e-5, on the route
  HeisenbergBonds picks and, for the pure RBM, on the amplitude route too."""
  from cgs_vmc_b200 import _native, operators, utils, wavefunctions
  from oracle import ed
  n = 12
  hp = utils.create_hparams(wavefunction_type=kind, num_sites=n, num_fc_layers=0 if kind == 'rbm' else 1,
                            fc_layer_size=24 if kind == 'rbm' else 8)
  wf = wavefunctions.build_wavefunction(hp).seed(9)
  cfg = ed.configs_of(ed.sz0_basis(n), n)
  assert cfg.shape == (924, n)
  inputs = torch.from_numpy(cfg).float().cuda()
  pairs = _lat().all_pairs(n)
  op = operators.HeisenbergBonds(pairs, 1.0, 1.0)
  v = op.local_value(wf, inputs).double()
  packed = packed_cuda(cfg)
  logabs, _ = wf.amplitudes(packed)
  w = torch.exp(2.0 * (logabs.double() - logabs.double().max()))
  w = w / w.sum()
  spec = oansatz.AnsatzSpec(kind, n, num_layers=hp.num_fc_layers, layer_size=hp.fc_layer_size,
                            nonlinearity=hp.nonlinearity)
  params = [p.detach().cpu().to(F64) for p in wf.get_trainable_variables()]
  psi_fn = lambda c: oansatz.psi(spec, params, torch.from_numpy(np.asarray(c)).to(F64), shift=0.0).numpy()
  exact = exact_bond_expectations(n, pairs, np.ones(len(pairs)), np.ones(len(pairs)), psi_fn)
  np.testing.assert_allclose((w[:, None] * v).sum(dim=0).cpu().numpy(), exact, rtol=0, atol=1e-5)
  if kind == 'rbm':
    amp = _amplitude_route(wf.native(), op.native(n), packed).double()
    np.testing.assert_allclose((w[:, None] * amp).sum(dim=0).cpu().numpy(), exact, rtol=0, atol=1e-5)


def test_api_probes_and_argument_errors():
  from cgs_vmc_b200 import _native, operators, utils, wavefunctions
  lib = _native.load()
  vp = ctypes.c_void_p
  conv = oansatz.AnsatzSpec('conv_1d', 12, num_layers=1, num_filters=2, kernel_size=3)
  others = [conv, oansatz.AnsatzSpec('fully_connected', 12, num_layers=1, layer_size=8),
            oansatz.AnsatzSpec('rbm', 12, num_layers=1, layer_size=8)]
  ham = _native.Hamiltonian(_lat().chain_bonds(12), 1.0, 1.0, 12)
  packed = packed_cuda(bits.random_sz0_configs(12, 4, np.random.default_rng(1)))
  vals = torch.empty(4, 12, device='cuda')
  for spec in others:
    a = make_native(spec, np.zeros(oansatz.num_params(spec), np.float32))
    assert lib.cgsvmc_bond_values(a._handle, ham._handle, None, 0, None, None) == _native.ERR_UNSUPPORTED
    assert lib.cgsvmc_bond_values(a._handle, ham._handle, vp(packed.data_ptr()), 4, vp(vals.data_ptr()),
                                  None) == _native.ERR_UNSUPPORTED
    with pytest.raises(NotImplementedError):
      a.bond_values(ham, packed)
  native, _, _, _ = _rbm(SHAPES['n12_h24'], 24, 1)
  h, p, o = native._handle, vp(packed.data_ptr()), vp(vals.data_ptr())
  # no-ops: no walkers, no bonds
  assert lib.cgsvmc_bond_values(h, ham._handle, None, 0, None, None) == _native.OK
  empty = _native.Hamiltonian(np.zeros((0, 2), np.int32), [], [], 12)
  assert lib.cgsvmc_bond_values(h, empty._handle, p, 4, None, None) == _native.OK
  assert tuple(native.bond_values(empty, packed).shape) == (4, 0)
  assert tuple(native.bond_values(ham, packed[:0]).shape) == (0, 12)
  z = torch.zeros(4, device='cuda')
  assert lib.cgsvmc_bond_values_from_amps(ham._handle, None, 0, None, None, None, None, None, None) == _native.OK
  assert lib.cgsvmc_bond_values_from_amps(empty._handle, p, 4, vp(z.data_ptr()), None, None, None, None,
                                          None) == _native.OK
  # INVALID: NULL handles and buffers, negative sizes, mismatched n_sites
  assert lib.cgsvmc_bond_values(None, ham._handle, p, 4, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_bond_values(h, None, p, 4, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_bond_values(h, ham._handle, p, -1, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_bond_values(h, ham._handle, None, 4, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_bond_values(h, ham._handle, p, 4, None, None) == _native.ERR_INVALID
  ham16 = _native.Hamiltonian(_lat().chain_bonds(16), 1.0, 1.0, 16)
  assert lib.cgsvmc_bond_values(h, ham16._handle, p, 4, o, None) == _native.ERR_INVALID
  fl = torch.zeros(4, 12, device='cuda')
  args = [p, 4, vp(z.data_ptr()), None, vp(fl.data_ptr()), None, o, None]
  assert lib.cgsvmc_bond_values_from_amps(ham._handle, *args) == _native.OK
  assert lib.cgsvmc_bond_values_from_amps(None, *args) == _native.ERR_INVALID
  for k in (0, 2, 4, 6):       # packed, logabs, flipped_logabs, values
    bad = list(args)
    bad[k] = None
    assert lib.cgsvmc_bond_values_from_amps(ham._handle, *bad) == _native.ERR_INVALID, k
  bad = list(args)
  bad[1] = -1
  assert lib.cgsvmc_bond_values_from_amps(ham._handle, *bad) == _native.ERR_INVALID
  # HeisenbergBonds on a conv ansatz: the amplitude route
  hp = utils.create_hparams(wavefunction_type='conv_1d', num_sites=12, num_conv_layers=1, num_conv_filters=2,
                            kernel_size=3)
  wf = wavefunctions.build_wavefunction(hp).seed(2)
  inputs = torch.from_numpy(bits.random_sz0_configs(12, 16, np.random.default_rng(2))).cuda()
  with pytest.raises(NotImplementedError):
    wf.native(12).bond_values(ham, packed)
  v = operators.HeisenbergBonds(_lat().chain_bonds(12), 1.0, 1.0).local_value(wf, inputs)
  assert tuple(v.shape) == (16, 12) and bool(torch.isfinite(v).all())
  torch.cuda.synchronize()


def _evaluator_setup(kind_overrides, seed):
  from cgs_vmc_b200 import graph_builders, utils, wavefunctions
  graph_builders.reset_num_epochs()
  hp = utils.create_hparams(**kind_overrides)
  return hp, wavefunctions.build_wavefunction(hp).seed(seed)


def test_evaluator_vector_sums_to_energy():
  """On one shared_resources and with no Monte-Carlo step in between, the
  HeisenbergBonds(NN, -1, 1) vector of the evaluator sums to its
  HeisenbergHamiltonian value to 1e-6 relative."""
  from cgs_vmc_b200 import evaluation, operators
  from cgs_vmc_b200.session import Session
  n = 16
  hp, wf = _evaluator_setup(dict(wavefunction_type='rbm', num_sites=n, num_fc_layers=0, fc_layer_size=16,
                                 batch_size=2048), 5)
  bonds = _lat().square_nn_bonds(4)
  ev = evaluation.MonteCarloOperatorEvaluator()
  shared = {}
  e_ops = ev.build_eval_ops(wavefunction=wf, operator=operators.HeisenbergHamiltonian(bonds, -1.0, 1.0),
                            hparams=hp, shared_resources=shared)
  b_ops = ev.build_eval_ops(wavefunction=wf, operator=operators.HeisenbergBonds(bonds, -1.0, 1.0),
                            hparams=hp, shared_resources=shared)
  s = Session()
  s.run(e_ops.mc_step, n_steps=10 * n)
  energy = s.run(e_ops.value)
  vec = s.run(b_ops.value)
  assert isinstance(vec, np.ndarray) and vec.dtype == np.float64 and vec.shape == (len(bonds),)
  assert abs(vec.sum() - energy) <= 1e-6 * abs(energy), (vec.sum(), energy)


def test_evaluator_correlations_match_exact():
  """Monte Carlo (fixed seeds): the 12-site chain's sampled correlations of
  all 66 pairs agree with the exact ones of the same parameters within 4
  error bars per pair (error bar as in test_monte_carlo_operator_evaluator)."""
  from cgs_vmc_b200 import evaluation, operators
  from cgs_vmc_b200.session import Session
  n = 12
  hp, wf = _evaluator_setup(dict(wavefunction_type='rbm', num_sites=n, num_fc_layers=0, fc_layer_size=24,
                                 batch_size=4096, num_equilibration_sweeps=20, num_monte_carlo_sweeps=2,
                                 num_evaluation_samples=40), 6)
  pairs = _lat().all_pairs(n)
  ev = evaluation.MonteCarloOperatorEvaluator()
  ops = ev.build_eval_ops(wavefunction=wf, operator=operators.HeisenbergBonds(pairs, 1.0, 1.0), hparams=hp,
                          shared_resources={})
  values = np.asarray(ev.run_evaluation(ops, Session(), hp, epoch_num=0))
  assert values.shape == (hp.num_evaluation_samples, len(pairs))
  spec = oansatz.AnsatzSpec('rbm', n, num_layers=0, layer_size=24)
  params = [p.detach().cpu().to(F64) for p in wf.get_trainable_variables()]
  psi_fn = lambda c: oansatz.psi(spec, params, torch.from_numpy(np.asarray(c)).to(F64), shift=0.0).numpy()
  exact = exact_bond_expectations(n, pairs, np.ones(len(pairs)), np.ones(len(pairs)), psi_fn)
  err = 2.0 * values.std(axis=0, ddof=1) / np.sqrt(len(values))
  dev = np.abs(values.mean(axis=0) - exact)
  assert np.all(dev < 4.0 * err + 1e-4), (dev / err).max()


def test_driver_writes_correlations(tmp_path):
  """run_training (8-site chain, --heisenberg_jx -1), then
  run_energy_evaluation with and without --correlations_file: the same Energy
  line, and an .npz with pairs, signs, mean, stderr, the symmetric matrix with
  diagonal 3/4 and a structure factor summing to 3N/4."""
  ckpt = str(tmp_path / 'gs')
  env = dict(os.environ, PYTHONPATH=REPO)
  common = 'batch_size=256,num_batches_per_epoch=3,num_equilibration_sweeps=2,fc_layer_size=8,num_fc_layers=0'
  subprocess.run([sys.executable, os.path.join(REPO, 'run_training.py'), '--checkpoint_dir', ckpt,
                  '--num_sites', '8', '--num_epochs', '3', '--wavefunction_type', 'rbm',
                  '--heisenberg_jx', '-1.0', '--optimizer', 'EnergyGradient', '--hparams', common],
                 check=True, env=env, timeout=300)
  base = [sys.executable, os.path.join(REPO, 'run_energy_evaluation.py'), '--checkpoint_dir', ckpt,
          '--heisenberg_jx', '-1.0', '--hparams', 'num_evaluation_samples=4']
  plain = subprocess.run(base, check=True, env=env, timeout=300, capture_output=True, text=True)
  path = str(tmp_path / 'corr.npz')
  with_corr = subprocess.run(base + ['--correlations_file', path], check=True, env=env, timeout=300,
                             capture_output=True, text=True)
  energy = [l for l in plain.stdout.splitlines() if l.startswith('Energy:')]
  assert len(energy) == 1
  assert energy == [l for l in with_corr.stdout.splitlines() if l.startswith('Energy:')]
  d = np.load(path)
  n = 8
  assert set(d.files) == {'pairs', 'signs', 'mean', 'stderr', 'matrix', 'structure_factor'}
  assert d['pairs'].shape == (28, 2) and d['mean'].shape == (28,) and d['stderr'].shape == (28,)
  np.testing.assert_array_equal(d['signs'], np.array([1, -1] * 4, np.int8))
  m = d['matrix']
  assert m.shape == (n, n)
  np.testing.assert_array_equal(m, m.T)
  np.testing.assert_array_equal(np.diag(m), np.full(n, 0.75))
  sq = d['structure_factor']
  assert sq.shape == (n, 1) and np.all(np.isfinite(sq))
  assert abs(sq.sum() - 0.75 * n) < 1e-9
