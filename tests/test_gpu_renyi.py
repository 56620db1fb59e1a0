"""-m gpu tests of the second Renyi entropy (cgsvmc_swap_values,
cgsvmc_swap_configs, cgsvmc_swap_values_from_amps, operators.RenyiSwap): the
fused pure-RBM kernel against the float64 reference for every KJ and both W
placements, the order rule that makes a region's value independent of the list
around it, the amplitude route for every ansatz kind, exact purities over all
pairs of the 12-site Sz = 0 basis, Monte Carlo through the evaluator, the
C-ABI's argument handling and the driver.  Deterministic (fixed seeds);
tolerances are stated per test."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_util import make_native, oracle_params, packed_cuda
from oracle import ansatz as oansatz
from oracle import bits, composite, ed
from renyi_oracle import exact_purity, swap_values
from test_gpu_bond_values import SHAPES, SUM_KINDS

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = torch.float64


def _prefixes(n):
  from cgs_vmc_b200 import lattices
  return lattices.prefix_regions(n)


def _masks(regions):
  from cgs_vmc_b200 import operators
  return operators.RenyiSwap(regions).masks(torch.device('cuda'))


def _region_list(n, rng):
  """bool [R, N]: prefixes, random masks, sparse masks, windows across the
  64-site words, the empty and the full region, complements."""
  pre = _prefixes(n)
  rnd = rng.random((12, n)) < 0.5
  sparse = rng.random((6, n)) < 0.1
  win = np.zeros((3, n), bool)
  for k, c in enumerate((64, 128, 192)):
    c = min(c, n // 2)
    win[k, max(0, c - 7):min(n, c + 9)] = True
  spread = np.zeros((1, n), bool)
  spread[0, [s for s in (3, 69, 133, 197, 250) if s < n]] = True
  ends = np.zeros((2, n), bool)
  ends[1] = True
  return np.concatenate([pre, rnd, sparse, win, spread, ends, ~pre[::max(1, len(pre) // 4)], ~rnd[:4]])


def _rbm(spec, seed, n_pairs):
  flat = oansatz.flatten(oansatz.init_params(spec, seed=seed, bias_scale=0.3, dtype=F64)).float()
  native = make_native(spec, flat.numpy())
  cfg = bits.random_sz0_configs(spec.n_sites, 2 * n_pairs, np.random.default_rng(seed))
  return native, oracle_params(spec, flat.numpy()), cfg, packed_cuda(cfg)


def _rules(c1, c2, regions):
  """(sector broken, swap gives back the pair) per (pair, region)."""
  m = regions[None, :, :]
  up1 = ((c1 > 0)[:, None, :] & m).sum(axis=2)
  up2 = ((c2 > 0)[:, None, :] & m).sum(axis=2)
  differ = (c1 != c2)[:, None, :]
  d = differ & m
  trivial = ~d.any(axis=2) | (d == differ).all(axis=2)
  return up1 != up2, trivial


def _check_fused(v, cfg, regions, spec, params):
  """Rule entries exact (0 where the sector is broken, 1.0 where the swap
  gives back the pair); the others against the float64 reference r with

    |v - r| <= r (2^-17 L + 4 H 2^-21 + 2^-20 (|log r| + 1)),

  L = sum_j lc(th1'_j) + lc(th1_j) + lc(th2'_j) + lc(th2_j).  log r is a sum of
  4H float32 log-cosh values: each carries the error of ex2 / lg2.approx
  (below 2^-21 absolute) and of its argument, theta, rounded over at most
  N + |D| additions (generously 2^-17 of |lc| per term); fast_exp adds a
  relative 2^-22 and the rounding of log r * log2(e) (2^-24 |log r|).  Entries
  with |log r| > 80 (near the float32 range) are not compared; at least 90 %
  of the computed entries are."""
  p = len(cfg) // 2
  c1, c2 = cfg[:p], cfg[p:]
  broken, trivial = _rules(c1, c2, regions)
  assert not np.any(v[broken]), 'sector rule'
  np.testing.assert_array_equal(v[~broken & trivial], 1.0)
  fn = lambda c: oansatz.log_amp(spec, params, c)
  ref = swap_values(c1, c2, regions, log_amp_fn=fn).numpy()
  comp = ~broken & ~trivial
  assert comp.sum() >= 50
  w, c = params[-2], params[-1]
  t1 = torch.from_numpy(c1).to(F64) @ w + c
  t2 = torch.from_numpy(c2).to(F64) @ w + c
  lsum = np.zeros(v.shape)
  for r in range(len(regions)):
    m = torch.from_numpy(regions[r])[None, :]
    t1s = torch.where(m, torch.from_numpy(c2), torch.from_numpy(c1)).to(F64) @ w + c
    t2s = torch.where(m, torch.from_numpy(c1), torch.from_numpy(c2)).to(F64) @ w + c
    lsum[:, r] = sum(oansatz.log_cosh(t).sum(dim=1).numpy() for t in (t1, t2, t1s, t2s))
  lr = np.log(np.where(comp, ref, 1.0))
  tol = 2.0 ** -17 * lsum + 4 * spec.layer_size * 2.0 ** -21 + 2.0 ** -20 * (np.abs(lr) + 1.0)
  keep = comp & (np.abs(lr) <= 80.0)
  assert keep.sum() >= 0.9 * comp.sum()
  err = np.abs(v.astype(np.float64) - ref)
  assert np.all(err[keep] <= (tol * ref)[keep]), float((err / (tol * ref))[keep].max())


@pytest.mark.parametrize('name', sorted(SHAPES))
def test_fused_kernel_matches_float64_oracle(name):
  spec = SHAPES[name]
  native, params, cfg, packed = _rbm(spec, 31, 67)
  regions = _region_list(spec.n_sites, np.random.default_rng(5))
  v = native.swap_values(packed, _masks(regions))
  assert tuple(v.shape) == (67, len(regions))
  _check_fused(v.cpu().numpy(), cfg, regions, spec, params)


@pytest.mark.parametrize('name', ['c2_6x6_h144', '16x16_h256'])
def test_region_value_does_not_depend_on_the_list(name):
  """Delta is summed over D in increasing site order whether it extends the
  previous region's or restarts: each region alone, inside a shuffled list and
  inside the prefix list gives bit-identical values."""
  spec = SHAPES[name]
  native, _, _, packed = _rbm(spec, 32, 150)
  n = spec.n_sites
  rng = np.random.default_rng(6)
  regions = _region_list(n, rng)
  alone = np.stack([native.swap_values(packed, _masks(regions[r:r + 1])).cpu().numpy()[:, 0]
                    for r in range(len(regions))], axis=1)
  order = rng.permutation(len(regions))
  shuffled = np.empty_like(alone)
  shuffled[:, order] = native.swap_values(packed, _masks(regions[order])).cpu().numpy()
  np.testing.assert_array_equal(shuffled, alone)
  listed = native.swap_values(packed, _masks(regions)).cpu().numpy()
  np.testing.assert_array_equal(listed, alone)
  pre = native.swap_values(packed, _masks(_prefixes(n))).cpu().numpy()
  np.testing.assert_array_equal(pre, alone[:, :n // 2])
  assert np.all(np.isfinite(alone))


def _amplitude_route(amplitudes, packed, n, masks):
  """cgsvmc_swap_configs + amplitudes + cgsvmc_swap_values_from_amps."""
  from cgs_vmc_b200 import _native
  p, r = packed.shape[0] // 2, masks.shape[0]
  logabs, sign = amplitudes(packed)
  swapped = _native.swap_configs(packed, n, masks)
  sl, ss = amplitudes(swapped.reshape(p * r * 2, -1))
  return _native.swap_values_from_amps(packed, n, masks, logabs.float().contiguous(), sign.float().contiguous(),
                                       sl.float().reshape(p, r, 2).contiguous(),
                                       ss.float().reshape(p, r, 2).contiguous())


def _native_amplitudes(native):
  return lambda packed: (native.log_amp(packed), torch.ones(packed.shape[0], device='cuda'))


@pytest.mark.parametrize('name', ['n12_h24', 'c2_6x6_h144'])
def test_fused_route_matches_amplitude_route(name):
  """The two routes agree to float32 accuracy (the amplitude route takes
  l' - l from two full forward passes: 2e-4 relative), the rule entries
  exactly."""
  spec = SHAPES[name]
  native, _, _, packed = _rbm(spec, 33, 300)
  masks = _masks(_region_list(spec.n_sites, np.random.default_rng(7)))
  fused = native.swap_values(packed, masks)
  amp = _amplitude_route(_native_amplitudes(native), packed, spec.n_sites, masks)
  exact = (amp == 0) | (amp == 1)
  assert bool(torch.equal(fused[exact], amp[exact]))
  torch.testing.assert_close(fused, amp, rtol=2e-4, atol=1e-7)


def _oracle_psi(wf, kind):
  """float64 psi_fn of a built wavefunction (composite.psi over its leaves)."""
  from cgs_vmc_b200 import _native
  kinds = {v: k for k, v in _native.ANSATZ_KINDS.items()}
  acts = {v: k for k, v in _native.ACTIVATIONS.items()}
  leaves = []
  for leaf in wf.leaves():
    d = leaf.native().desc
    spec = oansatz.AnsatzSpec(kinds[d.kind], d.n_sites, num_layers=d.num_layers, layer_size=d.layer_size,
                              num_filters=d.num_filters, kernel_size=d.kernel_size, size_x=d.size_x,
                              size_y=d.size_y, nonlinearity=acts[d.nonlinearity])
    params = oansatz.unflatten(spec, leaf.native().params.detach().cpu().to(F64))
    act = getattr(leaf, '_output_activation', 'exp') or 'exp'
    shift = leaf._exp_norm_shift if act == 'exp' else 0.0
    leaves.append(composite.Leaf(spec, params, act, shift))
  ckind = kind if kind in ('sum', 'prod') else 'single'
  return lambda c: composite.psi(ckind, leaves, torch.as_tensor(np.asarray(c)).to(F64))


@pytest.mark.parametrize('kind,overrides', SUM_KINDS,
                         ids=['rbm', 'fc', 'rbm_hidden', 'conv_1d', 'conv_2d', 'resnet_1d', 'fc_tanh', 'sum',
                              'prod'])
def test_amplitude_route_matches_reference(kind, overrides):
  """RenyiSwap.local_value of every ansatz kind (fused for the pure RBM, the
  amplitude route for the rest) against the float64 reference with psi from
  composite.psi: rule entries exact, the rest to 2e-3 (|r| + 1e-2) (two
  float32 forward passes per replica; a signed output divides by psi of the
  walkers, so pairs with a walker below 1e-2 of the median |psi| are left
  out)."""
  from cgs_vmc_b200 import operators, utils, wavefunctions
  hp = utils.create_hparams(wavefunction_type=kind, **overrides)
  wf = wavefunctions.build_wavefunction(hp).seed(7) if kind not in ('sum', 'prod') else \
      wavefunctions.build_wavefunction(hp)
  n = hp.num_sites
  rng = np.random.default_rng(8)
  regions = _region_list(n, rng)
  cfg = bits.random_sz0_configs(n, 128, rng)
  v = operators.RenyiSwap(regions).local_value(wf, torch.from_numpy(cfg).cuda()).cpu().numpy()
  assert v.shape == (64, len(regions)) and v.dtype == np.float32
  psi_fn = _oracle_psi(wf, kind)
  c1, c2 = cfg[:64], cfg[64:]
  ref = swap_values(c1, c2, regions, psi_fn=psi_fn).numpy()
  broken, trivial = _rules(c1, c2, regions)
  assert not np.any(v[broken])
  np.testing.assert_array_equal(v[~broken & trivial], 1.0)
  psi = np.abs(psi_fn(cfg).numpy())
  good = np.minimum(psi[:64], psi[64:]) >= 1e-2 * np.median(psi)
  assert good.sum() >= 48
  err = np.abs(v - ref)[good]
  assert np.all(err <= 2e-3 * (np.abs(ref[good]) + 1e-2)), float(err.max())


@pytest.mark.parametrize('kind', ['rbm', 'fully_connected'])
def test_exact_purity_over_all_basis_pairs(kind):
  """All 924 x 924 pairs of the 12-site Sz = 0 basis as walkers, weighted by
  pi(s1) pi(s2) from the device amplitudes: the weighted swap values equal
  exact_purity of the 6 prefix regions to 1e-5 on the route RenyiSwap picks
  and, for the pure RBM, on the amplitude route too."""
  from cgs_vmc_b200 import operators, utils, wavefunctions
  n = 12
  hp = utils.create_hparams(wavefunction_type=kind, num_sites=n, num_fc_layers=0 if kind == 'rbm' else 1,
                            fc_layer_size=24 if kind == 'rbm' else 8)
  wf = wavefunctions.build_wavefunction(hp).seed(9)
  cfg = ed.configs_of(ed.sz0_basis(n), n)
  dim = len(cfg)
  assert dim == 924
  i1, i2 = np.repeat(np.arange(dim), dim), np.tile(np.arange(dim), dim)
  basis_packed = packed_cuda(cfg)
  packed = torch.cat([basis_packed[torch.from_numpy(i1).cuda()], basis_packed[torch.from_numpy(i2).cuda()]])
  regions = _prefixes(n)
  op = operators.RenyiSwap(regions)
  from cgs_vmc_b200 import _native
  v = op.local_value(wf, _native.unpack_configs(packed, n)).double()
  logabs, _ = wf.amplitudes(basis_packed)
  pi = torch.exp(2.0 * (logabs.double() - logabs.double().max()))
  pi = pi / pi.sum()
  w = (pi[torch.from_numpy(i1).cuda()] * pi[torch.from_numpy(i2).cuda()])[:, None]
  params = [p.detach().cpu().to(F64) for p in wf.get_trainable_variables()]
  spec = oansatz.AnsatzSpec(kind, n, num_layers=hp.num_fc_layers, layer_size=hp.fc_layer_size,
                            nonlinearity=hp.nonlinearity)
  psi_fn = lambda c: oansatz.psi(spec, params, torch.from_numpy(np.asarray(c)).to(F64), shift=0.0).numpy()
  exact = np.array([exact_purity(n, psi_fn, m) for m in regions])
  assert np.all(exact < 0.999)
  np.testing.assert_allclose((w * v).sum(dim=0).cpu().numpy(), exact, rtol=0, atol=1e-5)
  if kind == 'rbm':
    amp = _amplitude_route(wf.amplitudes, packed, n, op.masks(torch.device('cuda'))).double()
    np.testing.assert_allclose((w * amp).sum(dim=0).cpu().numpy(), exact, rtol=0, atol=1e-5)


def test_evaluator_matches_exact_purity():
  """Monte Carlo (fixed seeds): the 12-site chain's sampled Tr rho_A^2 of the
  6 prefix regions agrees with exact_purity of the same parameters within 4
  error bars per region (error bar as in test_evaluator_correlations_match_exact)."""
  from cgs_vmc_b200 import evaluation, graph_builders, operators, utils, wavefunctions
  from cgs_vmc_b200.session import Session
  n = 12
  graph_builders.reset_num_epochs()
  hp = utils.create_hparams(wavefunction_type='rbm', num_sites=n, num_fc_layers=0, fc_layer_size=24,
                            batch_size=4096, num_equilibration_sweeps=20, num_monte_carlo_sweeps=2,
                            num_evaluation_samples=40)
  wf = wavefunctions.build_wavefunction(hp).seed(6)
  regions = _prefixes(n)
  ev = evaluation.MonteCarloOperatorEvaluator()
  ops = ev.build_eval_ops(wavefunction=wf, operator=operators.RenyiSwap(regions), hparams=hp,
                          shared_resources={})
  values = np.asarray(ev.run_evaluation(ops, Session(), hp, epoch_num=0))
  assert values.shape == (hp.num_evaluation_samples, len(regions)) and values.dtype == np.float64
  spec = oansatz.AnsatzSpec('rbm', n, num_layers=0, layer_size=24)
  params = [p.detach().cpu().to(F64) for p in wf.get_trainable_variables()]
  psi_fn = lambda c: oansatz.psi(spec, params, torch.from_numpy(np.asarray(c)).to(F64), shift=0.0).numpy()
  exact = np.array([exact_purity(n, psi_fn, m) for m in regions])
  err = 2.0 * values.std(axis=0, ddof=1) / np.sqrt(len(values))
  dev = np.abs(values.mean(axis=0) - exact)
  assert np.all(dev < 4.0 * err + 1e-4), (dev / err).max()


def test_api_probes_and_argument_errors():
  from cgs_vmc_b200 import _native
  lib = _native.load()
  vp = ctypes.c_void_p
  n = 12
  conv = oansatz.AnsatzSpec('conv_1d', n, num_layers=1, num_filters=2, kernel_size=3)
  others = [conv, oansatz.AnsatzSpec('fully_connected', n, num_layers=1, layer_size=8),
            oansatz.AnsatzSpec('rbm', n, num_layers=1, layer_size=8)]
  cfg = bits.random_sz0_configs(n, 8, np.random.default_rng(1))
  packed = packed_cuda(cfg)
  regions = _prefixes(n)
  masks = _masks(regions)
  vals = torch.empty(4, 6, device='cuda')
  for spec in others:
    a = make_native(spec, np.zeros(oansatz.num_params(spec), np.float32))
    assert lib.cgsvmc_swap_values(a._handle, None, 0, None, 0, None, None) == _native.ERR_UNSUPPORTED
    assert lib.cgsvmc_swap_values(a._handle, vp(packed.data_ptr()), 4, vp(masks.data_ptr()), 6,
                                  vp(vals.data_ptr()), None) == _native.ERR_UNSUPPORTED
    with pytest.raises(NotImplementedError):
      a.swap_values(packed, masks)
  native, _, _, _ = _rbm(SHAPES['n12_h24'], 34, 1)
  h, p, m, o = native._handle, vp(packed.data_ptr()), vp(masks.data_ptr()), vp(vals.data_ptr())
  # no-ops: no pairs, no regions
  assert lib.cgsvmc_swap_values(h, None, 0, None, 0, None, None) == _native.OK
  assert lib.cgsvmc_swap_values(h, p, 4, None, 0, None, None) == _native.OK
  assert tuple(native.swap_values(packed, masks[:0]).shape) == (4, 0)
  assert tuple(native.swap_values(packed[:0], masks).shape) == (0, 6)
  assert lib.cgsvmc_swap_configs(None, 0, n, None, 0, None, None) == _native.OK
  assert lib.cgsvmc_swap_configs(p, 4, n, None, 0, None, None) == _native.OK
  z = torch.zeros(8, device='cuda')
  assert lib.cgsvmc_swap_values_from_amps(None, 0, n, None, 0, None, None, None, None, None, None) == _native.OK
  assert lib.cgsvmc_swap_values_from_amps(p, 4, n, None, 0, vp(z.data_ptr()), None, None, None, None,
                                          None) == _native.OK
  # INVALID: NULL handles and buffers, negative sizes, bad n_sites
  assert lib.cgsvmc_swap_values(None, p, 4, m, 6, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_swap_values(h, p, -1, m, 6, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_swap_values(h, p, 4, m, -1, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_swap_values(h, None, 4, m, 6, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_swap_values(h, p, 4, None, 6, o, None) == _native.ERR_INVALID
  assert lib.cgsvmc_swap_values(h, p, 4, m, 6, None, None) == _native.ERR_INVALID
  sw = torch.empty(4, 6, 2, 1, dtype=torch.int64, device='cuda')
  args = [p, 4, n, m, 6, vp(sw.data_ptr()), None]
  assert lib.cgsvmc_swap_configs(*args) == _native.OK
  for k, bad_value in ((0, None), (1, -1), (2, 1), (2, 257), (3, None), (4, -1), (5, None)):
    bad = list(args)
    bad[k] = bad_value
    assert lib.cgsvmc_swap_configs(*bad) == _native.ERR_INVALID, (k, bad_value)
  sl = torch.zeros(4, 6, 2, device='cuda')
  args = [p, 4, n, m, 6, vp(z.data_ptr()), None, vp(sl.data_ptr()), None, o, None]
  assert lib.cgsvmc_swap_values_from_amps(*args) == _native.OK
  for k, bad_value in ((0, None), (1, -1), (2, 1), (3, None), (4, -1), (5, None), (7, None), (9, None)):
    bad = list(args)
    bad[k] = bad_value
    assert lib.cgsvmc_swap_values_from_amps(*bad) == _native.ERR_INVALID, (k, bad_value)
  with pytest.raises(ValueError):          # an odd number of walkers
    native.swap_values(packed[:7], masks)
  with pytest.raises(ValueError):          # regions with the wrong number of sites
    from cgs_vmc_b200 import operators, utils, wavefunctions
    wf = wavefunctions.build_wavefunction(utils.create_hparams(wavefunction_type='rbm', num_sites=n,
                                                               num_fc_layers=0, fc_layer_size=8)).seed(1)
    operators.RenyiSwap(_prefixes(n + 2)).local_value(wf, torch.from_numpy(cfg).cuda())
  torch.cuda.synchronize()


def test_mask_bits_above_n_are_ignored():
  """Masks with every bit at or above N set give the same values (both routes)
  and the same swapped configurations as the clean masks."""
  from cgs_vmc_b200 import _native
  for name in ('n12_h24', '10x10_h100'):
    spec = SHAPES[name]
    n = spec.n_sites
    native, _, _, packed = _rbm(spec, 35, 100)
    clean = _masks(_region_list(n, np.random.default_rng(9)))
    words = clean.cpu().numpy().view(np.uint64).copy()
    high = np.zeros(words.shape[1], np.uint64)
    for w in range(words.shape[1]):
      lo = n - 64 * w
      high[w] = np.uint64(0) if lo >= 64 else ~np.uint64(0) if lo <= 0 else ~((np.uint64(1) << np.uint64(lo)) - np.uint64(1))
    assert np.any(high != 0)
    dirty = torch.from_numpy((words | high[None, :]).view(np.int64)).cuda()
    assert bool(torch.equal(native.swap_values(packed, dirty), native.swap_values(packed, clean)))
    assert bool(torch.equal(_native.swap_configs(packed, n, dirty), _native.swap_configs(packed, n, clean)))
    amps = _native_amplitudes(native)
    assert bool(torch.equal(_amplitude_route(amps, packed, n, dirty), _amplitude_route(amps, packed, n, clean)))


def test_ragged_pair_count_beyond_one_grid():
  """3 grids of 148 SMs x 8 CTAs x 8 warps and 37 pairs more: every pair is
  computed (fused against the amplitude route), a sample against the float64
  reference."""
  spec = SHAPES['n12_h24']
  n_pairs = 3 * torch.cuda.get_device_properties(0).multi_processor_count * 64 + 37
  native, params, cfg, packed = _rbm(spec, 36, n_pairs)
  regions = _prefixes(12)
  masks = _masks(regions)
  fused = native.swap_values(packed, masks)
  amp = _amplitude_route(_native_amplitudes(native), packed, 12, masks)
  torch.testing.assert_close(fused, amp, rtol=2e-4, atol=1e-7)
  rows = np.unique(np.concatenate([np.arange(40), np.arange(n_pairs - 40, n_pairs),
                                   np.random.default_rng(2).choice(n_pairs, 200, replace=False)]))
  sub = np.concatenate([cfg[rows], cfg[n_pairs + rows]])
  _check_fused(fused.cpu().numpy()[rows], sub, regions, spec, params)


def test_driver_writes_renyi(tmp_path):
  """run_training (8-site chain, --heisenberg_jx -1), then
  run_energy_evaluation with and without --renyi_file: the same Energy line,
  and an .npz with the prefix regions, the swap means and errors and the
  entropies, all finite."""
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
  path = str(tmp_path / 'renyi.npz')
  with_renyi = subprocess.run(base + ['--renyi_file', path], check=True, env=env, timeout=300,
                              capture_output=True, text=True)
  energy = [l for l in plain.stdout.splitlines() if l.startswith('Energy:')]
  assert len(energy) == 1
  assert energy == [l for l in with_renyi.stdout.splitlines() if l.startswith('Energy:')]
  d = np.load(path)
  assert set(d.files) == {'regions', 'swap_mean', 'swap_stderr', 'entropy', 'entropy_stderr'}
  assert d['regions'].shape == (4, 8)
  np.testing.assert_array_equal(d['regions'], _prefixes(8))
  for key in ('swap_mean', 'swap_stderr', 'entropy', 'entropy_stderr'):
    assert d[key].shape == (4,) and np.all(np.isfinite(d[key])), key
  np.testing.assert_allclose(d['entropy'], -np.log(d['swap_mean']))
