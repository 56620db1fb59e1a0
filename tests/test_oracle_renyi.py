"""CPU checks of the second-Renyi references (tests/renyi_oracle.py) and of
lattices.prefix_regions: the replica-swap estimator enumerated over every pair
of the Sz = 0 basis equals the exact purity, and only with the sector rule."""
import os
import re

import numpy as np
import torch

from oracle import ansatz as oansatz
from oracle import ed
from oracle import lattices as olattices
from renyi_oracle import exact_purity, swap_values

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = torch.float64


def _prefixes(n):
  from cgs_vmc_b200 import lattices
  return lattices.prefix_regions(n)


def _rbm(n, h, seed):
  spec = oansatz.AnsatzSpec('rbm', n, num_layers=0, layer_size=h)
  params = oansatz.init_params(spec, seed=seed, bias_scale=0.3, dtype=F64)
  return lambda c: oansatz.log_amp(spec, params, torch.as_tensor(np.asarray(c)).to(F64))


def _table_psi(n, basis, vector):
  """psi_fn of a state given on the Sz = 0 basis, zero elsewhere (vectorised)."""
  table = np.zeros(1 << n)
  table[basis] = vector
  table = torch.from_numpy(table)
  weights = torch.from_numpy(1 << np.arange(n, dtype=np.int64))

  def psi_fn(c):
    c = torch.as_tensor(np.asarray(c))
    return table[((c > 0).to(torch.int64) * weights).sum(dim=1)]
  return psi_fn


def _enumerated(n, masks, log_amp_fn=None, psi_fn=None, sector_rule=True):
  """sum over all pairs of the Sz = 0 basis of pi(s1) pi(s2) swap(s1, s2)."""
  cfg = ed.configs_of(ed.sz0_basis(n), n)
  if log_amp_fn is not None:
    z = log_amp_fn(cfg).numpy()
    pi = np.exp(2.0 * (z - z.max()))
  else:
    pi = np.asarray(psi_fn(cfg), dtype=np.float64) ** 2
  pi = pi / pi.sum()
  dim = len(cfg)
  total = np.zeros(len(masks))
  block = max(1, 200000 // dim)
  for a0 in range(0, dim, block):
    a = np.arange(a0, min(dim, a0 + block))
    i1, i2 = np.repeat(a, dim), np.tile(np.arange(dim), len(a))
    v = swap_values(cfg[i1], cfg[i2], masks, log_amp_fn=log_amp_fn, psi_fn=psi_fn,
                    sector_rule=sector_rule).numpy()
    total += ((pi[i1] * pi[i2])[:, None] * v).sum(axis=0)
  return total


def _regions_10():
  rng = np.random.default_rng(4)
  masks = list(_prefixes(10)) + [rng.random(10) < 0.5 for _ in range(3)]
  masks.append(np.array([i % 2 == 0 for i in range(10)]))
  return np.array(masks)


def test_enumerated_estimator_equals_exact_purity_random_rbm():
  n = 10
  fn = _rbm(n, 12, 3)
  psi_fn = lambda c: torch.exp(fn(c))
  masks = _regions_10()
  est = _enumerated(n, masks, log_amp_fn=fn)
  exact = np.array([exact_purity(n, psi_fn, m) for m in masks])
  np.testing.assert_allclose(est, exact, rtol=0, atol=1e-12)
  assert np.all(exact < 1.0 - 1e-3) and np.all(exact > 0.0)


def test_enumerated_estimator_equals_exact_purity_chain12_ground_state():
  n = 12
  bonds = olattices.chain_bonds(n)
  _, basis, vec = ed.ground_state(n, bonds, [1.0] * n, [1.0] * n)
  psi_fn = _table_psi(n, basis, vec)
  masks = _prefixes(n)
  est = _enumerated(n, masks, psi_fn=psi_fn)
  exact = np.array([exact_purity(n, psi_fn, m) for m in masks])
  np.testing.assert_allclose(est, exact, rtol=0, atol=1e-12)
  s2 = -np.log(exact)
  assert abs(s2[0] - np.log(2.0)) < 1e-10   # the singlet leaves one site maximally mixed
  assert np.all(np.diff(s2[1::2]) > 0)      # S2(l) of even l grows up to the half chain


def test_without_the_sector_rule_the_estimator_is_another_state():
  """psi evaluated outside the walkers' sector measures a different state."""
  n = 10
  fn = _rbm(n, 12, 3)
  psi_fn = lambda c: torch.exp(fn(c))
  masks = _regions_10()
  naive = _enumerated(n, masks, log_amp_fn=fn, sector_rule=False)
  exact = np.array([exact_purity(n, psi_fn, m) for m in masks])
  assert np.abs(naive - exact).max() > 1e-2, np.abs(naive - exact).max()


def test_region_and_complement_have_equal_purity():
  n = 12
  fn = _rbm(n, 16, 7)
  psi_fn = lambda c: torch.exp(fn(c))
  rng = np.random.default_rng(2)
  for m in list(_prefixes(n)) + [rng.random(n) < 0.5 for _ in range(4)]:
    assert abs(exact_purity(n, psi_fn, m) - exact_purity(n, psi_fn, ~m)) < 1e-12


def test_single_configuration_has_zero_entropy():
  n = 10
  basis = ed.sz0_basis(n)
  vec = np.zeros(len(basis))
  vec[17] = 1.0
  psi_fn = _table_psi(n, basis, vec)
  rng = np.random.default_rng(3)
  masks = np.array(list(_prefixes(n)) + [rng.random(n) < 0.5 for _ in range(3)])
  for m in masks:
    assert abs(exact_purity(n, psi_fn, m) - 1.0) < 1e-15
  cfg = ed.configs_of(basis[17:18], n)
  np.testing.assert_array_equal(swap_values(cfg, cfg, masks, psi_fn=psi_fn).numpy(), np.ones((1, len(masks))))


def test_swap_values_rules():
  """The sector rule gives 0, an empty or whole D gives exactly 1."""
  n = 6
  fn = _rbm(n, 8, 1)
  c1 = np.array([[1, 1, 1, -1, -1, -1]], np.float64)
  c2 = np.array([[-1, 1, 1, 1, -1, -1]], np.float64)     # differ at sites 0 and 3
  masks = np.array([[1, 0, 0, 0, 0, 0],                   # one up in c1, none in c2: 0
                    [0, 1, 1, 0, 1, 1],                   # D empty: 1
                    [1, 0, 0, 1, 0, 0],                   # D holds every differing site: 1
                    [1, 1, 1, 1, 1, 1],                   # the full region: 1
                    [1, 1, 0, 0, 0, 0],                   # sector broken: 0
                    [1, 1, 0, 1, 0, 0]], bool)            # D = {0, 3} again: 1
  v = swap_values(c1, c2, masks, log_amp_fn=fn).numpy()
  np.testing.assert_array_equal(v, [[0.0, 1.0, 1.0, 1.0, 0.0, 1.0]])
  c3 = np.array([[-1, 1, -1, 1, 1, -1]], np.float64)     # differs from c1 at 0, 2, 3, 4
  m = np.array([[1, 0, 0, 0, 1, 0]], bool)               # D = {0, 4}: one up each side, a real swap
  fn64 = lambda c: torch.exp(fn(c))
  got = swap_values(c1, c3, m, log_amp_fn=fn).numpy()
  s1, s2 = np.where(m, c3, c1), np.where(m, c1, c3)
  want = (fn64(s1) * fn64(s2) / (fn64(c1) * fn64(c3))).numpy()
  np.testing.assert_allclose(got[:, 0], want, rtol=1e-12)
  np.testing.assert_allclose(swap_values(c1, c3, m, psi_fn=fn64).numpy(), got, rtol=1e-12)


def test_prefix_regions():
  r = _prefixes(9)
  assert r.shape == (4, 9) and r.dtype == bool
  for l in range(1, 5):
    np.testing.assert_array_equal(r[l - 1], np.arange(9) < l)
  assert _prefixes(36).shape == (18, 36)
  assert _prefixes(36)[5].sum() == 6        # 6 x 6: the first row is a cylinder of one row


def test_three_symbols_are_declared_and_bound():
  from cgs_vmc_b200 import _native
  text = re.sub(r'/\*.*?\*/', '', open(os.path.join(REPO, 'include', 'cgsvmc.h')).read(), flags=re.S)
  for name in ('cgsvmc_swap_values', 'cgsvmc_swap_configs', 'cgsvmc_swap_values_from_amps'):
    assert re.search(r'\b%s\s*\(' % name, text), name
    assert name in _native.EXPORTS
