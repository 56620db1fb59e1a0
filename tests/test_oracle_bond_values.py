"""CPU checks of the per-bond references (tests/bond_oracle.py) and of the
host-side helpers of the spin-spin correlations: all_pairs, marshall_signs,
structure_factor."""
import itertools
import os
import re

import numpy as np
import pytest
import torch

from bond_oracle import bond_values, exact_bond_expectations
from oracle import ansatz as oansatz
from oracle import bits, ed, hamiltonian
from oracle import lattices as olattices

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = torch.float64


def _lat():
  from cgs_vmc_b200 import lattices
  return lattices


def _rbm(n, h, seed):
  spec = oansatz.AnsatzSpec('rbm', n, num_layers=0, layer_size=h)
  params = oansatz.init_params(spec, seed=seed, bias_scale=0.3, dtype=F64)
  return lambda c: oansatz.log_amp(spec, params, c)


def test_bond_values_sum_to_local_energy():
  n = 12
  fn = _rbm(n, 24, 3)
  rng = np.random.default_rng(1)
  cfg = torch.from_numpy(bits.random_sz0_configs(n, 50, rng)).to(F64)
  pairs = _lat().all_pairs(n)
  jx = rng.choice([-1.0, 0.0, 0.5, 1.0], size=len(pairs))
  jz = rng.uniform(-1.0, 1.0, size=len(pairs))
  v = bond_values(cfg, pairs, jx, jz, fn)
  assert tuple(v.shape) == (50, len(pairs))
  e = hamiltonian.local_energy(cfg, pairs, jx, jz, fn)
  np.testing.assert_allclose(v.sum(dim=1).numpy(), e.numpy(), rtol=1e-12, atol=1e-12)
  # a bond with jx = 0 is its diagonal term alone
  z = jx == 0
  s = cfg.numpy()
  ij = np.asarray(pairs)
  np.testing.assert_array_equal(v.numpy()[:, z], 0.25 * jz[z] * s[:, ij[z, 0]] * s[:, ij[z, 1]])


@pytest.mark.parametrize('kind', ['chain', 'square'])
def test_exact_bond_expectations_sum_to_exact_expectation(kind):
  if kind == 'chain':
    n, bonds = 10, olattices.chain_bonds(10)
  else:
    n, bonds = 16, olattices.square_nn_bonds(4)
  fn = _rbm(n, 8, 5)
  psi_fn = lambda c: torch.exp(fn(torch.from_numpy(np.asarray(c)))).numpy()
  jx, jz = [-1.0] * len(bonds), [1.0] * len(bonds)
  per_bond = exact_bond_expectations(n, bonds, jx, jz, psi_fn)
  assert abs(per_bond.sum() - ed.exact_expectation(n, bonds, jx, jz, psi_fn)) < 1e-10


@pytest.mark.parametrize('kind', ['chain12', 'square4x4'])
def test_marshall_signs_undo_the_rotation(kind):
  """The ground state of the rotated Hamiltonian (jx = -1) with the Marshall
  signs' couplings gives the same correlations as the unrotated (jx = +1)
  ground state with plain S_i . S_j."""
  lat = _lat()
  if kind == 'chain12':
    n, bonds = 12, lat.chain_bonds(12)
  else:
    n, bonds = 16, lat.square_nn_bonds(4)
  nb = len(bonds)
  pairs = np.asarray(lat.all_pairs(n))
  signs = lat.marshall_signs(n, bonds, -1.0, 1.0)
  assert signs.dtype == np.int8 and set(np.unique(signs)) == {-1, 1}
  for i, j in bonds:                      # NN bonds join the two sublattices
    assert signs[i] != signs[j]
  _, basis_r, vec_r = ed.ground_state(n, bonds, [-1.0] * nb, [1.0] * nb)
  _, basis_p, vec_p = ed.ground_state(n, bonds, [1.0] * nb, [1.0] * nb)
  jx_rot = (signs[pairs[:, 0]] * signs[pairs[:, 1]]).astype(np.float64)
  ones = np.ones(len(pairs))
  rotated = exact_bond_expectations(n, pairs, jx_rot, ones, ed.lookup_amplitude(basis_r, vec_r))
  plain = exact_bond_expectations(n, pairs, ones, ones, ed.lookup_amplitude(basis_p, vec_p))
  np.testing.assert_allclose(rotated, plain, rtol=0, atol=1e-10)
  # the naive (unsigned) correlations of the rotated state differ in the transverse part
  naive = exact_bond_expectations(n, pairs, ones, ones, ed.lookup_amplitude(basis_r, vec_r))
  assert np.abs(naive - plain).max() > 0.1


def test_marshall_signs_cases():
  lat = _lat()
  ring5 = lat.chain_bonds(5)
  with pytest.raises(ValueError, match='bipartite'):
    lat.marshall_signs(5, ring5, -1.0, 1.0)
  with pytest.raises(ValueError, match='connect'):
    lat.marshall_signs(6, [(0, 1), (1, 2), (3, 4)], -1.0, 1.0)
  # nothing rotated: the unrotated antiferromagnet, the ferromagnet (-1, -1)
  np.testing.assert_array_equal(lat.marshall_signs(5, ring5, 1.0, 1.0), np.ones(5, np.int8))
  np.testing.assert_array_equal(lat.marshall_signs(5, ring5, -1.0, -1.0), np.ones(5, np.int8))
  # J1-J2: the NN bonds are rotated, the NNN bonds (+j2, +j2) are not and
  # join sites of the same sublattice
  ij, jx, jz = lat.j1j2_couplings(4, 0.5)
  s = lat.marshall_signs(16, ij, jx, jz)
  x, y = np.arange(16) // 4, np.arange(16) % 4
  np.testing.assert_array_equal(s, np.where((x + y) % 2 == 0, 1, -1).astype(np.int8))
  # a 3-column J.txt (jz = |jx|): the negative-jx bonds are the rotated ones
  jx3 = np.array([-1.0, -1.0, -1.0, 0.5], np.float32)
  s = lat.marshall_signs(4, [(0, 1), (1, 2), (2, 3), (0, 2)], jx3, np.abs(jx3))
  np.testing.assert_array_equal(s, np.array([1, -1, 1, -1], np.int8))
  with pytest.raises(ValueError, match='connect'):    # 0-1 and 2-3 rotated, nothing joins them
    lat.marshall_signs(4, [(0, 1), (0, 2), (2, 3), (1, 3)], jx3[[0, 3, 1, 3]], np.abs(jx3[[0, 3, 1, 3]]))


def test_all_pairs():
  pairs = _lat().all_pairs(6)
  assert pairs == list(itertools.combinations(range(6), 2))


@pytest.mark.parametrize('size_x,size_y', [(8, 1), (4, 4), (3, 5)])
def test_structure_factor_matches_brute_force(size_x, size_y):
  n = size_x * size_y
  rng = np.random.default_rng(n)
  c = rng.standard_normal((n, n))
  c = 0.5 * (c + c.T)
  np.fill_diagonal(c, 0.75)
  s = _lat().structure_factor(c, size_x, size_y)
  assert s.shape == (size_x, size_y) and s.dtype == np.float64
  for mx in range(size_x):
    for my in range(size_y):
      q = (2 * np.pi * mx / size_x, 2 * np.pi * my / size_y)
      total = 0j
      for i in range(n):
        for j in range(n):
          d = (i // size_y - j // size_y, i % size_y - j % size_y)
          total += np.exp(1j * (q[0] * d[0] + q[1] * d[1])) * c[i, j]
      assert abs(s[mx, my] - total.real / n) < 1e-12
      assert abs(total.imag) < 1e-9
  assert abs(s.sum() - 0.75 * n) < 1e-9        # sum_q S(q) = sum_i C_ii


def test_structure_factor_of_the_neel_state():
  """C_ij = 3/4 on the diagonal, (-1)^(x+y) / 4 off it: S(pi, pi) = N/4 + 1/2."""
  lat = _lat()
  n = 16
  x, y = np.arange(n) // 4, np.arange(n) % 4
  st = np.where((x + y) % 2 == 0, 1.0, -1.0)
  c = 0.25 * np.outer(st, st)
  np.fill_diagonal(c, 0.75)
  s = lat.structure_factor(c, 4, 4)
  assert abs(s[2, 2] - (0.25 * n + 0.5)) < 1e-12
  with pytest.raises(ValueError):
    lat.structure_factor(c, 4, 3)


def test_both_symbols_are_declared_and_bound():
  from cgs_vmc_b200 import _native
  text = re.sub(r'/\*.*?\*/', '', open(os.path.join(REPO, 'include', 'cgsvmc.h')).read(), flags=re.S)
  for name in ('cgsvmc_bond_values', 'cgsvmc_bond_values_from_amps'):
    assert re.search(r'\b%s\s*\(' % name, text), name
    assert name in _native.EXPORTS
