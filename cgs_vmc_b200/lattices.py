"""Bond lists of the lattices the drivers and benchmarks use (SURVEY.md 8(d)):
periodic chain (run_training.py:109), periodic L x L square lattice with site
index s = x * size_y + y (the reshape of wavefunctions.py:593), nearest and
next-nearest neighbours, and the coupling arrays of the Heisenberg / J1-J2
models in the reference's matrix-element convention (operators.py:165-169)."""
import numpy as np


def chain_bonds(n_sites):
  return [(i, (i + 1) % n_sites) for i in range(n_sites)]


def square_nn_bonds(size_x, size_y=None):
  size_y = size_x if size_y is None else size_y
  bonds = []
  for x in range(size_x):
    for y in range(size_y):
      s = x * size_y + y
      bonds.append((s, ((x + 1) % size_x) * size_y + y))
      bonds.append((s, x * size_y + (y + 1) % size_y))
  return bonds


def square_nnn_bonds(size_x, size_y=None):
  size_y = size_x if size_y is None else size_y
  bonds = []
  for x in range(size_x):
    for y in range(size_y):
      s = x * size_y + y
      xp = (x + 1) % size_x
      bonds.append((s, xp * size_y + (y + 1) % size_y))
      bonds.append((s, xp * size_y + (y - 1) % size_y))
  return bonds


def heisenberg_couplings(bonds, j_x=-1.0, j_z=1.0):
  """(ij int32 [n, 2], jx float32 [n], jz float32 [n]) with uniform couplings."""
  ij = np.asarray(bonds, dtype=np.int32).reshape(-1, 2)
  n = ij.shape[0]
  return ij, np.full(n, j_x, dtype=np.float32), np.full(n, j_z, dtype=np.float32)


def all_pairs(n_sites):
  """Every site pair (i, j) with i < j: the bonds of the full correlation
  matrix (operators.HeisenbergBonds)."""
  return [(i, j) for i in range(n_sites) for j in range(i + 1, n_sites)]


def prefix_regions(n_sites):
  """bool [N // 2, N]: row l - 1 holds sites 0 .. l - 1 (operators.RenyiSwap).
  On the periodic chain these are the intervals of the S2(l) curve; on the
  row-major square lattice (s = x * size_y + y) the prefixes of k * size_y
  sites are cylinders of k rows."""
  lengths = np.arange(1, n_sites // 2 + 1)
  return np.arange(n_sites)[None, :] < lengths[:, None]


def marshall_signs(n_sites, bonds, j_x, j_z):
  """int8 [N] of +-1: the sublattice signs of the Marshall rotation a
  Hamiltonian was written in.  Bonds with j_x * j_z < 0 are the rotated ones
  (--heisenberg_jx -1 gives (-1, +1)); the ferromagnet (-1, -1) and
  same-sublattice J2 bonds (+j2, +j2) are not.  The rotated bonds are
  2-coloured; without any the result is all +1.  In the rotated frame
  S_i . S_j has j_x = sign_i sign_j and j_z = 1.  Raises ValueError when the
  rotated bonds are not bipartite or do not connect every site."""
  ij = np.asarray(bonds, dtype=np.int64).reshape(-1, 2)
  n = ij.shape[0]
  jx = np.broadcast_to(np.asarray(j_x, dtype=np.float64), (n,))
  jz = np.broadcast_to(np.asarray(j_z, dtype=np.float64), (n,))
  rotated = ij[jx * jz < 0]
  signs = np.ones(n_sites, dtype=np.int8)
  if len(rotated) == 0:
    return signs
  adjacency = [[] for _ in range(n_sites)]
  for i, j in rotated:
    adjacency[i].append(j)
    adjacency[j].append(i)
  colour = np.zeros(n_sites, dtype=np.int8)     # 0: not reached yet
  colour[0] = 1
  stack = [0]
  while stack:
    i = stack.pop()
    for j in adjacency[i]:
      if colour[j] == 0:
        colour[j] = -colour[i]
        stack.append(j)
      elif colour[j] == colour[i]:
        raise ValueError('the Marshall-rotated bonds (j_x * j_z < 0) are not bipartite')
  if (colour == 0).any():
    raise ValueError('the Marshall-rotated bonds (j_x * j_z < 0) do not connect every site')
  signs[:] = colour
  return signs


def structure_factor(corr, size_x, size_y=1):
  """S(q) = (1/N) sum_ij cos(q . (r_i - r_j)) C_ij at every lattice momentum
  q = (2 pi m / size_x, 2 pi n / size_y) of a periodic size_x x size_y lattice
  (site s = x * size_y + y; a chain is size_y = 1).  corr: the symmetric
  [N, N] correlation matrix with C_ii = 3/4.  Returns float64 [size_x, size_y];
  S(pi, pi) / N is the squared staggered magnetisation."""
  corr = np.asarray(corr, dtype=np.float64)
  n = size_x * size_y
  if corr.shape != (n, n):
    raise ValueError('corr has shape %s, expected (%d, %d)' % (corr.shape, n, n))
  sites = np.arange(n)
  x, y = sites // size_y, sites % size_y
  qx = 2.0 * np.pi * np.arange(size_x) / size_x
  qy = 2.0 * np.pi * np.arange(size_y) / size_y
  # phase[q, s] = exp(i q . r_s); C symmetric and real, so the cosine sum is
  # the real part of phase C phase^H
  phase = np.exp(1j * (qx[:, None, None] * x[None, None, :] + qy[None, :, None] * y[None, None, :]))
  phase = phase.reshape(n, n)
  s = np.einsum('qi,ij,qj->q', phase, corr, phase.conj()).real / n
  return s.reshape(size_x, size_y)


def j1j2_couplings(size, j2=0.5):
  """NN bonds with (jx, jz) = (-1, 1) (Marshall-rotated) and NNN bonds with
  (+j2, j2): the rotation leaves same-sublattice bonds unchanged."""
  nn, nnn = square_nn_bonds(size), square_nnn_bonds(size)
  ij = np.asarray(nn + nnn, dtype=np.int32).reshape(-1, 2)
  jx = np.concatenate([np.full(len(nn), -1.0), np.full(len(nnn), j2)]).astype(np.float32)
  jz = np.concatenate([np.full(len(nn), 1.0), np.full(len(nnn), j2)]).astype(np.float32)
  return ij, jx, jz
