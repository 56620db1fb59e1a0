"""Mirror of the reference's operators.py on the CUDA library
(operators.py:13-287): Operator interface, HeisenbergBond and
HeisenbergHamiltonian.  j_x / j_z may be scalars (the reference) or one value
per bond (J1-J2; the reference expresses that as a sum of HeisenbergBond)."""
import numpy as np
import torch

from . import _native


class Operator:
  """Operator base class (operators.py:13-87)."""

  def build(self, wavefunction, inputs, psi=None):
    raise NotImplementedError

  def local_value(self, wavefunction, inputs, psi=None):
    raise NotImplementedError

  def apply_in_place(self, wavefunction, inputs, psi=None):
    raise NotImplementedError

  def apply(self, wavefunction):
    raise NotImplementedError


# values per chunk of walkers in _BondListOperator.bond_values (128 MB of float32);
# RenyiSwap keeps its swapped configurations per chunk under the same count
_BOND_VALUES_CHUNK = 1 << 25


class _BondListOperator(Operator):
  def __init__(self, bonds, j_x, j_z):
    self._bonds_list = [(int(a), int(b)) for a, b in bonds]
    n = len(self._bonds_list)
    self._j_x = j_x
    self._j_z = j_z
    self._jx_array = np.ascontiguousarray(np.broadcast_to(np.asarray(j_x, dtype=np.float32), (n,)))
    self._jz_array = np.ascontiguousarray(np.broadcast_to(np.asarray(j_z, dtype=np.float32), (n,)))
    self._native = {}

  def native(self, n_sites):
    if n_sites not in self._native:
      self._native[n_sites] = _native.Hamiltonian(
          np.asarray(self._bonds_list, dtype=np.int32).reshape(-1, 2), self._jx_array,
          self._jz_array, n_sites)
    return self._native[n_sites]

  def _evaluate(self, wavefunction, inputs):
    """(E_loc, log|psi|, sign psi, diag, offdiag / psi) on the device."""
    from . import graph_builders
    n = inputs.shape[1]
    packed = graph_builders.as_packed(inputs, n)
    ham = self.native(n)
    if wavefunction.fast_path:          # fused local-energy kernels
      a = wavefunction.native(n)
      e, z, diag, off = a.local_energy(ham, packed, want_parts=True)
      return e, z - wavefunction._exp_norm_shift, torch.ones_like(z), diag, off
    # signed / composite amplitudes: psi on the bond-flipped configurations of
    # cgsvmc_flip_enum through the parts' kernels, combined on the device
    wavefunction.connect(n)
    b = packed.shape[0]
    logabs, sign = wavefunction.amplitudes(packed)
    _, flipped = ham.flip_enum(packed, want_flipped=True)
    fl, fs = wavefunction.amplitudes(flipped.reshape(b * ham.n_bonds, -1))
    logabs, sign = logabs.float().contiguous(), sign.float().contiguous()
    e, diag, off = _native.local_energy_from_amps(
        ham, packed, logabs, sign, fl.float().reshape(b, ham.n_bonds).contiguous(),
        fs.float().reshape(b, ham.n_bonds).contiguous(), want_parts=True)
    return e, logabs, sign, diag, off

  def bond_values(self, wavefunction, inputs):
    """float32 [B, n_bonds]: each bond's term of the local value,
    jz/4 s_i s_j + jx/2 [s_i != s_j] psi(flipped) / psi.  A single pure RBM
    runs the fused kernel; every other wavefunction goes through psi on the
    bond-flipped configurations, like _evaluate.  Walkers are processed in
    chunks of at most _BOND_VALUES_CHUNK values (the flipped configurations of
    the amplitude route scale with it too)."""
    from . import graph_builders
    n = inputs.shape[1]
    packed = graph_builders.as_packed(inputs, n)
    ham = self.native(n)
    b, k = packed.shape[0], ham.n_bonds
    out = torch.empty(b, k, dtype=torch.float32, device=packed.device)
    if b == 0 or k == 0:
      return out
    fused = None
    if wavefunction.fast_path:
      fused = wavefunction.native(n)
      try:
        fused.bond_values(ham, packed[:0])        # no walkers: probes for support
      except NotImplementedError:
        fused = None
    else:
      wavefunction.connect(n)
    chunk = max(1, _BOND_VALUES_CHUNK // k)
    for c0 in range(0, b, chunk):
      pc, oc = packed[c0:c0 + chunk], out[c0:c0 + chunk]
      if fused is not None:
        fused.bond_values(ham, pc, out=oc)
        continue
      bc = pc.shape[0]
      logabs, sign = wavefunction.amplitudes(pc)
      _, flipped = ham.flip_enum(pc, want_flipped=True)
      fl, fs = wavefunction.amplitudes(flipped.reshape(bc * k, -1))
      _native.bond_values_from_amps(
          ham, pc, logabs.float().contiguous(), sign.float().contiguous(),
          fl.float().reshape(bc, k).contiguous(), fs.float().reshape(bc, k).contiguous(), out=oc)
    return out

  def build(self, wavefunction, inputs, psi=None):
    """(diagonal matrix element, off-diagonal term) of <R|O|psi>
    (operators.py:137-169, 227-247)."""
    _, logpsi, sign, diag, off = self._evaluate(wavefunction, inputs)
    return diag, off * sign * torch.exp(logpsi)

  def local_value(self, wavefunction, inputs, psi=None):
    """<R|O|psi> / <R|psi> (operators.py:171-181, 249-259)."""
    return self._evaluate(wavefunction, inputs)[0]

  def apply_in_place(self, wavefunction, inputs, psi=None):
    """<R|O|psi> (operators.py:183-193, 261-271)."""
    e, logpsi, sign, _, _ = self._evaluate(wavefunction, inputs)
    return e * sign * torch.exp(logpsi)

  def apply(self, wavefunction):
    raise NotImplementedError('Operator.apply builds a TransformedWavefunction (operators.py:90-125); '
                              'no driver uses it and it is outside the CUDA hot path')


class HeisenbergBond(_BondListOperator):
  """S_i . S_j on one bond (operators.py:128-210)."""

  def __init__(self, bond, j_x, j_z):
    super().__init__([bond], j_x, j_z)
    self._bond = tuple(bond)


class HeisenbergHamiltonian(_BondListOperator):
  """Heisenberg Hamiltonian on a bond list (operators.py:212-287)."""

  def __init__(self, bonds, j_x, j_z):
    super().__init__(bonds, j_x, j_z)
    self._heisenberg_bonds = self._bonds_list


class HeisenbergBonds(_BondListOperator):
  """Many HeisenbergBond at once: the local value is the vector of the bonds'
  local values, float32 [B, n_bonds], from one pass over the walkers.  With
  site pairs and j_x = j_z = 1 these are the spin-spin correlations
  S_i . S_j (lattices.all_pairs; in a Marshall-rotated frame j_x = sign_i
  sign_j, lattices.marshall_signs)."""

  def local_value(self, wavefunction, inputs, psi=None):
    return self.bond_values(wavefunction, inputs)

  def build(self, wavefunction, inputs, psi=None):
    raise NotImplementedError('HeisenbergBonds has a vector local value only')

  def apply_in_place(self, wavefunction, inputs, psi=None):
    raise NotImplementedError('HeisenbergBonds has a vector local value only')


class RenyiSwap(Operator):
  """The replica-swap estimator of the second Renyi entropy
  S2(A) = -log Tr rho_A^2 for every region A of `regions` (bool [R, N]).
  local_value pairs the walkers (row p with row P + p, P = B // 2; an odd
  last walker is unused) and returns float32 [P, R]: psi(sigma1')
  psi(sigma2') / (psi(sigma1) psi(sigma2)) for the pair with its spins in A
  exchanged, 0 where the replicas hold different numbers of up spins in A
  (the swapped pair leaves the sampled S^z sector) and exactly 1 where the
  swap gives back the pair (include/cgsvmc.h, cgsvmc_swap_values).  Its mean
  is Tr rho_A^2; MonteCarloOperatorEvaluator averages it over pairs."""

  def __init__(self, regions):
    regions = np.asarray(regions, dtype=bool)
    if regions.ndim != 2:
      raise ValueError('regions must be a bool [n_regions, n_sites] array, got shape %s' % (regions.shape,))
    self.regions = regions
    self._masks = {}

  def masks(self, device):
    """int64-viewed uint64 [R, W] site masks on `device` (packed bit convention)."""
    key = str(device)
    if key not in self._masks:
      r, n = self.regions.shape
      words = np.zeros((r, _native.n_words(n)), dtype=np.uint64)
      for i in range(n):
        words[:, i >> 6] |= self.regions[:, i].astype(np.uint64) << np.uint64(i & 63)
      self._masks[key] = torch.from_numpy(words.view(np.int64)).to(device)
    return self._masks[key]

  def local_value(self, wavefunction, inputs, psi=None):
    """float32 [B // 2, R].  A single pure RBM runs the fused kernel; every
    other wavefunction goes through psi on the swapped pairs.  Pairs are
    processed in chunks of at most _BOND_VALUES_CHUNK swapped configurations."""
    from . import graph_builders
    n = inputs.shape[1]
    if n != self.regions.shape[1]:
      raise ValueError('regions have %d sites, the walkers %d' % (self.regions.shape[1], n))
    packed = graph_builders.as_packed(inputs, n)
    p = packed.shape[0] // 2
    masks = self.masks(packed.device)
    r = masks.shape[0]
    out = torch.empty(p, r, dtype=torch.float32, device=packed.device)
    if p == 0 or r == 0:
      return out
    fused = None
    if wavefunction.fast_path:
      fused = wavefunction.native(n)
      try:
        fused.swap_values(packed[:0], masks)       # no pairs: probes for support
      except NotImplementedError:
        fused = None
    else:
      wavefunction.connect(n)
    chunk = max(1, _BOND_VALUES_CHUNK // (2 * r))
    for c0 in range(0, p, chunk):
      c1 = min(p, c0 + chunk)
      pc = packed[:2 * p] if c1 - c0 == p else torch.cat([packed[c0:c1], packed[p + c0:p + c1]])
      oc = out[c0:c1]
      if fused is not None:
        fused.swap_values(pc, masks, out=oc)
        continue
      logabs, sign = wavefunction.amplitudes(pc)
      swapped = _native.swap_configs(pc, n, masks)
      sl, ss = wavefunction.amplitudes(swapped.reshape((c1 - c0) * r * 2, -1))
      _native.swap_values_from_amps(
          pc, n, masks, logabs.float().contiguous(), sign.float().contiguous(),
          sl.float().reshape(c1 - c0, r, 2).contiguous(), ss.float().reshape(c1 - c0, r, 2).contiguous(),
          out=oc)
    return out

  def build(self, wavefunction, inputs, psi=None):
    raise NotImplementedError('RenyiSwap has a per-pair local value only')

  def apply_in_place(self, wavefunction, inputs, psi=None):
    raise NotImplementedError('RenyiSwap has a per-pair local value only')
