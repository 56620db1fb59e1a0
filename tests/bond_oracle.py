"""Float64 references for the per-bond local values (test infrastructure).

The per-bond forms of oracle.hamiltonian.local_energy and
oracle.ed.exact_expectation: each bond's term is kept instead of summed.  With
site pairs and jx = jz = 1 the terms are the spin-spin correlations S_i . S_j.
"""
import numpy as np
import torch

from oracle import ed, hamiltonian


def bond_values(configs, bonds_ij, jx, jz, log_amp_fn):
  """[B, n_bonds]: jz/4 s_i s_j + jx/2 [s_i != s_j] exp(z(flipped) - z) per
  bond; summed over bonds this is hamiltonian.local_energy.  The ratio is
  evaluated only on antiparallel bonds with jx != 0."""
  dtype = log_amp_fn(configs[:1]).dtype
  cfg = configs.to(dtype)
  z = log_amp_fn(cfg)
  out = torch.zeros(cfg.shape[0], len(bonds_ij), dtype=dtype)
  for k in range(len(bonds_ij)):
    d, pref, updated = hamiltonian.bond_terms(cfg, bonds_ij[k], float(jx[k]), float(jz[k]))
    out[:, k] = d
    act = pref != 0
    if bool(act.any()):
      zf = log_amp_fn(updated[act])
      out[act, k] = out[act, k] + pref[act] * torch.exp(zf - z[act])
  return out


def exact_bond_expectations(n_sites, bonds_ij, jx, jz, psi_fn):
  """<psi|term_k|psi> / <psi|psi> per bond over the Sz = 0 basis, with
  term_k = jz_k S^z_i S^z_j + jx_k (S^x_i S^x_j + S^y_i S^y_j); summed over
  bonds this is ed.exact_expectation.  psi_fn maps float64 configurations
  [dim, N] to amplitudes [dim]."""
  basis = ed.sz0_basis(n_sites)
  index = {int(s): k for k, s in enumerate(basis)}
  psi = np.asarray(psi_fn(ed.configs_of(basis, n_sites)), dtype=np.float64)
  norm = float(psi @ psi)
  bits = (basis[:, None] >> np.arange(n_sites)[None, :]) & 1
  ij = np.asarray(bonds_ij, dtype=np.int64).reshape(-1, 2)
  out = np.zeros(len(ij))
  for k, (i, j) in enumerate(ij):
    same = bits[:, i] == bits[:, j]
    diag = 0.25 * float(jz[k]) * np.where(same, 1.0, -1.0)
    val = float(np.sum(diag * psi * psi))
    if float(jx[k]) != 0.0:
      anti = np.nonzero(~same)[0]
      flipped = np.array([index[int(basis[a]) ^ ((1 << int(i)) | (1 << int(j)))] for a in anti], dtype=np.int64)
      val += 0.5 * float(jx[k]) * float(np.sum(psi[flipped] * psi[anti]))
    out[k] = val / norm
  return out
