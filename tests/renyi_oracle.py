"""Float64 references for the second Renyi entropy (test infrastructure).

The replica-swap estimator of S2(A) = -log Tr rho_A^2 (Hastings et al. 2010):
for two walkers sigma1, sigma2 from |psi|^2, sigma1' takes sigma1 outside A and
sigma2 inside A, sigma2' the other way round, and
  Tr rho_A^2 = E[ psi(sigma1') psi(sigma2') / (psi(sigma1) psi(sigma2)) ].
The walkers sample psi projected on their S^z sector, so a swapped pair that
leaves it has amplitude 0 (the sector rule); a swap that gives back the pair
is exactly 1.
"""
import numpy as np
import torch

from oracle import ed


def swap_values(configs1, configs2, masks, log_amp_fn=None, psi_fn=None, sector_rule=True):
  """float64 [P, R]: the swap value of pair (configs1[p], configs2[p]) (+-1,
  [P, N]) for each region of masks (bool [R, N]).  The amplitudes come from
  log_amp_fn (z = log psi + const, e.g. oracle.ansatz.log_amp) or psi_fn
  (e.g. oracle.composite.psi).  0 where the replicas hold different numbers of
  up spins in A (unless sector_rule is False: then psi is evaluated outside the
  sector too); exactly 1 where D = (sigma1 != sigma2) & A is empty or holds
  every differing site."""
  c1 = torch.as_tensor(np.asarray(configs1), dtype=torch.float64)
  c2 = torch.as_tensor(np.asarray(configs2), dtype=torch.float64)
  masks = torch.as_tensor(np.asarray(masks, dtype=bool))
  differ = c1 != c2
  out = torch.zeros(c1.shape[0], masks.shape[0], dtype=torch.float64)
  if log_amp_fn is not None:
    z0 = log_amp_fn(c1) + log_amp_fn(c2)
  else:
    p0 = psi_fn(c1) * psi_fn(c2)
  for r in range(masks.shape[0]):
    m = masks[r][None, :]
    d = differ & m
    same_sector = ((c1 > 0) & m).sum(dim=1) == ((c2 > 0) & m).sum(dim=1)
    trivial = ~d.any(dim=1) | (d == differ).all(dim=1)
    s1 = torch.where(m, c2, c1)
    s2 = torch.where(m, c1, c2)
    if log_amp_fn is not None:
      v = torch.exp(log_amp_fn(s1) + log_amp_fn(s2) - z0)
    else:
      v = psi_fn(s1) * psi_fn(s2) / p0
    v = torch.where(trivial, torch.ones_like(v), v)
    if sector_rule:
      v = torch.where(same_sector, v, torch.zeros_like(v))
    out[:, r] = v
  return out


def exact_purity(n_sites, psi_fn, mask):
  """Tr rho_A^2 of psi restricted to the Sz = 0 basis (zero elsewhere), by the
  singular values of psi reshaped over A x complement(A); A = mask (bool [N]).
  psi_fn maps float64 configurations [dim, N] to amplitudes [dim]."""
  basis = ed.sz0_basis(n_sites)
  psi = np.asarray(psi_fn(ed.configs_of(basis, n_sites)), dtype=np.float64)
  mask = np.asarray(mask, dtype=bool)
  inside, outside = np.nonzero(mask)[0], np.nonzero(~mask)[0]
  bits = (basis[:, None] >> np.arange(n_sites)[None, :]) & 1
  row = (bits[:, inside] << np.arange(len(inside))[None, :]).sum(axis=1)
  col = (bits[:, outside] << np.arange(len(outside))[None, :]).sum(axis=1)
  m = np.zeros((1 << len(inside), 1 << len(outside)))
  m[row, col] = psi
  sv = np.linalg.svd(m, compute_uv=False) ** 2
  return float(np.sum(sv ** 2) / np.sum(sv) ** 2)
