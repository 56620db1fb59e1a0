"""Float64 restatement of one cgsvmc_batch_steps call for the pure RBM (oracle
side; test infrastructure).

One call runs n_iters batch iterations.  Iteration i evaluates every walker at
its current configuration (log-amplitude z, local energy, the gradient sums'
O_b) and then runs n_steps Metropolis exchange steps on it with the Philox
steps step0 + i n_steps + k, k = 0 .. n_steps - 1:

  * the proposal is oracle.philox.fast_proposal: counter (step_lo, step_hi,
    walker_lo, walker_hi) with walker = walker_id0 + b, key = seed; the k_up-th
    up site is lowered and the k_dn-th down site raised;
  * a walker with no up or no down site proposes nothing and accepts nothing;
  * the move is accepted iff exp(2 dz) > u.

Next to every decision the oracle reports its margin |exp(2 dz) - u| / exp(2 dz)
so that a test can recognise the decisions that float32 rounding may flip.

theta = W^T sigma + c is kept in float64 and updated on accepted moves (it is
rebuilt from the spins at the start of every iteration); log-ratios and local
energies are differences of log cosh.  This is a restatement of the
semantics, not of the kernel's tables.
"""
import dataclasses
import math

import numpy as np

from . import philox

_LN2 = math.log(2.0)


def _log_cosh(x):
  ax = np.abs(x)
  return ax + np.log1p(np.exp(-2.0 * ax)) - _LN2


class Rbm:
  """A pure RBM (no hidden layers) from the flat float parameter layout
  a[N], a0[1], W[N, H], c[H] (include/cgsvmc.h), in float64."""

  def __init__(self, flat, n_sites, n_hidden):
    flat = np.asarray(flat, dtype=np.float64).reshape(-1)
    n, h = n_sites, n_hidden
    if flat.size != n + 1 + n * h + h:
      raise ValueError('expected %d parameters, got %d' % (n + 1 + n * h + h, flat.size))
    self.n_sites, self.n_hidden = n, h
    self.a = flat[:n]
    self.a0 = float(flat[n])
    self.w = flat[n + 1:n + 1 + n * h].reshape(n, h)
    self.c = flat[n + 1 + n * h:]

  @property
  def n_params(self):
    return self.n_sites + 1 + self.n_sites * self.n_hidden + self.n_hidden

  def theta(self, configs):
    return np.asarray(configs, dtype=np.float64) @ self.w + self.c

  def log_amp(self, configs, theta=None):
    configs = np.asarray(configs, dtype=np.float64)
    theta = self.theta(configs) if theta is None else theta
    return configs @ self.a + self.a0 + _log_cosh(theta).sum(axis=1)

  def exchange_log_ratio(self, theta, up, dn):
    """z(sigma') - z(sigma) for sigma' = sigma with the up site `up` lowered
    and the down site `dn` raised (one pair per row of theta); returns the
    change of theta as well."""
    dtheta = 2.0 * (self.w[dn] - self.w[up])
    dz = 2.0 * (self.a[dn] - self.a[up]) + (_log_cosh(theta + dtheta) - _log_cosh(theta)).sum(axis=1)
    return dz, dtheta

  def local_energy(self, configs, bonds_ij, jx, jz, theta=None):
    """(E_loc, diag, E_abs) with E_loc = sum_k jz_k/4 s_i s_j + jx_k/2
    [s_i != s_j] psi(flip_k)/psi (operators.py:249-259) and E_abs the same sum
    with |jx|, |jz| (the scale of the float32 rounding of E_loc)."""
    configs = np.asarray(configs, dtype=np.float64)
    theta = self.theta(configs) if theta is None else theta
    ij = np.asarray(bonds_ij, dtype=np.int64).reshape(-1, 2)
    jx = np.broadcast_to(np.asarray(jx, dtype=np.float64), (ij.shape[0],))
    jz = np.broadcast_to(np.asarray(jz, dtype=np.float64), (ij.shape[0],))
    b = configs.shape[0]
    diag = np.zeros(b)
    diag_abs = np.zeros(b)
    off = np.zeros(b)
    off_abs = np.zeros(b)
    for k in range(ij.shape[0]):
      i, j = ij[k]
      si, sj = configs[:, i], configs[:, j]
      diag += 0.25 * jz[k] * si * sj
      diag_abs += 0.25 * abs(jz[k])
      rows = np.flatnonzero(si != sj)
      if rows.size == 0 or jx[k] == 0.0:
        continue
      up = np.where(si[rows] > 0, i, j)
      dn = np.where(si[rows] > 0, j, i)
      dz, _ = self.exchange_log_ratio(theta[rows], up, dn)
      r = np.exp(dz)
      off[rows] += 0.5 * jx[k] * r
      off_abs[rows] += 0.5 * abs(jx[k]) * r
    return diag + off, diag, diag_abs + off_abs

  def grad_sums(self, configs, weights):
    """S[k] = sum_b weights[k, b] O_b with O_b = d z_b / d params (flat
    layout), and the bound sum_b |weights[k, b]| |O_b| per entry."""
    configs = np.asarray(configs, dtype=np.float64)
    weights = np.asarray(weights, dtype=np.float64).reshape(-1, configs.shape[0])
    t = np.tanh(self.theta(configs))
    out = []
    for w, s, o_t in ((weights, configs, t), (np.abs(weights), np.abs(configs), np.abs(t))):
      rows = []
      for k in range(w.shape[0]):
        rows.append(np.concatenate([w[k] @ s, [w[k].sum()], ((s * w[k][:, None]).T @ o_t).reshape(-1),
                                    w[k] @ o_t]))
      out.append(np.stack(rows))
    return out[0], out[1]


@dataclasses.dataclass
class ChainResult:
  configs: np.ndarray     # int8 [n_iters, B, N]: the walkers at the start of every iteration
  log_amp: np.ndarray     # [n_iters, B]: z there
  e_loc: np.ndarray       # [n_iters, B]: E_loc there
  e_abs: np.ndarray       # [n_iters, B]: E_loc with |couplings| (rounding scale)
  diag: np.ndarray        # [n_iters, B]: diagonal part of E_loc
  accepted: np.ndarray    # int64 [n_iters, B]: accepted moves of the iteration's sweep
  margin: np.ndarray      # [n_iters, n_steps, B]: |exp(2 dz) - u| / exp(2 dz); inf where nothing was proposed
  final: np.ndarray       # int8 [B, N]: the walkers after the last sweep


def kth_set(mask, k):
  """Index of the k-th (0-based) True entry of every row of a bool [B, N]
  array (rows with fewer than k + 1 return 0)."""
  return np.argmax(np.cumsum(mask, axis=1) > np.asarray(k)[:, None], axis=1)


def run_chain(rbm, configs, bonds_ij, jx, jz, seed, walker_id0, step0, n_steps, n_iters):
  """One cgsvmc_batch_steps call: see the module docstring."""
  cfg = np.array(configs, dtype=np.int8)
  b, n = cfg.shape
  walker_ids = np.uint64(walker_id0) + np.arange(b, dtype=np.uint64)
  shape = (n_iters, b)
  res = ChainResult(np.empty((n_iters, b, n), np.int8), np.empty(shape), np.empty(shape), np.empty(shape),
                    np.empty(shape), np.zeros(shape, np.int64), np.full((n_iters, n_steps, b), np.inf), None)
  rows = np.arange(b)
  for it in range(n_iters):
    res.configs[it] = cfg
    theta = rbm.theta(cfg)
    res.log_amp[it] = rbm.log_amp(cfg, theta)
    res.e_loc[it], res.diag[it], res.e_abs[it] = rbm.local_energy(cfg, bonds_ij, jx, jz, theta)
    for k in range(n_steps):
      step = int(step0) + it * int(n_steps) + k
      r0, r1, r2, _ = philox.walker_step_random(seed, walker_ids, step)
      up_mask = cfg > 0
      n_up = up_mask.sum(axis=1).astype(np.uint64)
      n_dn = np.uint64(n) - n_up
      k_up = (r0 * n_up) >> np.uint64(32)
      k_dn = (r1 * n_dn) >> np.uint64(32)
      u = philox.u32_to_unit(r2)
      can = (n_up > 0) & (n_dn > 0)
      up = kth_set(up_mask, k_up)
      dn = kth_set(~up_mask, k_dn)
      dz, dtheta = rbm.exchange_log_ratio(theta, up, dn)
      with np.errstate(over='ignore', invalid='ignore'):
        acc = can & (np.exp(2.0 * dz) > u)
        margin = np.abs(1.0 - u * np.exp(-2.0 * dz))
      res.margin[it, k] = np.where(can, np.where(np.isnan(margin), np.inf, margin), np.inf)
      sel = rows[acc]
      cfg[sel, up[acc]] = -1
      cfg[sel, dn[acc]] = 1
      theta[acc] += dtheta[acc]
      res.accepted[it] += acc
  res.final = cfg
  return res
