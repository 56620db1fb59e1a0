"""Stochastic reconfiguration (oracle side; test infrastructure).

Float64 restatement of cgs_vmc_b200.training.StochasticReconfigurationOptimizer
(not in the reference): with O_b = d z_b / d params over M walkers and <.> the
mean over them,
  S = <O O^T> - <O><O>^T,   F = <E O> - <E><O>,   (S + shift I) delta = F.
The per-walker gradients come from torch autograd on oracle.ansatz.log_amp.
"""
import numpy as np
import torch

from . import ansatz as _ansatz
from . import estimators


def _z_of_flat(spec, configs):
  return lambda flat: _ansatz.log_amp(spec, _ansatz.unflatten(spec, flat), configs)


def log_amp_jvp(spec, params, configs, tangent):
  """y[b] = sum_p d z_b / d params_p * tangent[p] (forward-mode autograd)."""
  flat = _ansatz.flatten(params)
  configs = configs.to(flat.dtype)
  _, y = torch.func.jvp(_z_of_flat(spec, configs), (flat,), (tangent.to(flat.dtype),))
  return y


def per_sample_grads(spec, params, configs):
  """O[b, p] = d z_b / d params_p, dense [B, P]."""
  flat = _ansatz.flatten(params)
  return torch.func.jacrev(_z_of_flat(spec, configs.to(flat.dtype)))(flat)


def sr_matrix(spec, params, configs):
  """Dense S = <O O^T> - <O><O>^T, [P, P]."""
  o = per_sample_grads(spec, params, configs)
  oc = o - o.mean(dim=0)
  return oc.T @ oc / o.shape[0]


def sr_forces(spec, params, configs, e_loc):
  """F = <E O> - <E><O>, [P]."""
  o = per_sample_grads(spec, params, configs)
  e = e_loc.to(o.dtype)
  return (e[:, None] * o).mean(dim=0) - e.mean() * o.mean(dim=0)


def sr_matvec(spec, params, configs, v, diag_shift):
  """(S + diag_shift I) v without forming S: y = O v - <O v>, then
  sum_b y_b O_b / M (a JVP and a vector-Jacobian product)."""
  y = log_amp_jvp(spec, params, configs, v)
  y = y - y.mean()
  sv = estimators.weighted_grad_sum(spec, params, configs.to(params[0].dtype), y[None, :])[0]
  return sv / configs.shape[0] + diag_shift * v


def sr_direction(spec, params, configs, e_loc, diag_shift):
  """delta = (S + diag_shift I)^-1 F by numpy.linalg.solve."""
  s = sr_matrix(spec, params, configs).numpy()
  f = sr_forces(spec, params, configs, e_loc).numpy()
  return np.linalg.solve(s + diag_shift * np.eye(s.shape[0]), f)
