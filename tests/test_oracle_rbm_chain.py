"""CPU checks of oracle/rbm_chain.py (the float64 Markov-chain restatement of
cgsvmc_batch_steps) against the step-by-step oracle: philox.fast_proposal,
ansatz.log_amp, hamiltonian.local_energy and estimators.weighted_grad_sum."""
import numpy as np
import pytest
import torch

from oracle import ansatz as oansatz
from oracle import bits, estimators, hamiltonian, lattices, philox, rbm_chain

F64 = torch.float64


def _walkers(n, b, rng):
  """Random Sz = 0 walkers, then all up, all down, all but one up and a single
  down site (the edges of the proposal rule)."""
  cfg = bits.random_sz0_configs(n, b, rng).astype(np.int8)
  cfg[0] = 1
  cfg[1] = -1
  cfg[2] = 1
  cfg[2, n // 2] = -1               # one down site: k_dn is always 0
  cfg[3] = -1
  cfg[3, n - 1] = 1                 # one up site, the last one
  return cfg


def _reference_chain(spec, params, cfg, ij, jx, jz, seed, walker_id0, step0, n_steps, n_iters):
  """The same chain one proposal at a time, through the per-walker oracle."""
  fn = lambda c: oansatz.log_amp(spec, params, c)
  cur = cfg.astype(np.float64)
  b = cur.shape[0]
  ids = np.uint64(walker_id0) + np.arange(b, dtype=np.uint64)
  out = []
  for it in range(n_iters):
    c64 = torch.from_numpy(cur)
    e = hamiltonian.local_energy(c64, ij, jx, jz, fn).numpy()
    out.append((cur.copy(), fn(c64).numpy(), e, np.zeros(b, np.int64)))
    for k in range(n_steps):
      step = step0 + it * n_steps + k
      n_up = (cur > 0).sum(axis=1)
      mov = np.flatnonzero((n_up > 0) & (n_up < cur.shape[1]))
      if mov.size == 0:
        continue
      down, up, u = philox.fast_proposal(cur[mov], seed, ids[mov], step)
      prop = cur[mov].copy()
      prop[np.arange(mov.size), down] += 2
      prop[np.arange(mov.size), up] -= 2
      dz = (fn(torch.from_numpy(prop)) - fn(torch.from_numpy(cur[mov]))).numpy()
      acc = np.exp(2 * dz) > u
      cur[mov[acc]] = prop[acc]
      out[-1][3][mov[acc]] += 1
  return out, cur


@pytest.mark.parametrize('n,h,n_steps,n_iters,step0,walker_id0', [
    (10, 6, 7, 3, 0, 0),                               # odd n_steps
    (12, 9, 5, 3, 2 ** 32 - 7, 3),                     # the step counter crosses 2^32
    (9, 4, 13, 2, 11, 2 ** 32 + 7),                    # walker ids above 2^32
    (17, 33, 4, 2, 2 ** 33 - 3, 2 ** 40 - 2),          # both, odd N, H past one 32-unit chunk
])
def test_chain_matches_step_by_step_oracle(n, h, n_steps, n_iters, step0, walker_id0):
  spec = oansatz.AnsatzSpec('rbm', n, num_layers=0, layer_size=h)
  params = [p * 1.5 for p in oansatz.init_params(spec, seed=n + h, bias_scale=0.2, dtype=F64)]
  flat = oansatz.flatten(params).numpy()
  rng = np.random.default_rng(n * h)
  cfg = _walkers(n, 24, rng)
  ij, jx, jz = lattices.heisenberg_couplings(lattices.chain_bonds(n), -1.0, 1.0)
  jx = jx * np.linspace(0.5, 1.5, len(jx)).astype(np.float32)      # per-bond couplings
  seed = 0x5EED + n
  rbm = rbm_chain.Rbm(flat, n, h)
  res = rbm_chain.run_chain(rbm, cfg, ij, jx, jz, seed, walker_id0, step0, n_steps, n_iters)
  ref, final = _reference_chain(spec, params, cfg, ij, jx, jz, seed, walker_id0, step0, n_steps, n_iters)
  # both sides are float64: a decision could only differ at an exact tie
  assert res.margin.min() > 1e-9
  for it, (c, z, e, acc) in enumerate(ref):
    assert np.array_equal(res.configs[it], c.astype(np.int8))
    np.testing.assert_allclose(res.log_amp[it], z, rtol=0, atol=1e-11)
    np.testing.assert_allclose(res.e_loc[it], e, rtol=1e-11, atol=1e-11)
    assert np.array_equal(res.accepted[it], acc)
  assert np.array_equal(res.final, final.astype(np.int8))
  # walkers that cannot move propose nothing: all up / all down stay put
  assert np.all(res.accepted[:, :2] == 0) and np.all(np.isinf(res.margin[:, :, :2]))
  assert np.array_equal(res.final[:2], cfg[:2])
  # the single-down and single-up walkers do move, and keep their Sz
  assert res.accepted[:, 2:4].sum() > 0
  assert np.array_equal(res.final.sum(axis=1), cfg.sum(axis=1))
  # diag part, and E_abs = sum |jz| / 4 + the off-diagonal terms with |jx|
  c64 = torch.from_numpy(res.configs[0].astype(np.float64))
  d_o, _ = hamiltonian.build(c64, ij, jx, jz, lambda c: torch.ones(c.shape[0], dtype=F64))
  np.testing.assert_allclose(res.diag[0], d_o.numpy(), rtol=0, atol=1e-12)
  off_abs = hamiltonian.local_energy(c64, ij, np.abs(jx), 0 * jz, lambda c: oansatz.log_amp(spec, params, c))
  np.testing.assert_allclose(res.e_abs[0], off_abs.numpy() + 0.25 * np.abs(jz).sum(), rtol=1e-11, atol=1e-11)


def test_grad_sums_match_autograd():
  n, h, b = 11, 13, 40
  spec = oansatz.AnsatzSpec('rbm', n, num_layers=0, layer_size=h)
  params = oansatz.init_params(spec, seed=3, bias_scale=0.3, dtype=F64)
  rng = np.random.default_rng(5)
  cfg = rng.choice([-1.0, 1.0], size=(b, n))
  w = rng.normal(size=(3, b))
  rbm = rbm_chain.Rbm(oansatz.flatten(params).numpy(), n, h)
  s, bound = rbm.grad_sums(cfg, w)
  c64 = torch.from_numpy(cfg)
  ref = estimators.weighted_grad_sum(spec, params, c64, torch.from_numpy(w)).numpy()
  np.testing.assert_allclose(s, ref, rtol=1e-12, atol=1e-12)
  # the bound is sum_b |w_b| |O_b| (|sigma| = 1, |tanh theta| from the signed parameters)
  t = np.abs(np.tanh(cfg @ rbm.w + rbm.c))
  np.testing.assert_allclose(bound[:, n + 1 + n * h:], np.abs(w) @ t, rtol=1e-12)
  np.testing.assert_allclose(bound[:, :n + 1], np.repeat(np.abs(w).sum(axis=1)[:, None], n + 1, axis=1),
                             rtol=1e-12)
  assert np.all(np.abs(s) <= bound * (1 + 1e-12))
  assert rbm.n_params == oansatz.num_params(spec)


def test_kth_set_matches_flatnonzero():
  rng = np.random.default_rng(0)
  mask = rng.random((200, 70)) < 0.3
  mask[0] = True
  mask[1] = False
  mask[1, 69] = True
  cnt = mask.sum(axis=1)
  k = (rng.random(200) * cnt).astype(np.int64)
  got = rbm_chain.kth_set(mask, k)
  for r in range(200):
    assert got[r] == np.flatnonzero(mask[r])[k[r]]
