"""-m gpu: every variant of the pure-RBM walker kernel (rbm2) against a float64
replay of the Markov chain (oracle/rbm_chain.py).

The walker kernel `walker_kernel<NW, LPW, KJV, WS, MC, PT>` is compiled for
1, 2 and 4 spin words, 8 or 16 lanes per walker (KJV = HP / 32 = 1 .. 8), three
table placements (PT: image and bond-pair table in shared memory; WS: image in
shared memory, two-row ratio loop; GL: image and pair table in global memory),
with or without the fused sweep, with the gradient on the tensor cores or in
FP32 register tiles, and with the walkers kept in registers between
iterations or read back.  Each case below names the variant it must run; the
first assertion of every case is the library's own plan query
(Ansatz.rbm2_plan), so that a moved threshold fails here instead of silently
losing coverage, and the last test checks that the cases together cover every
(NW, KJV) pair, every placement and both settings of the two switches.

Each case runs cgsvmc_batch_steps (the epoch kernel of training and bench.py)
and checks it against the oracle's trajectory:

  1. z and E_loc of every iteration at the oracle's configurations, within the
     bounds of test_log_amp_vs_oracle / test_local_energy_vs_oracle;
  2. the final configurations bit for bit and the acceptance count, except
     for walkers after a near-tie (a decision within 1e-4 relative of
     exp(2 dz) = u, the band of test_fast_sampler_matches_oracle_philox): those
     are quarantined from that decision on, and they may be at most 0.5 % of
     the walker-iterations per 32 steps of an iteration;
  3. the energy statistics against the float64 sums of the returned E_loc;
  4. the gradient sums against the float64 sums over the oracle's
     trajectories (bound derived in _grad_tolerance);
  5. with n_steps = 0 the configurations stay put and every iteration must
     reproduce the first bit for bit (the re-parked 2W rows, the read-back and
     the tensor-core drains on unchanged input), sums = n_iters x one pass;
  6. the split entry points on the initial configurations: local_energy,
     weighted_grad_sum (K = 3), log_amp, mc_steps (one sweep) and
     log_amp_jvp (refused at three spin words, for which it is not built),
     which run the kernels without the fused sweep and rbm.cu.
"""
import dataclasses
import math

import numpy as np
import pytest
import torch

from oracle import ansatz as oansatz
from oracle import bits, lattices, rbm_chain

pytestmark = pytest.mark.gpu

U = 2.0 ** -24               # float32 unit roundoff
TIE_BAND = 1e-4              # near-tie band of the accept decision (relative)


def _quarantine_limit(n_walker_iters, n_steps):
  """Most walker-iterations that may be quarantined: 0.5 % for every 32
  decisions of an iteration.  A decision falls in the band with probability
  at most 2 TIE_BAND (u is uniform), so about n_steps x 2e-4 x acceptance of
  the walker-iterations meet one: 0.2 % at 32 steps and 30 % acceptance."""
  return 0.005 * n_walker_iters * max(1.0, n_steps / 32.0)
PAIR_TABLE = {'PT': 1, 'WS': 0, 'GL': 2}


@dataclasses.dataclass
class Case:
  n: int
  h: int
  lattice: str               # 'chain' | 'sq' | 'j1j2'
  batch: int
  n_iters: int
  n_steps: int
  expect: tuple              # (nw, lpw, kjv, placement, tc_grad, keeps_walkers); None: rbm2 declines
  scale: float = 1.0
  step0: int = 0
  walker_id0: int = 0
  edges: bool = False        # all up / all down / one down / one up walkers among the random ones
  seed: int = 1

  @property
  def id(self):
    s = 'N%d_H%d_%s_B%d' % (self.n, self.h, self.lattice, self.batch)
    if self.scale != 1.0:
      s += '_x%g' % self.scale
    if self.step0 or self.walker_id0:
      s += '_offsets'
    return s


CASES = [
    # one spin word
    Case(16, 7, 'chain', 1001, 3, 16, (1, 8, 1, 'PT', 0, 1), edges=True),
    Case(16, 7, 'chain', 1, 3, 7, (1, 8, 1, 'PT', 0, 1)),
    Case(16, 7, 'chain', 3, 3, 7, (1, 8, 1, 'PT', 0, 1), edges=True),
    Case(36, 40, 'sq', 999, 3, 36, (1, 8, 2, 'PT', 1, 1)),
    Case(39, 95, 'chain', 777, 3, 13, (1, 8, 3, 'PT', 1, 1), edges=True),     # largest M = 3 x 40
    Case(64, 96, 'chain', 601, 2, 64, (1, 8, 3, 'PT', 0, 1), edges=True),     # full word
    Case(64, 96, 'sq', 601, 2, 64, (1, 8, 3, 'WS', 0, 1)),
    Case(36, 100, 'j1j2', 501, 2, 36, (1, 8, 4, 'WS', 0, 1)),
    Case(64, 100, 'j1j2', 401, 2, 64, (1, 8, 4, 'GL', 0, 1)),
    Case(36, 159, 'sq', 10000, 5, 7, (1, 8, 5, 'PT', 1, 0)),                  # HP - H = 1, read-back, 10 passes
    Case(36, 144, 'j1j2', 501, 2, 36, (1, 8, 5, 'WS', 0, 1), scale=4.0),      # C2 J1-J2, renormalising every 4 steps
    Case(36, 144, 'j1j2', 801, 3, 36, (1, 8, 5, 'WS', 0, 1)),                 # C2 J1-J2
    Case(64, 144, 'sq', 401, 2, 64, (1, 8, 5, 'GL', 0, 1)),
    Case(40, 180, 'chain', 501, 2, 40, (1, 16, 6, 'WS', 0, 1)),
    Case(36, 224, 'sq', 501, 2, 36, (1, 16, 7, 'WS', 0, 1)),
    Case(64, 200, 'sq', 401, 2, 64, (1, 16, 7, 'GL', 0, 1)),
    Case(16, 256, 'j1j2', 501, 2, 16, (1, 16, 8, 'WS', 0, 1)),
    # two spin words
    Case(65, 32, 'chain', 501, 3, 13, (2, 8, 1, 'PT', 0, 1), step0=2 ** 32 - 5, walker_id0=2 ** 32 + 7),
    Case(100, 40, 'sq', 401, 2, 100, (2, 8, 2, 'WS', 0, 1)),
    Case(128, 96, 'chain', 301, 2, 128, (2, 8, 3, 'GL', 0, 1)),               # full words
    Case(65, 128, 'chain', 401, 2, 65, (2, 8, 4, 'PT', 0, 1), edges=True),
    Case(100, 144, 'sq', 301, 2, 100, (2, 8, 5, 'GL', 0, 1)),
    Case(65, 192, 'chain', 301, 2, 65, (2, 16, 6, 'WS', 0, 1)),
    Case(100, 224, 'sq', 301, 2, 100, (2, 16, 7, 'GL', 0, 1)),
    Case(128, 256, 'chain', 251, 2, 128, (2, 16, 8, 'GL', 0, 1)),
    # three words (run as four) and four
    Case(129, 7, 'chain', 401, 2, 129, (4, 8, 1, 'PT', 0, 1), edges=True),
    Case(144, 32, 'sq', 301, 2, 144, (4, 8, 1, 'WS', 0, 1)),
    Case(129, 64, 'chain', 301, 2, 129, (4, 8, 2, 'WS', 0, 1)),
    Case(192, 65, 'chain', 251, 2, 192, (4, 8, 3, 'GL', 0, 1)),
    Case(144, 96, 'sq', 251, 2, 144, (4, 8, 3, 'GL', 0, 1)),
    Case(196, 128, 'chain', 201, 2, 196, (4, 8, 4, 'GL', 0, 1)),
    Case(144, 160, 'sq', 201, 2, 144, (4, 8, 5, 'GL', 0, 1)),
    Case(196, 192, 'sq', 201, 2, 196, (4, 16, 6, 'GL', 0, 1)),
    Case(144, 224, 'j1j2', 151, 2, 144, (4, 16, 7, 'GL', 0, 1)),
    Case(256, 256, 'sq', 201, 2, 256, (4, 16, 8, 'GL', 0, 1)),                # C5
    # rbm2 declines (512 bonds at H = 144): the per-iteration fallback
    Case(256, 144, 'sq', 201, 2, 256, None),
]


def _couplings(case):
  if case.lattice == 'chain':
    return lattices.heisenberg_couplings(lattices.chain_bonds(case.n))
  size = int(round(math.sqrt(case.n)))
  assert size * size == case.n
  if case.lattice == 'sq':
    return lattices.heisenberg_couplings(lattices.square_nn_bonds(size))
  return lattices.j1j2_couplings(size, 0.5)


def _problem(case):
  """float32 parameters (as the device sees them, in float64), couplings and
  initial walkers of a case."""
  spec = oansatz.AnsatzSpec('rbm', case.n, num_layers=0, layer_size=case.h)
  params = oansatz.init_params(spec, seed=case.n * 1000 + case.h + case.seed, bias_scale=0.1,
                               dtype=torch.float64)
  flat = (oansatz.flatten(params).numpy() * case.scale).astype(np.float32)
  rng = np.random.default_rng(case.n * 7 + case.h + case.seed)
  cfg = bits.random_sz0_configs(case.n, case.batch, rng).astype(np.int8)
  if case.edges:
    b = case.batch
    rows = sorted({0, min(1, b - 1), b // 2, b - 1})
    kinds = ['up', 'down', 'one_down', 'one_up']
    for r, kind in zip(rows, kinds[:len(rows)]):
      cfg[r] = 1 if kind in ('up', 'one_down') else -1
      if kind == 'one_down':
        cfg[r, case.n // 3] = -1
      if kind == 'one_up':
        cfg[r, case.n - 1] = 1
  ij, jx, jz = _couplings(case)
  return spec, flat, cfg, (ij, jx, jz)


def _amp_scale(rbm):
  """Sum of |terms| entering z (the same for every configuration): the scale
  of the float32 rounding of a forward pass (gpu_util.amp_scale)."""
  x = np.abs(rbm.w).sum(axis=0) + np.abs(rbm.c)
  return np.abs(rbm.a).sum() + abs(rbm.a0) + (np.logaddexp(x, -x) - math.log(2.0)).sum() + 1.0


def _e_scale(e_abs, diag):
  return np.abs(e_abs) + 2.0 * np.abs(diag) + 1.0


def _check_plan(plan, expect):
  if expect is None:
    assert plan is None
    return
  nw, lpw, kjv, place, tc, keep = expect
  assert plan is not None
  got = (plan['nw'], plan['lpw'], plan['kjv'],
         'PT' if plan['pair_table'] == 1 else ('WS' if plan['tables_in_smem'] else 'GL'),
         plan['tc_grad'], plan['keeps_walkers'])
  assert got == (nw, lpw, kjv, place, tc, keep), (got, plan)
  assert plan['pair_table'] == PAIR_TABLE[place]
  assert plan['tables_in_smem'] == (place != 'GL')


def _grad_tolerance(n, p, passes, n_adds, tc, bound, w_abs_sum, exact_row0=True):
  """Per-entry bound on |S_gpu - S_oracle| of gradient sums formed by the
  launch plan p (`passes` walker batches per CTA, `n_adds` float32 additions
  into the output after the cross-CTA sum).

  Terms: w_kb O_bp with O_b = (sigma, 1, sigma_i tanh theta_j, tanh theta_j),
  |O_bp| <= 1.  The weights are exact inputs to both sides (1 and the kernel's
  own E_loc, which the oracle sum uses too, or given float32 weights).

  * Per-term error of tanh theta: the kernel forms it as p - m from the
    normalised state, a product of N + 1 rounded table factors: at most
    (N + 8) u absolute (d tanh / d theta <= 1).  With the gradient on the
    tensor cores tanh theta is split into two fp16 planes (22 bits): + 2^-22;
    E_loc into three pieces (33 bits): + 2^-32 relative.  sigma and 1 are exact.
  * Accumulation: a term passes through at most D float32 additions, so the
    sum is off by at most D u sum_b |w_kb O_bp| (first order).
      register tiles, W and c: D = wpc / 4 (a lane's walkers) + 2 (shuffle
        reduction) + passes (+= across passes) + grid (cross-CTA) + n_adds;
      register tiles, a and a0: D = passes x wpc (one running sum over every
        walker of the CTA) + grid + n_adds;
      tensor cores: accumulation truncates (2 u per addition) over the slots of
        one MMA (K = walkers) and the 8 passes of a drain segment, then float32
        adds over the drains and the CTAs: D = 2 (slots + 8) + drains + grid + n_adds.
  * With weights 1, row 0 of the a / a0 block sums +-1 and 1: integers below
    2^24, exact in float32 on both paths.
  """
  if tc:
    d_w = d_a = 2 * (p['slots'] + 8) + -(-passes // 8) + p['grid'] + n_adds
    eps_t = (n + 8) * U + 2.0 ** -22
  else:
    d_w = p['wpc'] / 4 + 2 + passes + p['grid'] + n_adds
    d_a = passes * p['wpc'] + p['grid'] + n_adds
    eps_t = (n + 8) * U
  tol = np.empty_like(bound)
  tol[:, :n + 1] = d_a * U * bound[:, :n + 1]
  if exact_row0:
    tol[0, :n + 1] = 0.0
  tol[:, n + 1:] = d_w * U * bound[:, n + 1:] + eps_t * w_abs_sum[:, None]
  if tc:
    tol[1] += 2.0 ** -32 * bound[1]
  return tol + 1e-6


def _epoch_grad_tolerance(a, ham, case, bound, w_abs_sum):
  """_grad_tolerance of one batch_steps call: one launch of the walker kernel,
  or (rbm2 declines) one accumulate per iteration, whose gradient pass is a
  weighted_grad_sum launch with weights (1, E_loc)."""
  plan = a.rbm2_plan(ham, case.batch, 'batch_steps')
  per_cta = lambda p: -(-p['n_batches'] // p['grid'])
  if plan is not None:
    return _grad_tolerance(case.n, plan, per_cta(plan) * case.n_iters, 1, plan['tc_grad'] == 1, bound, w_abs_sum)
  p = a.rbm2_plan(None, case.batch, 'weighted_grad_sum')
  return _grad_tolerance(case.n, p, per_cta(p), case.n_iters, False, bound, w_abs_sum)


def _run_batch_steps(native, a, ham, packed, case, n_steps, n_iters):
  b = case.batch
  sums = torch.zeros(2, a.num_params, dtype=torch.float32, device='cuda')
  stats = torch.zeros(4, dtype=torch.float64, device='cuda')
  count = torch.zeros(1, dtype=torch.int64, device='cuda')
  e = torch.empty(n_iters, b, dtype=torch.float32, device='cuda')
  z = torch.empty(n_iters, b, dtype=torch.float32, device='cuda')
  a.batch_steps(ham, packed, n_iters, sums, stats, n_steps, 0x5EED + case.n, walker_id0=case.walker_id0,
                step0=case.step0, accept_count=count, e_loc_out=e, log_amp_out=z)
  torch.cuda.synchronize()
  return (e.cpu().numpy().astype(np.float64), z.cpu().numpy().astype(np.float64), sums.cpu().numpy().astype(np.float64),
          stats.cpu().numpy(), int(count.item()))


def _check_stats(stats, e):
  """stats = (sum E, sum E^2, count, 0) of the float32 local energies e,
  summed in float64: 1e-12 of the sums of magnitudes (the summation order
  differs)."""
  assert abs(stats[0] - e.sum()) <= 1e-12 * np.abs(e).sum()
  assert abs(stats[1] - (e * e).sum()) <= 1e-12 * (e * e).sum()
  assert stats[2] == e.size and stats[3] == 0.0


def _quarantine(res, n_steps):
  """Per walker: the iteration of its first near-tie decision (n_iters when
  there is none) and the number of steps from that decision on."""
  n_iters, _, b = res.margin.shape
  if n_steps == 0:
    return np.full(b, n_iters), np.zeros(b, np.int64)
  tie = (res.margin <= TIE_BAND).reshape(n_iters * n_steps, b)
  first = np.where(tie.any(axis=0), np.argmax(tie, axis=0), n_iters * n_steps)
  return first // n_steps, n_iters * n_steps - first


@pytest.fixture(scope='module')
def native():
  from cgs_vmc_b200 import _native
  _native.load()
  return _native


@pytest.mark.parametrize('case', CASES, ids=lambda c: c.id)
def test_batch_steps_vs_chain_oracle(native, case):
  from gpu_util import make_native, packed_cuda, unpack_np
  spec, flat, cfg, (ij, jx, jz) = _problem(case)
  a = make_native(spec, flat)
  ham = native.Hamiltonian(ij, jx, jz, case.n)
  plan = a.rbm2_plan(ham, case.batch, 'batch_steps')
  _check_plan(plan, case.expect)
  rbm = rbm_chain.Rbm(flat, case.n, case.h)
  b, n, n_iters, n_steps = case.batch, case.n, case.n_iters, case.n_steps

  # ---- the chain ----
  packed = packed_cuda(cfg)
  e, z, sums, stats, count = _run_batch_steps(native, a, ham, packed, case, n_steps, n_iters)
  res = rbm_chain.run_chain(rbm, cfg, ij, jx, jz, 0x5EED + n, case.walker_id0, case.step0, n_steps, n_iters)
  q_iter, q_steps = _quarantine(res, n_steps)
  n_q = int((q_iter < n_iters).sum())
  excluded = int((n_iters - np.minimum(q_iter + 1, n_iters)).sum() + n_q)
  print('\n%s plan=%s quarantined=%d walkers, %d of %d walker-iterations' %
        (case.id, plan, n_q, excluded, b * n_iters))
  assert excluded <= _quarantine_limit(b * n_iters, n_steps) or excluded == 0
  # 1. per-iteration values where the walker still follows the oracle (up to
  #    and including the iteration of its first near-tie)
  live = np.arange(n_iters)[:, None] <= q_iter[None, :]
  amp_tol = 4e-6 * _amp_scale(rbm)
  dz = np.abs(z - res.log_amp)
  assert np.all(dz[live] <= amp_tol), (dz[live].max(), amp_tol)
  de = np.abs(e - res.e_loc)
  e_tol = 2e-5 * _e_scale(res.e_abs, res.diag)
  assert np.all(de[live] <= e_tol[live]), (de[live] / e_tol[live]).max()
  # 2. final configurations and acceptance count
  final = unpack_np(packed, n).astype(np.int8)
  clean = q_iter >= n_iters
  assert np.array_equal(final[clean], res.final[clean]), np.flatnonzero(~np.all(final == res.final, axis=1))
  assert np.array_equal(final.sum(axis=1), cfg.sum(axis=1).astype(np.int64))          # Sz per walker
  assert abs(count - int(res.accepted.sum())) <= int(q_steps[~clean].sum())
  # 3. energy statistics from the returned local energies
  _check_stats(stats, e)
  # 4. gradient sums over the oracle trajectories, weights (1, E_loc of the kernel)
  s_ref = np.zeros_like(sums)
  s_bound = np.zeros_like(sums)
  w_abs = np.zeros(2)
  for it in range(n_iters):
    w = np.stack([np.ones(b), e[it]])
    s_i, bd_i = rbm.grad_sums(res.configs[it], w)
    s_ref += s_i
    s_bound += bd_i
    w_abs += np.abs(w).sum(axis=1)
  tol = _epoch_grad_tolerance(a, ham, case, s_bound, w_abs)
  n_qwi = excluded            # quarantined walker-iterations: |O| <= 1 on both sides
  tol[0] += 2.0 * n_qwi
  tol[1] += 2.0 * np.abs(e).max() * n_qwi
  err = np.abs(sums - s_ref)
  assert np.all(err <= tol), (np.unravel_index(np.argmax(err / tol), err.shape), (err / tol).max())

  # 5. n_steps = 0: the same variant, nothing moves, every iteration repeats the first
  assert a.rbm2_plan(ham, b, 'batch_steps') == plan
  packed0 = packed_cuda(cfg)
  e0, z0, sums0, stats0, count0 = _run_batch_steps(native, a, ham, packed0, case, 0, n_iters)
  assert count0 == 0 and torch.equal(packed0, packed_cuda(cfg))
  for it in range(n_iters):
    assert np.array_equal(e0[it], e[0]) and np.array_equal(z0[it], z[0]), it
  w = np.stack([np.ones(b), e[0]])
  s1, bd1 = rbm.grad_sums(cfg, w)
  tol0 = _epoch_grad_tolerance(a, ham, case, n_iters * bd1, n_iters * np.abs(w).sum(axis=1))
  err0 = np.abs(sums0 - n_iters * s1)
  assert np.all(err0 <= tol0), (np.unravel_index(np.argmax(err0 / tol0), err0.shape), (err0 / tol0).max())
  _check_stats(stats0, np.broadcast_to(e[0], (n_iters, b)))

  # 6. the split entry points on the initial configurations
  p0 = packed_cuda(cfg)
  e_s, z_s, d_s, _ = a.local_energy(ham, p0, want_parts=True)
  e_s, z_s, d_s = (t.cpu().numpy().astype(np.float64) for t in (e_s, z_s, d_s))
  assert np.all(np.abs(e_s - res.e_loc[0]) <= 2e-5 * _e_scale(res.e_abs[0], res.diag[0]))
  np.testing.assert_allclose(d_s, res.diag[0], rtol=0, atol=1e-5)
  assert np.all(np.abs(z_s - res.log_amp[0]) <= amp_tol)
  z_l = a.log_amp(p0).cpu().numpy().astype(np.float64)
  assert np.all(np.abs(z_l - res.log_amp[0]) <= amp_tol)
  rng = np.random.default_rng(n + case.h)
  w3 = rng.normal(size=(3, b)).astype(np.float32)
  g = a.weighted_grad_sum(p0, torch.from_numpy(w3).cuda()).cpu().numpy().astype(np.float64)
  g_ref, g_bound = rbm.grad_sums(cfg, w3.astype(np.float64))
  wplan = a.rbm2_plan(None, b, 'weighted_grad_sum')
  g_tol = _grad_tolerance(n, wplan, -(-wplan['n_batches'] // wplan['grid']), 1, False, g_bound,
                          np.abs(w3).sum(axis=1).astype(np.float64), exact_row0=False)
  assert np.all(np.abs(g - g_ref) <= g_tol), (np.abs(g - g_ref) / g_tol).max()
  tangent = torch.from_numpy(rng.normal(size=a.num_params).astype(np.float32)).cuda()
  if (n + 63) // 64 == 3:
    # the JVP kernel is built for 1, 2 and 4 spin words (cgsvmc_log_amp_jvp in
    # include/cgsvmc.h): three must be refused, not misread as four
    with pytest.raises(NotImplementedError):
      a.log_amp_jvp(p0, tangent)
  else:
    y = a.log_amp_jvp(p0, tangent).cpu().numpy().astype(np.float64)
    t = np.tanh(rbm.theta(cfg))
    v = tangent.cpu().numpy().astype(np.float64)
    va, va0, vw, vc = v[:n], v[n], v[n + 1:n + 1 + n * case.h].reshape(n, case.h), v[n + 1 + n * case.h:]
    c64 = cfg.astype(np.float64)
    y_ref = c64 @ va + va0 + (t * (c64 @ vw + vc)).sum(axis=1)
    y_abs = np.abs(va).sum() + abs(va0) + (np.abs(t) * (np.abs(vw).sum(axis=0) + np.abs(vc))).sum(axis=1)
    assert np.all(np.abs(y - y_ref) <= 1e-5 * y_abs + 1e-6), np.abs(y - y_ref).max()
  # one sweep of the sampler kernel, log-amplitudes of where it ends
  z_mc = torch.empty(b, dtype=torch.float32, device='cuda')
  cnt = torch.zeros(1, dtype=torch.int64, device='cuda')
  a.mc_steps(p0, n, 0xBEEF, walker_id0=case.walker_id0, step0=case.step0, accept_count=cnt, log_amp_out=z_mc)
  sweep = rbm_chain.run_chain(rbm, cfg, ij, jx, jz, 0xBEEF, case.walker_id0, case.step0, n, 1)
  sq_iter, sq_steps = _quarantine(sweep, n)
  ok = sq_iter >= 1
  got = unpack_np(p0, n).astype(np.int8)
  assert (~ok).sum() <= _quarantine_limit(b, n) or (~ok).sum() == 0
  assert np.array_equal(got[ok], sweep.final[ok])
  assert abs(int(cnt.item()) - int(sweep.accepted.sum())) <= int(sq_steps[~ok].sum())
  z_end = rbm.log_amp(sweep.final)
  assert np.all(np.abs(z_mc.cpu().numpy().astype(np.float64)[ok] - z_end[ok]) <= amp_tol)


def test_cases_cover_every_variant(native):
  """The cases' batch_steps plans together hit every (NW, KJV) pair, every
  placement of every word count, the tensor-core gradient and the register
  tiles, and walkers kept in registers and read back; and every case that
  names a variant gets it."""
  from gpu_util import make_native
  seen = set()
  for case in CASES:
    spec = oansatz.AnsatzSpec('rbm', case.n, num_layers=0, layer_size=case.h)
    a = make_native(spec, np.zeros(oansatz.num_params(spec), dtype=np.float32))
    ij, jx, jz = _couplings(case)
    ham = native.Hamiltonian(ij, jx, jz, case.n)
    plan = a.rbm2_plan(ham, case.batch, 'batch_steps')
    _check_plan(plan, case.expect)
    if plan is not None:
      seen.add((plan['nw'], plan['kjv'], 'PT' if plan['pair_table'] == 1 else ('WS' if plan['tables_in_smem'] else 'GL'),
                plan['tc_grad'], plan['keeps_walkers']))
  pairs = {(nw, kjv) for nw, kjv, *_ in seen}
  assert pairs == {(nw, kjv) for nw in (1, 2, 4) for kjv in range(1, 9)}, sorted(pairs)
  for nw in (1, 2, 4):
    assert {pl for w, _, pl, _, _ in seen if w == nw} == {'PT', 'WS', 'GL'}, nw
  assert {tc for *_, tc, _ in seen} == {0, 1}
  assert {keep for *_, keep in seen} == {0, 1}
  assert sum(c.expect is None for c in CASES) >= 1
  assert sum(c.n_steps % 8 != 0 and c.n_steps < c.n for c in CASES) >= 2


def test_plan_query_arguments(native):
  """The plan query allocates nothing and answers for every entry point; it
  refuses bad arguments like the entry points do."""
  from gpu_util import make_native
  spec = oansatz.AnsatzSpec('rbm', 36, num_layers=0, layer_size=144)
  a = make_native(spec, np.zeros(oansatz.num_params(spec), dtype=np.float32))
  ij, jx, jz = lattices.heisenberg_couplings(lattices.square_nn_bonds(6))
  ham = native.Hamiltonian(ij, jx, jz, 36)
  for mode in native.RBM2_PLAN_MODES:
    p = a.rbm2_plan(ham, 8192, mode)
    assert p is not None and p['supported'] == 1 and p['nw'] == 1 and p['kjv'] == 5
  assert a.rbm2_plan(ham, 8192, 'mc_steps')['pair_table'] == 0
  assert a.rbm2_plan(ham, 8192, 'weighted_grad_sum')['tc_grad'] == 0
  with pytest.raises(ValueError):
    a.rbm2_plan(ham, 0, 'batch_steps')
  with pytest.raises(ValueError):
    a.rbm2_plan(None, 10, 'local_energy')
  with pytest.raises(ValueError):
    a.rbm2_plan(ham, 10, 'no_such_mode')
  other = native.Hamiltonian([(0, 1)], -1.0, 1.0, 12)
  with pytest.raises(ValueError):
    a.rbm2_plan(other, 10, 'accumulate')
  fc = native.Ansatz('fully_connected', 36, num_layers=1, layer_size=8)
  assert fc.rbm2_plan(ham, 10, 'batch_steps') is None
