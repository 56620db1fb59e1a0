"""Mirror of the reference's training.py for its working optimizers:
EnergyGradientOptimizer (training.py:506-623),
SupervisedWavefunctionOptimizer (135-212), LogOverlapSWO (298-404),
DualSamplingSWO (407-503) and LogOverlapImaginaryTimeSWO (626-778), with the
same TrainOps tuples, registries and epoch schedules.  Every estimator is the
one device primitive S_k = sum_b w_kb O_b (cgsvmc_weighted_grad_sum) with
different weight columns (SURVEY.md appendix A.5).  The Metropolis loops of the
reference (one session.run per step) collapse into one persistent-kernel
launch per sweep group; `session.run(train_ops.mc_step)` still performs a
single step for drop-in callers.

StochasticReconfigurationOptimizer goes beyond the reference: the natural
gradient of VMC for the pure RBM, with S applied matrix-free through
cgsvmc_log_amp_jvp and cgsvmc_weighted_grad_sum.
"""
import collections
import copy
import math
import types

import torch

from . import _native, distributed, engine, graph_builders, wavefunctions
from .session import Op

TrainOpsTraditional = collections.namedtuple('TrainingOpsTraditional', [
    'accumulate_gradients', 'apply_gradients', 'reset_gradients', 'mc_step', 'acc_rate',
    'metrics', 'epoch_increment', 'update_wf_norm'])
TrainOpsSWO = collections.namedtuple('TrainingOpsSWO', [
    'train_step', 'accumulate_gradients', 'apply_gradients', 'reset_gradients', 'mc_step',
    'acc_rate', 'metrics', 'energy', 'update_supervisor', 'update_normalization',
    'epoch_increment', 'update_wf_norm'])
TrainOpsSupervised = collections.namedtuple('TrainingOpsSupervised', [
    'accumulate_gradients', 'apply_gradients', 'reset_gradients', 'mc_step', 'acc_rate',
    'metrics', 'epoch_increment', 'update_wf_norm'])


def piecewise_constant(x, boundaries, values):
  """tf.train.piecewise_constant: values[0] for x <= boundaries[0], ..."""
  for b, v in zip(boundaries, values):
    if x <= b:
      return v
  return values[len(boundaries)]


class _Optimizer:
  """Applies a gradient to the flat parameter buffer with the learning-rate
  schedule of create_sgd_optimizer (training.py:84-91)."""

  def __init__(self, hparams):
    self._rates = list(hparams.learning_rates)
    self._stops = list(hparams.learning_rate_stops)

  def learning_rate(self):
    return piecewise_constant(int(graph_builders.get_or_create_num_epochs()), self._stops, self._rates)


class AdamOptimizer(_Optimizer):
  """tf.train.AdamOptimizer(lr, beta2=hparams.beta2): beta1 = 0.9, eps = 1e-8,
  theta -= lr * sqrt(1 - b2^t) / (1 - b1^t) * m / (sqrt(v) + eps); one kernel
  per update (cgsvmc_adam_step)."""

  def __init__(self, hparams):
    super().__init__(hparams)
    self.beta1, self.beta2, self.eps = 0.9, float(hparams.beta2), 1e-8
    self.m = self.v = None
    self.t = 0
    self.t_dev = self.lr_dev = None      # device copies for captured steps

  def _state(self, params):
    if self.m is None:
      self.m = torch.zeros_like(params)
      self.v = torch.zeros_like(params)

  def apply_gradients(self, params, grad=None, sums=None, stats=None, num_batches=1.0):
    """`grad`, or the energy gradient formed from (sums, stats, num_batches)
    inside the update kernel (training.py:562-567)."""
    self._state(params)
    self.t += 1
    if grad is not None:
      grad = grad.contiguous()
    _native.adam_step(params, self.m, self.v, grad=grad, sums=sums, stats=stats,
                      num_batches=num_batches, lr=self.learning_rate(), beta1=self.beta1,
                      beta2=self.beta2, eps=self.eps, t=self.t)

  def epoch_end(self, params, local_sums, local_stats, num_batches, stats_out, total_sums=None,
                total_stats=None, total_payload=None):
    """apply_gradients on the totals + the totals' statistics to `stats_out` +
    reset of the local accumulators in ONE kernel (cgsvmc_epoch_end;
    training.py:618-622)."""
    self._state(params)
    self.t += 1
    if getattr(self, '_ticket', None) is None:
      self._ticket = torch.zeros(1, dtype=torch.int32, device=params.device)
    _native.epoch_end(params, self.m, self.v, local_sums, local_stats, self._ticket, total_sums=total_sums,
                      total_stats=total_stats, total_payload=total_payload, num_batches=num_batches,
                      lr=self.learning_rate(), beta1=self.beta1, beta2=self.beta2, eps=self.eps, t=self.t,
                      stats_out=stats_out)

  def device_state(self, params):
    """(t_dev, lr_dev): step count and learning rate in device memory for a
    captured update; sync_device() refreshes them before a replay."""
    self._state(params)
    if self.t_dev is None:
      self.t_dev = torch.zeros(1, dtype=torch.int64, device=params.device)
      self.lr_dev = torch.zeros(1, dtype=torch.float32, device=params.device)
      self._lr_on_dev = self._t_on_dev = None
    return self.t_dev, self.lr_dev

  def sync_device(self, steps_in_replay):
    """Call before replaying a graph that takes `steps_in_replay` captured
    updates: pushes a changed learning rate, keeps the host count in step."""
    lr = self.learning_rate()
    if lr != self._lr_on_dev:
      self.lr_dev.fill_(lr)
      self._lr_on_dev = lr
    if self._t_on_dev != self.t:           # eager updates were taken in between
      self.t_dev.fill_(self.t)
    self.t += steps_in_replay
    self._t_on_dev = self.t

  def apply_gradients_captured(self, params, grad):
    """The update with t / lr read on the device (inside a graph capture)."""
    t_dev, lr_dev = self.device_state(params)
    _native.adam_step(params, self.m, self.v, grad=grad, lr_dev=lr_dev, beta1=self.beta1,
                      beta2=self.beta2, eps=self.eps, t_dev=t_dev)


class GradientDescentOptimizer(_Optimizer):
  def apply_gradients(self, params, grad=None, sums=None, stats=None, num_batches=1.0):
    if grad is None:
      nb = float(num_batches)
      grad = sums[1] / nb - (stats[0] / stats[2]).float() * sums[0] / nb
    params.add_(grad, alpha=-self.learning_rate())


OPTIMIZERS = {      # training.py:76-81; rms_prop / momentum never worked there
    'adam': AdamOptimizer,   # (beta2 is passed to every class, training.py:91)
    'gradient': GradientDescentOptimizer,
}


def create_sgd_optimizer(hparams):
  if hparams.optimizer not in OPTIMIZERS:
    raise NotImplementedError('optimizer=%r: only adam (the one that works in the reference, '
                              'SURVEY.md appendix B-5) and gradient are built' % hparams.optimizer)
  return OPTIMIZERS[hparams.optimizer](hparams)


def _update_norm_op(wavefunction, configs):
  """wavefunction.update_norm(wavefunction(configs)) of training.py:584, 377,
  726 with the batch maximum taken in the log domain."""
  if not wavefunction.fast_path:
    return wavefunction.update_norm(lambda: wavefunction(configs))
  return wavefunction.update_norm(lambda: wavefunction(configs),
                                  log_amplitudes=lambda: wavefunction.log_amplitude(configs))


def _epoch_increment():
  def run():
    graph_builders.get_or_create_num_epochs().add_(1)
  return Op(run, 'epoch_increment')


class _Model:
  """What an optimizer needs from a wavefunction, on either evaluation route
  (wavefunctions.py: `fast_path` = one ansatz with exp output on the fused
  kernels; otherwise signed / composite amplitudes through amplitudes()):
  (log|psi|, sign), the estimator primitive S_k = sum_b w_kb O_b over all
  trainable parameters, and the parameter update, leaf by leaf."""

  def __init__(self, wavefunction, n_sites, hparams=None):
    wavefunction.connect(n_sites)
    self.wavefunction = wavefunction
    self.fast = bool(wavefunction.fast_path)
    self.leaves = wavefunction.leaves()
    self.leaf_params = [leaf.native().params for leaf in self.leaves]
    for params in self.leaf_params:      # replicas start from rank 0's parameters
      distributed.broadcast_(params)
    self.num_params = sum(int(p.numel()) for p in self.leaf_params)
    self.device = self.leaf_params[0].device
    self.optimizers = ([create_sgd_optimizer(hparams) for _ in self.leaves]
                       if hparams is not None else None)
    self.ansatz = wavefunction.native(n_sites) if self.fast else None

  def log_psi(self, packed):
    """(log|psi|, sign psi), float32 [B] each."""
    if self.fast:
      z = self.ansatz.log_amp(packed) - self.wavefunction._exp_norm_shift
      return z, torch.ones_like(z)
    logabs, sign = self.wavefunction.amplitudes(packed)
    return logabs.float(), sign.float()

  def weighted_grad_sum(self, packed, weights, out):
    """out[K, P] += sum_b weights[k, b] d log psi_b / d params."""
    weights = weights.reshape(-1, packed.shape[0]).float().contiguous()
    if self.fast:
      self.ansatz.weighted_grad_sum(packed, weights, out=out)
    else:
      out.add_(self.wavefunction.weighted_grad_sum(packed, weights))
    return out

  def apply_gradients(self, flat_grad):
    off = 0
    for params, optimizer in zip(self.leaf_params, self.optimizers):
      n = int(params.numel())
      optimizer.apply_gradients(params, flat_grad[off:off + n])
      off += n


class _GenericEnergyGradientSums:
  """engine.EnergyGradientSums for signed / composite wavefunctions: the local
  energy through Operator.local_value (amplitude-agnostic route), then the two
  gradient sums and the energy statistics."""

  def __init__(self, model, hamiltonian, configs):
    self.model, self.hamiltonian, self.configs = model, hamiltonian, configs
    self.sums = torch.zeros(2, model.num_params, dtype=torch.float32, device=model.device)
    self.stats = torch.zeros(4, dtype=torch.float64, device=model.device)
    self.n_batches = 0

  def reset(self):
    self.sums.zero_()
    self.stats.zero_()
    self.n_batches = 0

  def accumulate(self, ham=None, packed=None):
    packed = self.configs.packed
    e = self.hamiltonian.local_value(self.model.wavefunction, self.configs).float().contiguous()
    self.model.weighted_grad_sum(packed, torch.stack([torch.ones_like(e), e]), self.sums)
    _native.energy_stats(e, self.stats)
    self.n_batches += 1
    return e

  mean_energy = engine.EnergyGradientSums.mean_energy
  gradient = engine.EnergyGradientSums.gradient


class WavefunctionOptimizer:
  """Parent class for ground state optimizers (training.py:94-132)."""

  def build_opt_ops(self, wavefunction, hamiltonian, hparams, shared_resources):
    raise NotImplementedError

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number=0):
    raise NotImplementedError


class EnergyGradientOptimizer(WavefunctionOptimizer):
  """Energy-gradient optimisation, training.py:506-623."""

  use_cuda_graph = True     # replay accumulate + sweep as one captured graph per batch

  def build_opt_ops(self, wavefunction, hamiltonian, hparams, shared_resources):
    n_sites = hparams.num_sites
    local_batch, walker_id0 = distributed.shard(hparams.batch_size)
    configs = graph_builders.get_configs(shared_resources, local_batch, n_sites,
                                         walker_id0=walker_id0)
    mc_step, acc_rate = graph_builders.get_monte_carlo_sampling(
        shared_resources, configs, wavefunction)
    model = _Model(wavefunction, n_sites, hparams)
    ansatz = model.ansatz
    ham = hamiltonian.native(n_sites)
    sums = (engine.EnergyGradientSums(ansatz, local_batch) if model.fast
            else _GenericEnergyGradientSums(model, hamiltonian, configs))
    # The walker-sharded totals live in their own buffers: the local
    # accumulators stay local, so metrics / apply_gradients may be run in the
    # middle of an epoch and accumulation continued (training.py:550-564 are
    # running means over every accumulate call since the last reset).
    state = {'reduced': False}
    if distributed.world_size() > 1:
      total = types.SimpleNamespace(sums=torch.zeros_like(sums.sums),
                                    stats=torch.zeros_like(sums.stats))
    else:
      total = sums

    def accumulate():                      # training.py:539-558, one batch
      sums.accumulate(ham, configs.packed)
      state['reduced'] = False

    def reduce_once():
      if total is not sums and not state['reduced']:
        distributed.allreduce_sums(sums.sums, sums.stats, total.sums, total.stats)
      state['reduced'] = True

    def global_gradient():                 # training.py:562-564 on the all-reduced sums
      nb = float(sums.n_batches)
      mean_e = (total.stats[0] / total.stats[2]).float()
      return total.sums[1] / nb - mean_e * total.sums[0] / nb

    def apply_gradients():                 # training.py:562-567
      reduce_once()
      if len(model.leaf_params) == 1:      # gradient formed inside the update kernel
        model.optimizers[0].apply_gradients(model.leaf_params[0], sums=total.sums, stats=total.stats,
                                            num_batches=sums.n_batches)
      else:
        model.apply_gradients(global_gradient())

    def metrics():                         # mean_energy, training.py:555, 582
      reduce_once()
      return float((total.stats[0] / total.stats[2]).item())

    def reset():                           # training.py:568
      sums.reset()
      state['reduced'] = False

    self.sums = sums
    n_sweep_steps = hparams.num_monte_carlo_sweeps * n_sites
    graphed = {}

    def batch_step():
      """accumulate_gradients followed by one sweep group (training.py:614-617)
      as one replayed CUDA graph around cgsvmc_batch_step."""
      if 'g' not in graphed:
        graphed['g'] = engine.GraphedBatchStep(configs.state, ansatz, ham, sums, n_sweep_steps)
      graphed['g'].replay()
      state['reduced'] = False

    def epoch_steps(n_batches):
      """The whole inner loop of run_optimization_epoch (training.py:614-617) as
      one replayed CUDA graph around cgsvmc_batch_steps: for the pure RBM ONE
      persistent kernel for all n_batches iterations."""
      key = ('e', int(n_batches))
      if key not in graphed:
        graphed[key] = engine.GraphedEpoch(configs.state, ansatz, ham, sums, n_sweep_steps, int(n_batches))
      graphed[key].replay()
      state['reduced'] = False

    host_stats = {}

    def epoch_end():
      """apply_gradients, metrics and reset_gradients (training.py:618-622) as
      one all-reduce (walker-sharded runs) + ONE kernel that also stores the
      energy statistics into pinned host memory; returns the mean energy."""
      if 'h' not in host_stats:
        host_stats['h'] = torch.zeros(4, dtype=torch.float64).pin_memory()
        host_stats['done'] = torch.cuda.Event()
      payload = None
      if total is not sums and not state['reduced']:
        payload = distributed.allreduce_payload(sums.sums, sums.stats)
      elif total is not sums:       # already reduced by a metrics / apply_gradients call of the caller
        payload = distributed.pack_sums(total.sums, total.stats)
      model.optimizers[0].epoch_end(model.leaf_params[0], sums.sums, sums.stats, sums.n_batches,
                                    host_stats['h'], total_payload=payload)
      host_stats['done'].record()
      sums.n_batches = 0
      state['reduced'] = False
      host_stats['done'].synchronize()
      h = host_stats['h']
      return float(h[0] / h[2])

    self._batch_step = Op(batch_step, 'batch_step') if (self.use_cuda_graph and model.fast) else None
    self._epoch_steps = Op(epoch_steps, 'epoch_steps') if (self.use_cuda_graph and model.fast) else None
    fusable = (self.use_cuda_graph and model.fast and len(model.leaf_params) == 1 and
               isinstance(model.optimizers[0], AdamOptimizer))
    self._epoch_end = Op(epoch_end, 'epoch_end') if fusable else None
    return TrainOpsTraditional(
        accumulate_gradients=Op(accumulate, 'accumulate_gradients'),
        apply_gradients=Op(apply_gradients, 'apply_gradients'),
        reset_gradients=Op(reset, 'reset_gradients'),
        mc_step=mc_step, acc_rate=acc_rate,
        metrics=Op(metrics, 'mean_energy'),
        epoch_increment=_epoch_increment(),
        update_wf_norm=_update_norm_op(wavefunction, configs))

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number=0):
    """training.py:589-623."""
    session.run(train_ops.mc_step,
                n_steps=hparams.num_equilibration_sweeps * hparams.num_sites)
    if train_ops.update_wf_norm is not None:
      session.run(train_ops.update_wf_norm)
    session.run(train_ops.reset_gradients)
    fused = getattr(self, '_batch_step', None)
    fused_epoch = getattr(self, '_epoch_steps', None)
    if fused_epoch is not None and hparams.num_batches_per_epoch > 0:
      # the loop below in one library call (same trajectories and local
      # energies as the per-batch launches, tests/test_gpu_rbm.py)
      session.run(fused_epoch, n_batches=hparams.num_batches_per_epoch)
    else:
      for _ in range(hparams.num_batches_per_epoch):
        if fused is not None:       # the same two ops, fused and graph-replayed
          session.run(fused)
        else:
          session.run(train_ops.accumulate_gradients)
          session.run(train_ops.mc_step,
                      n_steps=hparams.num_monte_carlo_sweeps * hparams.num_sites)
    fused_end = getattr(self, '_epoch_end', None)
    if fused_end is not None:     # the three ops below as one kernel
      energy = session.run(fused_end)
    else:
      session.run(train_ops.apply_gradients)
      energy = session.run(train_ops.metrics)
      session.run(train_ops.reset_gradients)
    session.run(train_ops.epoch_increment)
    return energy


def sr_matvec(ansatz, packed, o_mean, v, n_samples, diag_shift, allreduce=distributed.allreduce_):
  """(S + diag_shift I) v with S = <O O^T> - <O><O>^T over `n_samples` walkers,
  without forming S: y_b = O_b . v - <O> . v over the local walkers `packed`
  (one cgsvmc_log_amp_jvp launch), then sum_b y_b O_b (one
  cgsvmc_weighted_grad_sum launch), summed over the walker shards by
  `allreduce` (a float64 P-vector in, the sum over all shards out).  o_mean, v:
  float64 [P] on the device; returns float64 [P]."""
  y = ansatz.log_amp_jvp(packed, v.float())
  y = (y.double() - torch.dot(o_mean, v)).float()
  sv = ansatz.weighted_grad_sum(packed, y.reshape(1, -1))[0].double()
  return allreduce(sv) / n_samples + diag_shift * v


def conjugate_gradient(matvec, b, tolerance, max_iterations, check_every=5):
  """Solves A x = b for a symmetric positive definite A given as `matvec`,
  from x = 0, on b's device and dtype.  Stops once ||r|| <= tolerance ||b||,
  tested every `check_every` iterations (each test is one device-to-host
  read), or after `max_iterations`.  Returns (x, iterations, ||r|| / ||b||)
  with r the recursively updated residual."""
  x = torch.zeros_like(b)
  b_norm = float(torch.linalg.vector_norm(b))
  if b_norm == 0.0:
    return x, 0, 0.0
  tiny = torch.finfo(b.dtype).tiny
  r = b.clone()
  p = r.clone()
  rs = torch.dot(r, r)
  it = 0
  while it < max_iterations:
    ap = matvec(p)
    alpha = rs / torch.dot(p, ap).clamp_min(tiny)
    x.add_(alpha * p)
    r.sub_(alpha * ap)
    rs_new = torch.dot(r, r)
    it += 1
    if it % check_every == 0 and math.sqrt(float(rs_new)) <= tolerance * b_norm:
      rs = rs_new
      break
    p = r + (rs_new / rs.clamp_min(tiny)) * p
    rs = rs_new
  return x, it, math.sqrt(float(rs)) / b_norm


def _require_pure_rbm(wavefunction, n_sites):
  """Stochastic reconfiguration needs cgsvmc_log_amp_jvp, which is built for the
  pure RBM; checked before anything is allocated."""
  ok = (isinstance(wavefunction, wavefunctions.RestrictedBoltzmannNetwork) and
        wavefunction._num_layers == 0 and wavefunction._layer_size <= 256 and
        n_sites <= 256 and _native.n_words(n_sites) != 3)
  if not ok:
    raise NotImplementedError(
        'StochasticReconfiguration needs a single pure RBM: wavefunction_type=rbm with '
        'num_fc_layers=0, fc_layer_size <= 256 and num_sites <= 128 or 193..256 (got %s, num_sites=%d)'
        % (type(wavefunction).__name__, n_sites))


class StochasticReconfigurationOptimizer(WavefunctionOptimizer):
  """Stochastic reconfiguration (the natural gradient of VMC) for the pure RBM;
  the reference has no such optimizer.

  An epoch samples like EnergyGradientOptimizer.run_optimization_epoch (one
  captured cgsvmc_batch_step per batch) and keeps the configurations every
  batch is accumulated on.  With M the number of walkers of the epoch on all
  ranks, <.> the mean over them and O_b = d log psi_b / d params, it then
  solves
    (S + sr_diag_shift I) delta = F,
    S = <O O^T> - <O><O>^T,  F = <E O> - <E><O>
  by conjugate gradient (float64 vectors, x0 = 0, ||r|| <= sr_cg_tolerance ||F||
  or sr_cg_max_iterations), with S applied matrix-free (sr_matvec).  S and F
  are the textbook covariances, WITHOUT the factor B that
  EnergyGradientOptimizer's gradient carries.

  delta goes through hparams.optimizer: optimizer=gradient is classic SR,
  params -= lr delta, and is the recommended setting; with adam, Adam receives
  delta as its gradient.  After every solve `cg_iterations`, `cg_residual`
  (relative) and `direction` (delta) hold its result."""

  def build_opt_ops(self, wavefunction, hamiltonian, hparams, shared_resources):
    n_sites = hparams.num_sites
    _require_pure_rbm(wavefunction, n_sites)
    local_batch, walker_id0 = distributed.shard(hparams.batch_size)
    configs = graph_builders.get_configs(shared_resources, local_batch, n_sites,
                                         walker_id0=walker_id0)
    mc_step, acc_rate = graph_builders.get_monte_carlo_sampling(
        shared_resources, configs, wavefunction)
    model = _Model(wavefunction, n_sites, hparams)
    ansatz = model.ansatz
    ham = hamiltonian.native(n_sites)
    sums = engine.EnergyGradientSums(ansatz, local_batch)
    if distributed.world_size() > 1:
      total = types.SimpleNamespace(sums=torch.zeros_like(sums.sums),
                                    stats=torch.zeros_like(sums.stats))
    else:
      total = sums
    # the configurations of every batch since the last reset (1.3 MB at 6x6,
    # 8192 walkers, 20 batches)
    store = torch.empty(max(1, hparams.num_batches_per_epoch), local_batch, _native.n_words(n_sites),
                        dtype=torch.int64, device=model.device)
    state = {'reduced': False, 'stored': 0}
    diag_shift = float(hparams.sr_diag_shift)
    tolerance, max_iterations = float(hparams.sr_cg_tolerance), int(hparams.sr_cg_max_iterations)
    n_sweep_steps = hparams.num_monte_carlo_sweeps * n_sites
    graphed = {}

    def record():
      """Stores the configurations the next accumulation sees, on the stream
      that accumulation runs on."""
      k = state['stored']
      if k == store.shape[0]:
        raise RuntimeError('StochasticReconfiguration keeps %d batches (num_batches_per_epoch) per update: '
                           'apply or reset the gradients first' % k)
      store[k].copy_(configs.packed)
      state['stored'] = k + 1

    def accumulate():
      record()
      sums.accumulate(ham, configs.packed)
      state['reduced'] = False

    def batch_step():
      """accumulate_gradients followed by one sweep group, as one replayed
      CUDA graph around cgsvmc_batch_step."""
      if 'g' not in graphed:
        graphed['g'] = engine.GraphedBatchStep(configs.state, ansatz, ham, sums, n_sweep_steps)
      record()
      graphed['g'].replay()
      state['reduced'] = False

    def reduce_once():
      if total is not sums and not state['reduced']:
        distributed.allreduce_sums(sums.sums, sums.stats, total.sums, total.stats)
      state['reduced'] = True

    def solve():
      if state['stored'] == 0:
        raise RuntimeError('StochasticReconfiguration: no batch accumulated since the last reset')
      reduce_once()
      m = total.stats[2]
      s0, s1 = total.sums[0].double(), total.sums[1].double()
      o_mean = s0 / m
      forces = (s1 - total.stats[0] / m * s0) / m
      packed = store[:state['stored']].reshape(-1, store.shape[2])
      delta, self.cg_iterations, self.cg_residual = conjugate_gradient(
          lambda v: sr_matvec(ansatz, packed, o_mean, v, m, diag_shift), forces, tolerance, max_iterations)
      self.direction = delta
      return delta

    def apply_gradients():
      model.apply_gradients(solve().float())

    def metrics():
      reduce_once()
      return float((total.stats[0] / total.stats[2]).item())

    def reset():
      sums.reset()
      state['reduced'] = False
      state['stored'] = 0

    self.sums, self.sample_store, self.cg_iterations, self.cg_residual = sums, store, None, None
    self._batch_step, self._state = Op(batch_step, 'batch_step'), state
    return TrainOpsTraditional(
        accumulate_gradients=Op(accumulate, 'accumulate_gradients'),
        apply_gradients=Op(apply_gradients, 'apply_gradients'),
        reset_gradients=Op(reset, 'reset_gradients'),
        mc_step=mc_step, acc_rate=acc_rate,
        metrics=Op(metrics, 'mean_energy'),
        epoch_increment=_epoch_increment(),
        update_wf_norm=_update_norm_op(wavefunction, configs))

  def stored_configs(self):
    """The configurations accumulated since the last reset, int64 [M_local, W]."""
    return self.sample_store[:self._state['stored']].reshape(-1, self.sample_store.shape[2])

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number=0):
    """EnergyGradientOptimizer's epoch with the SR update; returns the mean
    energy of the epoch's samples."""
    session.run(train_ops.mc_step,
                n_steps=hparams.num_equilibration_sweeps * hparams.num_sites)
    if train_ops.update_wf_norm is not None:
      session.run(train_ops.update_wf_norm)
    session.run(train_ops.reset_gradients)
    for _ in range(hparams.num_batches_per_epoch):
      session.run(self._batch_step)
    session.run(train_ops.apply_gradients)
    energy = session.run(train_ops.metrics)
    session.run(train_ops.reset_gradients)
    session.run(train_ops.epoch_increment)
    return energy


class SupervisedWavefunctionOptimizer:
  """SWO with |psi|^2 sampling and the adjusted L2 loss, training.py:135-212.

  One batch = one sweep group + one optimizer step (training.py:208-212): the
  ratio psi_target sqrt(2^N) / psi, the loss and the gradient weights are one
  kernel (cgsvmc_swo_weights), the gradient one cgsvmc_weighted_grad_sum, the
  Adam update one cgsvmc_adam_step; nothing is read back to the host.  Because
  the parameters move every batch, the walker-sharded run all-reduces the
  P-vector gradient every batch -- that exchange is part of the algorithm.
  With `use_cuda_graph` (fast-path wavefunctions, Adam) sweep + train step are
  replayed as captured CUDA graphs (two halves around the all-reduce when
  sharded)."""

  use_cuda_graph = True

  def build_opt_ops(self, wavefunction, target_wavefunction, hparams, shared_resources):
    n_sites = hparams.num_sites
    local_batch, walker_id0 = distributed.shard(hparams.batch_size)
    configs = graph_builders.get_configs(shared_resources, local_batch, n_sites,
                                         walker_id0=walker_id0)
    mc_step, acc_rate = graph_builders.get_monte_carlo_sampling(
        shared_resources, configs, wavefunction)
    model = _Model(wavefunction, n_sites, hparams)
    target = _Model(target_wavefunction, n_sites)
    dev = model.device
    grad = torch.zeros(1, model.num_params, dtype=torch.float32, device=dev)
    weights = torch.zeros(1, local_batch, dtype=torch.float32, device=dev)
    loss_acc = torch.zeros(2, dtype=torch.float64, device=dev)      # sum (1 - r)^2, walkers
    log_norm = 0.5 * n_sites * math.log(2.0)       # sqrt(2^N), training.py:170
    total = float(hparams.batch_size)

    def loss_and_weights(acc):
      # r = psi_target * sqrt(2^N) / psi in the log domain; loss = mean (1 - r)^2
      z, sg = model.log_psi(configs.packed)
      zt, st = target.log_psi(configs.packed)
      signed = not (model.fast and target.fast)
      _native.swo_weights(z.contiguous(), zt.contiguous(), log_norm, total,
                          sign=sg.contiguous() if signed else None,
                          sign_target=st.contiguous() if signed else None,
                          out=weights, loss_acc=acc)

    def gradient():
      loss_and_weights(None)
      grad.zero_()
      model.weighted_grad_sum(configs.packed, weights, grad)

    def train_step():                      # optimizer.minimize(loss), training.py:175
      gradient()
      distributed.allreduce_(grad)
      model.apply_gradients(grad[0])

    def metrics():
      loss_acc.zero_()
      loss_and_weights(loss_acc)
      acc = distributed.allreduce_(loss_acc.clone())
      return float((acc[0] / acc[1]).item())

    # ---- captured batch: sweep group + train step ---------------------------
    n_sweep_steps = hparams.num_monte_carlo_sweeps * n_sites
    graphable = (self.use_cuda_graph and model.fast and target.fast and
                 all(isinstance(o, AdamOptimizer) for o in model.optimizers))
    captured = {}

    def capture():
      state, ansatz, opt, params = configs.state, model.ansatz, model.optimizers[0], model.leaf_params[0]
      opt.device_state(params)
      lib = _native.load()

      def front():       # sweep on the current parameters, then loss weights and the local gradient
        _native.check(lib.cgsvmc_ansatz_params_changed(ansatz._handle))    # tables follow the last update
        state.mc_steps_graph(ansatz, n_sweep_steps)
        gradient()

      def back():
        opt.apply_gradients_captured(params, grad[0])

      state.step_dev.fill_(state.step)
      saved = (state.packed.clone(), state.accept_count.clone(), params.clone(), opt.m.clone(),
               opt.v.clone(), opt.t_dev.clone())
      side = torch.cuda.Stream(device=dev)
      side.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(side):        # warm-up sizes every scratch buffer
        front(); back()
      torch.cuda.current_stream().wait_stream(side)
      torch.cuda.synchronize()
      for dst, src in zip((state.packed, state.accept_count, params, opt.m, opt.v, opt.t_dev), saved):
        dst.copy_(src)
      state.step_dev.fill_(state.step)
      graphs = []
      sharded = distributed.world_size() > 1
      for body in ((front, back) if sharded else (lambda: (front(), back()),)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
          body()
        graphs.append(g)
      captured.update(graphs=graphs, sharded=sharded, opt=opt, state=state, params=params)

    def batch_step():
      """One iteration of training.py:208-212."""
      if not captured:
        try:
          capture()
        except NotImplementedError:        # no capturable sampler for this shape: the two ops, eagerly
          captured['eager'] = True
      if captured.get('eager'):
        mc_step(n_steps=n_sweep_steps)
        train_step()
        return
      state, opt = captured['state'], captured['opt']
      if state.step != captured.get('expected_step'):
        state.step_dev.fill_(state.step)
      opt.sync_device(1)
      captured['graphs'][0].replay()
      if captured['sharded']:
        distributed.allreduce_(grad)
        captured['graphs'][1].replay()
      torch.autograd.graph.increment_version(captured['params'])
      state.step += n_sweep_steps
      state.proposed += n_sweep_steps * state.batch_size
      captured['expected_step'] = state.step

    self._batch_step = Op(batch_step, 'batch_step') if graphable else None
    return TrainOpsSupervised(
        accumulate_gradients=None, apply_gradients=Op(train_step, 'train_step'),
        reset_gradients=None, mc_step=mc_step, acc_rate=acc_rate,
        metrics=Op(metrics, 'loss'), update_wf_norm=None,
        epoch_increment=_epoch_increment())

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number):
    """training.py:192-212."""
    del epoch_number
    fused = getattr(self, '_batch_step', None)
    for _ in range(hparams.num_batches_per_epoch):
      if fused is not None:       # the same two ops as one replayed graph
        session.run(fused)
        continue
      session.run(train_ops.mc_step,
                  n_steps=hparams.num_monte_carlo_sweeps * hparams.num_sites)
      session.run(train_ops.apply_gradients)
    session.run(train_ops.epoch_increment)


class _OverlapSums:
  """Accumulators of the log-overlap gradient shared by LogOverlapSWO and
  LogOverlapImaginaryTimeSWO (training.py:336-360, 672-699): with O_b =
  d log psi_b and a per-walker ratio r_b,
    g = mean_batches(sum_b O_b) - mean_batches(sum_b r_b O_b) / mean_samples(r)
  (tf.gradients sums over the batch, tf.metrics.mean_tensor averages over
  accumulate calls, tf.metrics.mean over samples).  One packed float32 buffer
  [2P + 4] = [S_1 | S_r | sum r, sum e, n, 0] is the all-reduce payload."""

  def __init__(self, model, local_batch):
    dev = model.device
    self.model, self.P = model, model.num_params
    self.buf = torch.zeros(2 * self.P + 4, dtype=torch.float32, device=dev)
    self.sums = self.buf[:2 * self.P].view(2, self.P)
    self.tail = self.buf[2 * self.P:]
    self.scratch = torch.zeros(2, self.P, dtype=torch.float32, device=dev)
    self.weights = torch.ones(2, local_batch, dtype=torch.float32, device=dev)
    self.n_batches = 0
    self.reduced = False

  def reset(self):
    self.buf.zero_()
    self.n_batches = 0
    self.reduced = False

  def accumulate(self, packed, ratio, energy=None):
    self.weights[1].copy_(ratio)
    self.scratch.zero_()
    self.model.weighted_grad_sum(packed, self.weights, self.scratch)
    self.sums.add_(self.scratch)
    self.tail[0] += ratio.sum()
    if energy is not None:
      self.tail[1] += energy.sum()
    self.tail[2] += float(ratio.numel())
    self.n_batches += 1
    self.reduced = False

  def _reduce(self):
    if not self.reduced:
      distributed.allreduce_(self.buf)
      self.reduced = True

  def gradient(self):
    self._reduce()
    nb = float(self.n_batches)
    mean_ratio = self.tail[0] / self.tail[2]
    return self.sums[0] / nb - (self.sums[1] / nb) / mean_ratio

  def mean_energy(self):
    self._reduce()
    return float((self.tail[1] / self.tail[2]).item())


class LogOverlapSWO:
  """SWO with |psi|^2 sampling and log |<psi|phi>|^2 as the objective,
  training.py:298-404."""

  def build_opt_ops(self, wavefunction, target_wavefunction, hparams, shared_resources):
    n_sites = hparams.num_sites
    local_batch, walker_id0 = distributed.shard(hparams.batch_size)
    configs = graph_builders.get_configs(shared_resources, local_batch, n_sites,
                                         walker_id0=walker_id0)
    mc_step, acc_rate = graph_builders.get_monte_carlo_sampling(
        shared_resources, configs, wavefunction)
    model = _Model(wavefunction, n_sites, hparams)
    target = _Model(target_wavefunction, n_sites)
    sums = _OverlapSums(model, local_batch)

    def accumulate():                      # ratio = psi_target / psi, training.py:339
      z, sg = model.log_psi(configs.packed)
      zt, st = target.log_psi(configs.packed)
      sums.accumulate(configs.packed, sg * st * torch.exp(zt - z))

    def apply_gradients():                 # training.py:358-362
      model.apply_gradients(sums.gradient())

    self.sums = sums
    return TrainOpsSupervised(
        accumulate_gradients=Op(accumulate, 'accumulate_gradients'),
        apply_gradients=Op(apply_gradients, 'apply_gradients'),
        reset_gradients=Op(sums.reset, 'reset_gradients'),
        mc_step=mc_step, acc_rate=acc_rate, metrics=None,
        update_wf_norm=_update_norm_op(wavefunction, configs),
        epoch_increment=_epoch_increment())

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number):
    """training.py:382-404."""
    del epoch_number
    for _ in range(hparams.num_batches_per_epoch):
      session.run(train_ops.mc_step,
                  n_steps=hparams.num_monte_carlo_sweeps * hparams.num_sites)
      session.run(train_ops.reset_gradients)
      session.run(train_ops.accumulate_gradients)
      session.run(train_ops.apply_gradients)
    session.run(train_ops.epoch_increment)


class DualSamplingSWO:
  """SWO sampling |psi|^2 of both the trainee and the target with the plain
  L2 loss mean (psi - t)^2, training.py:407-503."""

  TARGET_SEED_XOR = 0x7A46E7      # the target walkers get their own Philox key

  def build_opt_ops(self, wavefunction, target_wavefunction, hparams, shared_resources):
    n_sites = hparams.num_sites
    local_half, walker_id0 = distributed.shard(hparams.batch_size // 2)
    psi_configs = graph_builders.get_configs(shared_resources, local_half, n_sites,
                                             walker_id0=walker_id0)
    target_configs = graph_builders.get_configs(
        shared_resources, local_half, n_sites,
        configs_id=graph_builders.ResourceName.TARGET_CONFIGS,
        seed=0xC65 ^ self.TARGET_SEED_XOR, walker_id0=walker_id0)
    # explicit, separate samplers for the two wavefunctions (training.py:441-447)
    target_mc_step, target_acc = graph_builders.build_monte_carlo_sampling(
        target_configs, target_wavefunction)
    psi_mc_step, psi_acc = graph_builders.build_monte_carlo_sampling(psi_configs, wavefunction)
    model = _Model(wavefunction, n_sites, hparams)
    target = _Model(target_wavefunction, n_sites)
    grad = torch.zeros(1, model.num_params, dtype=torch.float32, device=model.device)
    log_norm = 0.5 * n_sites * math.log(2.0)       # sqrt(2^N), training.py:451
    total = float(2 * local_half * distributed.world_size())

    def mc_step(n_steps=1):
      psi_mc_step(n_steps=n_steps)
      target_mc_step(n_steps=n_steps)

    def acc_rate():
      return [psi_acc(), target_acc()]

    def loss_and_weights():
      packed = torch.cat([psi_configs.packed, target_configs.packed], dim=0)
      z, sg = model.log_psi(packed)
      zt, st = target.log_psi(packed)
      psi = sg * torch.exp(z)
      t = st * torch.exp(zt + log_norm)
      diff = psi - t
      loss = (diff * diff).sum() / total                 # training.py:461-463
      weights = (2.0 * diff * psi / total).reshape(1, -1).contiguous()
      return packed, loss, weights

    def train_step():                      # optimizer.minimize(loss), training.py:466
      packed, loss, weights = loss_and_weights()
      grad.zero_()
      model.weighted_grad_sum(packed, weights, grad)
      distributed.allreduce_(grad)
      model.apply_gradients(grad[0])
      return loss

    def metrics():
      _, loss, _ = loss_and_weights()
      return float(distributed.allreduce_(loss.clone()).item())

    self.loss_and_weights, self.model = loss_and_weights, model
    return TrainOpsSupervised(
        accumulate_gradients=None, apply_gradients=Op(train_step, 'train_step'),
        reset_gradients=None, mc_step=Op(mc_step, 'mc_step'), acc_rate=Op(acc_rate, 'acc_rate'),
        metrics=Op(metrics, 'loss'), update_wf_norm=None,
        epoch_increment=_epoch_increment())

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number):
    """training.py:483-503."""
    del epoch_number
    for _ in range(hparams.num_batches_per_epoch):
      session.run(train_ops.mc_step,
                  n_steps=hparams.num_monte_carlo_sweeps * hparams.num_sites)
      session.run(train_ops.apply_gradients)
    session.run(train_ops.epoch_increment)


class LogOverlapImaginaryTimeSWO(WavefunctionOptimizer):
  """Imaginary-time SWO through the log-overlap gradient, training.py:626-778:
  the supervisor psi_O is a deep copy of the trainee refreshed once per epoch
  and the target is (1 - beta H) psi_O."""

  def build_opt_ops(self, wavefunction, hamiltonian, hparams, shared_resources):
    n_sites = hparams.num_sites
    local_batch, walker_id0 = distributed.shard(hparams.batch_size)
    configs = graph_builders.get_configs(shared_resources, local_batch, n_sites,
                                         walker_id0=walker_id0)
    mc_step, acc_rate = graph_builders.get_monte_carlo_sampling(
        shared_resources, configs, wavefunction)
    model = _Model(wavefunction, n_sites, hparams)
    wf_omega = copy.deepcopy(wavefunction)        # supervisor, training.py:661
    wf_omega.connect(n_sites)
    beta = float(hparams.time_evolution_beta)
    sums = _OverlapSums(model, local_batch)

    def accumulate():
      # H psi_O = E_loc[psi_O] psi_O (apply_in_place, operators.py:261-271), so
      # ratio = (psi_O - beta H psi_O) / psi = (psi_O / psi) (1 - beta E_O)
      e_omega, z_omega, s_omega, _, _ = hamiltonian._evaluate(wf_omega, configs)
      z, sg = model.log_psi(configs.packed)
      ratio = sg * s_omega * torch.exp(z_omega - z) * (1.0 - beta * e_omega)
      sums.accumulate(configs.packed, ratio, energy=e_omega)

    def apply_gradients():                 # training.py:693-701
      model.apply_gradients(sums.gradient())

    self.sums, self.supervisor = sums, wf_omega
    return TrainOpsSWO(
        train_step=None,
        accumulate_gradients=Op(accumulate, 'accumulate_gradients'),
        apply_gradients=Op(apply_gradients, 'apply_gradients'),
        reset_gradients=Op(sums.reset, 'reset_gradients'),
        mc_step=mc_step, acc_rate=acc_rate, metrics=None,
        energy=Op(sums.mean_energy, 'mean_energy'),
        update_supervisor=wavefunctions.module_transfer_ops(wavefunction, wf_omega),
        update_normalization=None,
        epoch_increment=_epoch_increment(),
        update_wf_norm=_update_norm_op(wavefunction, configs))

  def run_optimization_epoch(self, train_ops, session, hparams, epoch_number=0):
    """training.py:729-778."""
    session.run(train_ops.mc_step,
                n_steps=hparams.num_equilibration_sweeps * hparams.num_sites)
    if train_ops.update_wf_norm is not None:
      session.run(train_ops.update_wf_norm)
    session.run(train_ops.update_supervisor)
    for _ in range(hparams.num_batches_per_epoch):
      session.run(train_ops.mc_step,
                  n_steps=hparams.num_monte_carlo_sweeps * hparams.num_sites)
      session.run(train_ops.reset_gradients)
      session.run(train_ops.accumulate_gradients)
      session.run(train_ops.apply_gradients)
    session.run(train_ops.epoch_increment)
    return session.run(train_ops.energy)


def _not_built(name, why):
  class _NotBuilt:
    def __init__(self, *args, **kwargs):
      raise NotImplementedError('%s: %s' % (name, why))
  _NotBuilt.__name__ = name
  return _NotBuilt


GROUND_STATE_OPTIMIZERS = {     # training.py:913-917
    'EnergyGradient': EnergyGradientOptimizer,
    'LogOverlapITSWO': LogOverlapImaginaryTimeSWO,
    'ITSWO': _not_built('ImaginaryTimeSWO',
                        'raises AttributeError at graph build in the reference '
                        '(hparams.time_evolution_befta, training.py:812)'),
}

# Ground-state optimizers the reference does not have.  They are kept apart so
# that GROUND_STATE_OPTIMIZERS names exactly what the reference registers;
# ground_state_optimizer() and run_training.py --optimizer take both.
EXTRA_GROUND_STATE_OPTIMIZERS = {
    'StochasticReconfiguration': StochasticReconfigurationOptimizer,
}


def ground_state_optimizer(name):
  """The ground-state optimizer class registered under `name`."""
  if name in GROUND_STATE_OPTIMIZERS:
    return GROUND_STATE_OPTIMIZERS[name]
  if name in EXTRA_GROUND_STATE_OPTIMIZERS:
    return EXTRA_GROUND_STATE_OPTIMIZERS[name]
  raise KeyError('unknown ground-state optimizer %r: one of %s' % (
      name, sorted(GROUND_STATE_OPTIMIZERS) + sorted(EXTRA_GROUND_STATE_OPTIMIZERS)))

SUPERVISED_OPTIMIZERS = {       # training.py:920-925
    'SWO': SupervisedWavefunctionOptimizer,
    'LogOverlapSWO': LogOverlapSWO,
    'DualSamplingSWO': DualSamplingSWO,
    'BasisIterSWO': _not_built('BasisIterationSWO',
                               'calls the non-existent scipy.special.binomi in the reference '
                               '(training.py:246)'),
}
