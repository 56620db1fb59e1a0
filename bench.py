#!/usr/bin/env python
"""Benchmark of the VMC hot path (BASELINE.json metric: walker-steps/sec and
E_loc evals/sec).  Headline workload C2 = 6x6 Heisenberg, RBM (H = 144), 8192
walkers per GPU; the other BASELINE configurations (C1, C3, C4, C5) are
measured the same way and reported as keyed sub-results of the one JSON line.

A "step" is one batch iteration of EnergyGradientOptimizer.run_optimization_epoch
(training.py:614-617): `accumulate_gradients` (local energy of every walker,
the two gradient sums, energy statistics) followed by one Monte-Carlo sweep
(num_monte_carlo_sweeps * num_sites Metropolis steps per walker).  The timed
region runs WHOLE EPOCHS: after every min(50, steps) steps the epoch end of
training.py:618-622 -- all-reduce of the [2P + 4] payload over the walker
shards, gradient + Adam update, read-back of the mean energy, reset, and the
rebuild of the derived parameter tables in the next step -- is inside the
timed region, whatever --steps is.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--dump-outputs DIR]

Prints one JSON line (see DESIGN.md section "Measurement" for every field).
--dump-outputs DIR also writes what the timed headline run left its caller
after the last timed step as DIR/<name>.npy (see dump_outputs); the inputs are
seeded, so two builds run with the same arguments can be compared array by
array.
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOAD = 'C2: 6x6 square-lattice Heisenberg (72 NN bonds, jx=-1, jz=1), rbm H=144, 8192 walkers/GPU'
N_SITES, SIZE, HIDDEN, WALKERS = 36, 6, 144, 8192
SWEEP_STEPS = N_SITES            # num_monte_carlo_sweeps (1) * num_sites
SEED = 0xC65
EPOCH_BATCHES = 50               # num_batches_per_epoch default (utils.py:132-138)
L2_FLUSH_BYTES = 256 << 20
DUMP_CONFIG_BYTES = 32 << 20     # --dump-outputs: larger walker sets are written as a seeded row sample

# The BASELINE.json configurations (SURVEY.md 8(a) sizes, 8(d) synthetic inputs).
# walkers = per GPU; max_steps bounds the timed steps of the slow configurations
# so that the default run stays within a few minutes.
CONFIGS = {
    'C1': dict(desc='C1: chain-20 Heisenberg (20 bonds), fully_connected 20-80-80-80-1, 1024 walkers/GPU',
               hp=dict(wavefunction_type='fully_connected', num_sites=20, num_fc_layers=3, fc_layer_size=80),
               lattice='chain', walkers=1024, f_fwd=28960, f_inc=26080, max_steps=200),
    'C2': dict(desc=WORKLOAD,
               hp=dict(wavefunction_type='rbm', num_sites=36, size_x=6, size_y=6, num_fc_layers=0,
                       fc_layer_size=HIDDEN),
               lattice='square', walkers=WALKERS, max_steps=1 << 30),
    'C3': dict(desc='C3: 10x10 J1-J2 (J2=0.5, 400 bonds), conv_2d 5 layers x 16 filters x 5x5, 8192 walkers/GPU '
                    '(65536 over 8 GPUs)',
               hp=dict(wavefunction_type='conv_2d', num_sites=100, size_x=10, size_y=10, num_conv_layers=5,
                       num_conv_filters=16, kernel_size=5),
               lattice='j1j2', walkers=8192, f_fwd=5.2e6, max_steps=6),
    'C4': dict(desc='C4: SWO (SupervisedWavefunctionOptimizer) on 6x6, conv_2d 5x16x5x5 trainee vs a fixed '
                    'conv_2d target, 8192 walkers/GPU',
               hp=dict(wavefunction_type='conv_2d', num_sites=36, size_x=6, size_y=6, num_conv_layers=5,
                       num_conv_filters=16, kernel_size=5),
               lattice=None, walkers=8192, f_fwd=1.872e6, max_steps=10),
    'C5': dict(desc='C5: 16x16 Heisenberg (512 bonds), rbm H=256, 131072 walkers/GPU (1M over 8 GPUs)',
               hp=dict(wavefunction_type='rbm', num_sites=256, size_x=16, size_y=16, num_fc_layers=0,
                       fc_layer_size=256),
               lattice='square', walkers=131072, max_steps=20),
}


def parse_args():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=200)
  ap.add_argument('--warmup', type=int, default=20)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--walkers', type=int, default=WALKERS, help='walkers per GPU (C2)')
  ap.add_argument('--configs', default='C1,C3,C4,C5',
                  help='other BASELINE configurations to report as sub-results ("" = none)')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write the outputs of the last timed C2 step as DIR/<name>.npy (rank 0; --impl ours)')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs applies to --impl ours')
  return args


def peaks():
  path = os.path.join(REPO, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    p = json.load(open(path))
    return dict(hbm_gbs=p['hbm_gbs'], sm_max_mhz=p.get('sm_max_mhz', 1965.0),
                bf16_tflops=p.get('bf16_tflops', 1590.0),
                bf16_tflops_sustained=p.get('bf16_tflops_sustained', 1400.0), source='measured')
  return dict(hbm_gbs=6650.0, sm_max_mhz=1965.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0,
              source='fallback')


def bonds_for(cfg):
  from cgs_vmc_b200 import lattices
  hp = cfg['hp']
  if cfg['lattice'] == 'chain':
    return lattices.heisenberg_couplings(lattices.chain_bonds(hp['num_sites']), -1.0, 1.0)
  if cfg['lattice'] == 'square':
    return lattices.heisenberg_couplings(lattices.square_nn_bonds(hp['size_x']), -1.0, 1.0)
  if cfg['lattice'] == 'j1j2':
    return lattices.j1j2_couplings(hp['size_x'], 0.5)
  raise ValueError(cfg['lattice'])


def config_dict(walkers):
  """The `config` object of the JSON line -- identical for both arms."""
  return {'workload': WORKLOAD, 'walkers_per_gpu': walkers, 'mc_steps_per_step': SWEEP_STEPS, 'n_bonds': 72}


# ----------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------
class ClockSampler:
  """Samples SM clock and throttle reasons through NVML from a background
  thread while the timed region runs (the region lasts milliseconds, far below
  nvidia-smi's own start-up time, so the CLI loop of the profiling recipe
  cannot be used here; the NVML fields are the same ones it prints)."""

  def __init__(self, index, period_s=0.002):
    import threading
    self.samples, self.max_mhz, self.reasons = [], None, set()
    self._stop = threading.Event()
    self._thread = None
    try:
      import pynvml
      pynvml.nvmlInit()
      self._nv = pynvml
      self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
    except Exception:   # NVML unavailable: report nulls
      self._nv = None
      return
    self._period = period_s
    self._thread = threading.Thread(target=self._run, daemon=True)
    self._thread.start()

  def _run(self):
    nv = self._nv
    names = {
        'hw_slowdown': nv.nvmlClocksThrottleReasonHwSlowdown,
        'hw_thermal_slowdown': nv.nvmlClocksThrottleReasonHwThermalSlowdown,
        'sw_thermal_slowdown': nv.nvmlClocksThrottleReasonSwThermalSlowdown,
        'sw_power_cap': nv.nvmlClocksThrottleReasonSwPowerCap,
    }
    while not self._stop.is_set():
      try:
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for k, bit in names.items():
          if mask & bit:
            self.reasons.add(k)
      except Exception:
        pass
      self._stop.wait(self._period)

  def stop(self):
    if self._thread is not None:
      self._stop.set()
      self._thread.join(timeout=2)
    sm = float(np.median(self.samples)) if self.samples else None
    return dict(sm_mhz=sm, sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons),
                samples=len(self.samples))


# ----------------------------------------------------------------------------
# CPU arm: the reference-equivalent op sequence on the host cores
# ----------------------------------------------------------------------------
def cpu_arm(name, walkers, steps, warmup):
  """Times oracle/cpu_baseline.py (the reference's op sequence in torch-CPU
  float32 on all host threads) on configuration `name` with `walkers` walkers
  per step."""
  from cgs_vmc_b200 import wavefunctions
  from oracle import ansatz as oansatz
  from oracle import bits, cpu_baseline
  cfg = CONFIGS[name]
  hp = cfg['hp']
  n = hp['num_sites']
  if hp['wavefunction_type'] in ('fully_connected', 'rbm'):
    spec = oansatz.AnsatzSpec(hp['wavefunction_type'], n, num_layers=hp['num_fc_layers'],
                              layer_size=hp['fc_layer_size'], size_x=hp.get('size_x', 1),
                              size_y=hp.get('size_y', 1))
  else:
    spec = oansatz.AnsatzSpec(hp['wavefunction_type'], n, num_layers=hp['num_conv_layers'],
                              num_filters=hp['num_conv_filters'], kernel_size=hp['kernel_size'],
                              size_x=hp['size_x'], size_y=hp['size_y'])
  gen = torch.Generator().manual_seed(1234)
  shapes = [tuple(s) for _, s in oansatz.param_shapes(spec)]
  flat = torch.cat([t.reshape(-1) for t in wavefunctions._sonnet_init(shapes, gen)]).float()
  ij, jx, jz = bonds_for(cfg)
  cores = os.cpu_count() or 1
  torch.set_num_threads(cores)
  configs = bits.random_sz0_configs(n, walkers, np.random.default_rng(1234))
  vmc = cpu_baseline.ReferenceEquivalentVMC(spec, flat, ij, jx, jz, configs, seed=SEED)
  times = cpu_baseline.time_steps(vmc, n, steps, warmup)
  t = float(np.mean(times))
  return dict(walker_steps_per_sec=walkers * n / t, eloc_evals_per_sec=walkers / t,
              ms_per_step=t * 1e3, cores=cores, walkers=walkers, steps=steps)


def run_reference(args, rank):
  """--impl reference: the reference's CPU implementation of the same step.
  TensorFlow 1.x / Sonnet v1 are not installable in this image, so this is
  the op-for-op torch-CPU restatement (oracle/cpu_baseline.py, kind "port").
  Under torchrun only rank 0 works."""
  if rank != 0:
    return
  # bounded sample: the full batch per step unless K steps of it would exceed
  # ~4 minutes on this host (probed with one step); then 2048 walkers per step
  # and per-walker throughput is what is reported
  probe = cpu_arm('C2', args.walkers, 1, 0)
  budget_s = 240.0
  fits = probe['ms_per_step'] * 1e-3 * (args.steps + args.warmup) <= budget_s
  sample_walkers = args.walkers if fits else min(args.walkers, 2048)
  r = cpu_arm('C2', sample_walkers, args.steps, args.warmup)
  line = {
      'impl': 'reference', 'metric': 'walker_steps_per_sec', 'value': r['walker_steps_per_sec'],
      'unit': 'walker-steps/s', 'eloc_evals_per_sec': r['eloc_evals_per_sec'],
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': config_dict(args.walkers),
      'cpu_baseline': {'value': r['walker_steps_per_sec'], 'unit': 'walker-steps/s',
                       'cores': r['cores'], 'kind': 'port',
                       'sample': '%d steps of the same workload on %d of the %d walkers per step, '
                                 'torch-CPU float32 restatement of the TF graph, all host threads'
                                 % (args.steps, sample_walkers, args.walkers)},
      'e2e': {'value': r['walker_steps_per_sec'], 'unit': 'walker-steps/s',
              'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  print(json.dumps(line))


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------
def ev():
  return torch.cuda.Event(enable_timing=True)


def max_over_ranks(value, dev, world):
  t = torch.tensor([value], dtype=torch.float64, device=dev)
  if world > 1:
    import torch.distributed as dist
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  return float(t.item())


class EnergyGradientWorkload:
  """One walker shard of an EnergyGradient run on the engine-level pieces the
  public optimizer is made of (training.EnergyGradientOptimizer): captured
  batch step, float64 all-reduce of the sums, gradient + Adam in one kernel."""

  def __init__(self, name, walkers, rank, world, dev):
    from cgs_vmc_b200 import _native, engine, training, utils, wavefunctions
    cfg = CONFIGS[name]
    self.name, self.cfg, self.B, self.rank, self.world, self.dev = name, cfg, walkers, rank, world, dev
    hp = utils.create_hparams(batch_size=walkers * world, **cfg['hp'])
    self.hp = hp
    self.n = hp.num_sites
    self.sweep_steps = hp.num_monte_carlo_sweeps * self.n
    # Sonnet-default parameters (truncated normal, sigma = 1/sqrt(fan_in), zero
    # biases) from torch.Generator seed 1234, SURVEY.md 8(d)
    self.wf = wavefunctions.build_wavefunction(hp).seed(1234)
    self.ansatz = self.wf.native(self.n)
    self.ij, jx, jz = bonds_for(cfg)
    self.ham = _native.Hamiltonian(self.ij, jx, jz, self.n, device=dev)
    self.state = engine.WalkerState(walkers, self.n, seed=SEED, walker_id0=rank * walkers, device=dev)
    self.sums = engine.EnergyGradientSums(self.ansatz, walkers, device=dev)
    self.opt = training.AdamOptimizer(hp)
    P = self.ansatz.num_params
    self.host_stats = torch.zeros(4, dtype=torch.float64).pin_memory()
    self.state.mc_steps(self.ansatz, 20 * self.n if name in ('C1', 'C2') else self.n)   # equilibrate a little
    self.graphed = engine.GraphedBatchStep(self.state, self.ansatz, self.ham, self.sums, self.sweep_steps)
    self.fused = self.ansatz.kind == 'rbm' and hp.num_fc_layers == 0
    self.epochs = {}
    self.launches = 0
    self.allreduce_ms = []
    self.energies = []

  def step(self):
    version = self.ansatz.params._version
    rebuilt = getattr(self, '_seen_version', None) != version
    self._seen_version = version
    self.graphed.replay()
    # pure RBM: ONE kernel (estimators + sweep + cross-CTA reduction; + table
    # build and bond-pair table after a parameter update); tile networks: fill,
    # local energy, copy, gradient, reduction, statistics, sampler, counter
    self.launches += (1 + (2 if rebuilt else 0)) if self.fused else 8

  def prepare_epoch(self, n_batches):
    """Pure RBM: the n_batches batch iterations of an epoch as ONE persistent
    kernel (cgsvmc_batch_steps, engine.GraphedEpoch)."""
    from cgs_vmc_b200 import engine
    if not self.fused or n_batches < 2 or os.environ.get('CGSVMC_BENCH_PER_STEP') == '1':
      return False
    if n_batches not in self.epochs:
      self.epochs[n_batches] = engine.GraphedEpoch(self.state, self.ansatz, self.ham, self.sums,
                                                   self.sweep_steps, n_batches)
    return True

  def run_epoch(self, n_batches):
    version = self.ansatz.params._version
    rebuilt = getattr(self, '_seen_version', None) != version
    self._seen_version = version
    self.epochs[n_batches].replay()
    self.launches += 1 + (2 if rebuilt else 0)

  def epoch_end(self):
    """training.py:618-622: apply_gradients (all-reduce over the walker shards,
    gradient, Adam), metrics (mean energy read back), reset_gradients -- the
    float64 all-reduce (N > 1) + ONE kernel (cgsvmc_epoch_end) that reads the
    all-reduced payload, applies the Adam step, stores the energy statistics
    into pinned host memory and zeroes the accumulators; the same call
    EnergyGradientOptimizer.run_optimization_epoch makes."""
    from cgs_vmc_b200 import distributed
    a0, a1 = ev(), ev()
    a0.record()
    payload = distributed.allreduce_payload(self.sums.sums, self.sums.stats) if self.world > 1 else None
    a1.record()
    self.opt.epoch_end(self.ansatz.params, self.sums.sums, self.sums.stats, self.sums.n_batches,
                       self.host_stats, total_payload=payload)
    done = torch.cuda.Event()
    done.record()
    self.sums.n_batches = 0
    done.synchronize()                      # session.run(metrics) returns the energy to the host
    self.energies.append(float(self.host_stats[0] / self.host_stats[2]))
    self.allreduce_ms.append((a0, a1))
    self.launches += 1

  def n_active_bonds(self):
    mask, _ = self.ham.flip_enum(self.state.packed[:512], want_flipped=False)
    words = mask.cpu().numpy().reshape(-1).astype(np.int64) & 0xffffffff
    return float(sum(bin(int(v)).count('1') for v in words)) / min(self.B, 512)


class SupervisedWorkload:
  """C4: SupervisedWavefunctionOptimizer through the public API
  (training.py:135-212): one step = one sweep group + one train step (loss
  weights, gradient, all-reduce of the gradient over the shards, Adam)."""

  def __init__(self, name, walkers, rank, world, dev):
    from cgs_vmc_b200 import graph_builders, training, utils, wavefunctions
    from cgs_vmc_b200.session import Session
    cfg = CONFIGS[name]
    self.name, self.cfg, self.B, self.rank, self.world, self.dev = name, cfg, walkers, rank, world, dev
    hp = utils.create_hparams(batch_size=walkers * world, num_batches_per_epoch=1, **cfg['hp'])
    self.hp, self.n = hp, hp.num_sites
    self.sweep_steps = hp.num_monte_carlo_sweeps * self.n
    self.wf = wavefunctions.build_wavefunction(hp).seed(1234)
    self.target = wavefunctions.build_wavefunction(hp).seed(4321)
    self.ansatz = self.wf.native(self.n)
    self.target.native(self.n)
    self.opt = training.SupervisedWavefunctionOptimizer()
    self.shared = {}
    self.ops = self.opt.build_opt_ops(wavefunction=self.wf, target_wavefunction=self.target, hparams=hp,
                                      shared_resources=self.shared)
    self.session = Session()
    self.configs = self.shared[graph_builders.ResourceName.CONFIGS]
    self.session.run(self.ops.mc_step, n_steps=self.n)
    # bring psi_target sqrt(2^N) to the trainee's scale so the loss is O(1)
    z = self.wf.log_amplitude(self.configs)
    zt = self.target.log_amplitude(self.configs)
    offset = (zt - z).double().mean().reshape(1)
    from cgs_vmc_b200 import distributed
    distributed.allreduce_(offset)
    self.target._exp_norm_shift += float(offset.item()) / world + 0.5 * self.n * math.log(2.0)
    self.launches = 0
    self.allreduce_ms = []
    self.energies = []
    self.fused = False

  def step(self):
    if self.opt._batch_step is not None:
      self.session.run(self.opt._batch_step)
    else:
      self.session.run(self.ops.mc_step, n_steps=self.sweep_steps)
      self.session.run(self.ops.apply_gradients)
    self.launches += 9    # sampler, counter, 2 x amplitudes, loss weights, gradient, reduction, Adam, counter

  def epoch_end(self):
    self.energies.append(self.session.run(self.ops.metrics))      # the loss, read back like the driver does
    self.launches += 3

  def n_active_bonds(self):
    return 0.0


def time_workload(w, steps, warmup, flush, world, dev, clock_index=None, force_per_step=False):
  """W warm-up steps (with one epoch end), then K steps in epochs of
  min(EPOCH_BATCHES, K) with the epoch end inside the timed region.  Returns
  device times (max over ranks).  Pure RBM: the batch iterations of an epoch
  are ONE launch (persistent kernel, cgsvmc_batch_steps); the event pairs then
  bracket whole epochs and the L2 flush sits between launches."""
  import torch.distributed as dist
  epoch_len = max(1, min(EPOCH_BATCHES, steps))
  per_epoch = not force_per_step and hasattr(w, 'prepare_epoch') and w.prepare_epoch(epoch_len)
  for _ in range(max(warmup, 3)):
    w.step()
    flush.zero_()
  w.epoch_end()
  w.step()                                 # the rebuilding variant of the step, once
  flush.zero_()
  w.epoch_end()
  tail = steps % epoch_len               # a shorter last epoch gets its own captured launch
  tail_epoch = per_epoch and tail >= 2 and w.prepare_epoch(tail)
  if per_epoch:
    for _ in range(2):                     # and of the epoch launch
      w.run_epoch(epoch_len)
      flush.zero_()
      w.epoch_end()
    if tail_epoch:
      w.run_epoch(tail)
      flush.zero_()
      w.epoch_end()
  w.launches = 0
  w.allreduce_ms = []
  w.energies = []
  clock = ClockSampler(clock_index) if clock_index is not None else None
  marks = []
  ends = []
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  torch.cuda.synchronize()
  wall0 = time.perf_counter()
  k = 0
  while k < steps:
    n = min(epoch_len, steps - k)
    if per_epoch and (n == epoch_len or (tail_epoch and n == tail)):
      m0, m1 = ev(), ev()
      m0.record()
      w.run_epoch(n)
      m1.record()
      marks.append((m0, m1))
      flush.zero_()                        # L2 flush, outside the event pairs
    else:
      for _ in range(n):
        m0, m1 = ev(), ev()
        m0.record()
        w.step()
        m1.record()
        marks.append((m0, m1))
        flush.zero_()
    k += n
    e0, e1 = ev(), ev()
    e0.record()
    w.epoch_end()
    e1.record()
    ends.append((e0, e1))
  torch.cuda.synchronize()
  wall = time.perf_counter() - wall0
  if world > 1:
    dist.barrier()
  clocks = clock.stop() if clock else None
  t_steps = sum(m[0].elapsed_time(m[1]) for m in marks) * 1e-3
  t_ends = sum(a.elapsed_time(b) for a, b in ends) * 1e-3
  t_ar = sum(a.elapsed_time(b) for a, b in w.allreduce_ms) * 1e-3
  out = dict(total_s=max_over_ranks(t_steps + t_ends, dev, world),
             steps_s=max_over_ranks(t_steps, dev, world),
             epoch_end_s=max_over_ranks(t_ends, dev, world),
             allreduce_s=max_over_ranks(t_ar, dev, world),
             n_epoch_ends=len(ends), epoch_len=epoch_len, wall_s=wall, clocks=clocks,
             launches=w.launches, energies=list(w.energies), per_epoch_launch=bool(per_epoch))
  return out


def roofline_for(w, t_step, n_act, pk):
  """Roofline of the dominant kernel(s) of one step of workload `w` from the
  ALGORITHMIC work of SURVEY.md 8(d) and the CUDA-event time of the step."""
  cfg, B, n = w.cfg, w.B, w.n
  steps = w.sweep_steps
  kind = cfg['hp']['wavefunction_type']
  f_hz = pk['sm_max_mhz'] * 1e6
  fp32_peak = 148 * 128 * 2 * f_hz / 1e12
  if kind == 'rbm':
    H = cfg['hp']['fc_layer_size']
    f_inc = 4 * H + 4
    f_fwd = 2 * n * H + 2 * n + 6 * H
    f_grad = 2 * 2 * (n + 1) * (H + 1)
    ratios = B * (n_act + steps)
    flop = B * (f_fwd + f_grad) + ratios * f_inc
    mufu = ratios * (H // 4 + 1) + B * 3 * H
    P = n * H + H + n + 1
    bytes_alg = B * ((n + 63) // 64) * 16 + B * 8 + 148 * 2 * P * 4
    smem_peak = 148 * 128 * f_hz / 1e12
    smem_alg = ratios * 2 * H * 4 + B * (n // 2) * H * 4
    return {
        'kernel': 'rbm2::walker_kernel<MC> (cgsvmc_batch_step(s): E_loc + gradient sums%s + sweep)' % (
            ' on tcgen05' if (n <= 39 and H < 160) else ''),
        'bound': 'shared-memory bandwidth (walker state and ratio tables are SM-resident; neither HBM nor the '
                 'tensor pipe bounds this kernel, SURVEY.md 8(d))' + (
                     '; at H=256 the 786 KB tables do not fit shared memory and are read through L1/L2'
                     if H > 160 else ''),
        'achieved': smem_alg / t_step / 1e12, 'peak': smem_peak, 'unit': 'TB/s',
        'frac': smem_alg / t_step / 1e12 / smem_peak, 'traffic': None,
        'peak_source': 'derived: 148 SM x 128 B/clk x sm_max_mhz (%s clock; 128 B/clk/SM confirmed by '
                       'profiles/microbench/fp32_pipes.cu)' % pk['source'],
        'what': 'algorithmic shared-memory bytes: 2 x H x 4 B per amplitude ratio + N/2 x H x 4 B per state build',
        'fp32': {'achieved': flop / t_step / 1e12, 'peak': fp32_peak, 'unit': 'TFLOP/s',
                 'frac': flop / t_step / 1e12 / fp32_peak,
                 'peak_source': 'derived: 148 SM x 128 FP32 lanes x 2 x sm_max_mhz'},
        'mufu': {'achieved': mufu / t_step / 1e12, 'peak': 148 * 16 * f_hz / 1e12, 'unit': 'Ttranscendental/s',
                 'frac': mufu / t_step / 1e12 / (148 * 16 * f_hz / 1e12)},
        'hbm': {'achieved': bytes_alg / t_step / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                'frac': bytes_alg / t_step / 1e9 / pk['hbm_gbs'], 'peak_source': pk['source']},
        'kernel_ms': t_step * 1e3, 'n_active_bonds_mean': n_act,
        'kernel_ms_is': 'CUDA-event time of the captured launch on the launching stream divided by the batch '
                        'iterations it runs (one persistent kernel per epoch for the headline; fused kernel + '
                        'reduction per step otherwise); ncu share of the kernel: profiles/ launch list'}
  f_fwd = cfg['f_fwd']
  if w.name == 'C4':        # sweep + two amplitude passes (trainee, target) + forward/backward gradient
    flop = B * (steps * f_fwd + 2 * f_fwd + 3 * f_fwd)
    what = 'B x (N sampler forwards + psi + psi_target + forward/backward gradient (3 F_fwd)) x F_fwd'
  else:
    f_inc = cfg.get('f_inc', f_fwd)
    flop = B * (steps * f_inc + f_fwd + n_act * f_inc + 4 * f_fwd)
    what = ('B x (N sampler ratios x F_inc + E_loc (F_fwd + n_active x F_inc) + gradient of two weight '
            'columns (4 F_fwd)); F_inc = F_fwd for conv (no incremental credit)')
  peak = pk['bf16_tflops_sustained']
  if kind == 'fully_connected':
    return {'kernel': 'fc_warp.cu warp-per-walker sampler (batches <= 2048) / fc_tc.cu tcgen05 sampler, fc_tc.cu tcgen05 '
                      'local energy, fc_tc_grad.cu tcgen05 gradient sums',
            'bound': 'tensor', 'achieved': flop / t_step / 1e12, 'peak': peak, 'unit': 'TFLOP/s',
            'frac': flop / t_step / 1e12 / peak, 'traffic': None,
            'peak_source': '%s bf16 cuBLAS, sustained' % pk['source'],
            'frac_of_split_peak': flop / t_step / 1e12 / (peak / 6.0),
            'split': 'float32-grade products from fp16 MMAs: 6 tensor-core products per algorithmic product '
                     '(three-way split of activations and weights), so the useful ceiling is peak / 6',
            'fp32': {'achieved': flop / t_step / 1e12, 'peak': fp32_peak, 'unit': 'TFLOP/s',
                     'frac': flop / t_step / 1e12 / fp32_peak,
                     'peak_source': 'derived: 148 SM x 128 FP32 lanes x 2 x sm_max_mhz'},
            'what': what, 'kernel_ms': t_step * 1e3, 'n_active_bonds_mean': n_act,
            'note': 'at 1024 walkers the step is latency-bound: the sweep runs on the warp-per-walker kernel '
                    '(fc_warp.cu, FP32 SIMT, 7 warps per SM; floor = one shared-memory weight read per warp), '
                    'local energy and gradient on tcgen05 tiles of 128 items; profiles/ holds the 65536-walker '
                    'numbers where the tensor path is 2.5-3.4x the SIMT path'}
  return {'kernel': 'conv_tc.cu tcgen05 kernels (sampler, local energy) + conv_tc_grad.cu tcgen05 gradient sums',
          'bound': 'tensor', 'achieved': flop / t_step / 1e12, 'peak': peak, 'unit': 'TFLOP/s',
          'frac': flop / t_step / 1e12 / peak, 'traffic': None,
          'peak_source': '%s bf16 cuBLAS, sustained' % pk['source'],
          'frac_of_split_peak': flop / t_step / 1e12 / (peak / 5.0),
          'split': 'float32-grade products from fp16 MMAs: 5 tensor-core products per algorithmic product '
                   '(two activation planes x three weight planes), so the useful ceiling is peak / 5; with 16 '
                   'filters an MMA has N <= 48 and the layer is bound by MMA issue / operand fetch, not the pipe',
          'what': what, 'kernel_ms': t_step * 1e3, 'n_active_bonds_mean': n_act}


def result_for(w, timing, steps, world, pk):
  B = w.B
  total = timing['total_s']
  t_step = timing['steps_s'] / steps
  n_act = w.n_active_bonds()
  res = {
      'workload': w.cfg['desc'], 'walkers_per_gpu': B, 'mc_steps_per_step': w.sweep_steps,
      'n_bonds': int(len(w.ij)) if hasattr(w, 'ij') else None, 'n_params': int(w.ansatz.num_params),
      'steps': steps, 'value': B * world * w.sweep_steps * steps / total, 'unit': 'walker-steps/s',
      'ms_per_step': total / steps * 1e3,
      'step_ms': t_step * 1e3, 'epoch_end_ms': timing['epoch_end_s'] / timing['n_epoch_ends'] * 1e3,
      'allreduce_ms': timing['allreduce_s'] / max(1, timing['n_epoch_ends']) * 1e3 if world > 1 else 0.0,
      'collectives_in_timed_region': timing['n_epoch_ends'] if world > 1 else 0,
      'epoch_len': timing['epoch_len'], 'gpu_launches': timing['launches'],
      'finite': bool(np.all(np.isfinite(timing['energies']))),
      'last_epoch_metric': timing['energies'][-1] if timing['energies'] else None,
      'roofline': roofline_for(w, t_step, n_act, pk),
  }
  if w.name != 'C4':
    res['eloc_evals_per_sec'] = B * world * steps / total
  else:
    res['collectives_in_timed_region'] = steps if world > 1 else 0   # the gradient all-reduce of every train step
    res['allreduce_ms'] = None
  return res


def dump_outputs(w, timing, out_dir):
  """Writes what an EnergyGradient run of workload `w` leaves its caller after
  the last timed step (an epoch end) to out_dir/<name>.npy:
    params          float32 [P]     parameters after the last Adam update
    energy_stats    float64 [4]     sum E, sum E^2, walkers of the last epoch, 0
    epoch_energies  float64 [E]     mean energy of every timed epoch
    accepted_moves  float64 [1]     accepted Metropolis moves of this shard so far
    configs         float32 [B, N]  walker configurations (+-1) of this shard
  Walker sets above DUMP_CONFIG_BYTES are written as a fixed, seeded sample of
  rows, and config_rows (float64) holds their indices."""
  torch.cuda.synchronize()
  configs = w.state.configs().cpu().numpy()
  arrays = {
      'params': w.ansatz.params.detach().cpu().numpy().astype(np.float32),
      'energy_stats': w.host_stats.numpy().astype(np.float64),
      'epoch_energies': np.asarray(timing['energies'], dtype=np.float64),
      'accepted_moves': w.state.accept_count.cpu().numpy().astype(np.float64),
  }
  if configs.nbytes > DUMP_CONFIG_BYTES:
    rows = np.sort(np.random.default_rng(SEED).choice(
        configs.shape[0], DUMP_CONFIG_BYTES // configs[0].nbytes, replace=False))
    configs = configs[rows]
    arrays['config_rows'] = rows.astype(np.float64)
  arrays['configs'] = configs.astype(np.float32)
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(a))


def parity_selfcheck(rank, world, dev):
  """N > 1: the all-reduced [sum O | sum E O | sum E, sum E^2, n | accepted
  moves] of `world` real shards equals the same quantities of `world` virtual
  shards run one after another on rank 0's GPU (walker ids r * B ...)."""
  import torch.distributed as dist
  from cgs_vmc_b200 import _native, engine, utils, wavefunctions
  cfg = CONFIGS['C2']
  hp = utils.create_hparams(batch_size=1024 * world, **cfg['hp'])
  wf = wavefunctions.build_wavefunction(hp).seed(1234)
  ansatz = wf.native(N_SITES)
  ij, jx, jz = bonds_for(cfg)
  ham = _native.Hamiltonian(ij, jx, jz, N_SITES, device=dev)
  B = 1024

  def shard(r):
    state = engine.WalkerState(B, N_SITES, seed=SEED, walker_id0=r * B, device=dev)
    sums = engine.EnergyGradientSums(ansatz, B, device=dev)
    state.mc_steps(ansatz, N_SITES)
    for _ in range(3):
      sums.batch_step(ham, state, SWEEP_STEPS)
    return torch.cat([sums.sums.reshape(-1).double(), sums.stats,
                      state.accept_count.double()])

  mine = shard(rank)
  dist.all_reduce(mine)
  if rank != 0:
    return None
  virtual = sum(shard(r) for r in range(world))
  P2 = 2 * ansatz.num_params
  scale = float(virtual[:P2].abs().max())
  err_sums = float((mine[:P2] - virtual[:P2]).abs().max()) / scale
  err_stats = float(((mine[P2:P2 + 2] - virtual[P2:P2 + 2]).abs() / virtual[P2:P2 + 2].abs()).max())
  exact = bool(mine[P2 + 2] == virtual[P2 + 2] and mine[-1] == virtual[-1])
  return {'parity_ok': bool(err_sums < 1e-6 and err_stats < 1e-12 and exact),
          'sums_max_rel_err': err_sums, 'energy_stats_max_rel_err': err_stats,
          'walkers_and_accepted_moves_exact': exact,
          'what': 'all-reduce over %d real shards vs %d virtual shards on rank 0 (1024 walkers each, 3 batch '
                  'steps): gradient sums (float32 per shard, summed in float64), sum E / sum E^2 (float64), '
                  'walker count and accepted moves (exact)' % (world, world)}


def run_ours(args, rank, world, local_rank):
  import torch.distributed as dist
  from cgs_vmc_b200 import _native, engine
  _native.require_cuda()
  torch.cuda.set_device(local_rank)
  dev = torch.device('cuda', local_rank)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
    warm = torch.zeros(1 << 16, dtype=torch.float64, device=dev)
    for _ in range(3):                     # communicator set-up outside every timed region
      dist.all_reduce(warm)
    torch.cuda.synchronize()
  pk = peaks()
  flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
  B = args.walkers

  # ---- headline: C2, device-resident inputs -------------------------------------
  w = EnergyGradientWorkload('C2', B, rank, world, dev)
  timing = time_workload(w, args.steps, args.warmup, flush, world, dev,
                         clock_index=local_rank if rank == 0 else None)
  if args.dump_outputs and rank == 0:     # before anything below steps the walkers again
    dump_outputs(w, timing, args.dump_outputs)
  main = result_for(w, timing, args.steps, world, pk)
  P = w.ansatz.num_params
  # the same epochs with one launch per batch iteration (cgsvmc_batch_step), for comparison
  per_step_launch = None
  if timing['per_epoch_launch']:
    tps = time_workload(w, args.steps, 3, flush, world, dev, force_per_step=True)
    per_step_launch = {
        'value': B * world * w.sweep_steps * args.steps / tps['total_s'], 'unit': 'walker-steps/s',
        'ms_per_step': tps['total_s'] / args.steps * 1e3, 'step_ms': tps['steps_s'] / args.steps * 1e3,
        'what': 'one captured graph (one cooperative kernel incl. the cross-CTA reduction) per batch '
                'iteration, L2 flushed between iterations'}

  # per-phase device times of the split launches (how the fused time divides), outside the timed region
  phase = [[ev() for _ in range(3)] for _ in range(20)]
  for k in range(20):
    phase[k][0].record()
    w.sums.accumulate(w.ham, w.state.packed)
    phase[k][1].record()
    w.state.mc_steps(w.ansatz, SWEEP_STEPS)
    phase[k][2].record()
    flush.zero_()
  torch.cuda.synchronize()
  w.sums.reset()
  t_acc = float(np.mean([m[0].elapsed_time(m[1]) for m in phase])) * 1e-3
  t_mc = float(np.mean([m[1].elapsed_time(m[2]) for m in phase])) * 1e-3

  # ---- e2e: the same epochs through host buffers -----------------------------------
  # engine.HostFedBatchStep: the float32 [B, N] configuration tensor of the
  # reference (graph_builders.py:92-125) comes from pinned host memory every
  # step (copy stream, double-buffered); pack + batch step + the device->host
  # copy of the energy statistics are one captured graph per slot; the epoch
  # end (all-reduce, gradient + Adam, mean energy to the host) runs every
  # min(50, steps) steps.  Every copy is inside the timed region.
  host_cfg = torch.empty(B, N_SITES, dtype=torch.float32).pin_memory()
  host_cfg.copy_(w.state.configs().cpu())
  fed = engine.HostFedBatchStep(w.state, w.ansatz, w.ham, w.sums, SWEEP_STEPS)
  epoch_len = timing['epoch_len']
  d2h = [0]

  def e2e_run(n, host_input):
    for k in range(n):
      fed.submit(host_input)
      d2h[0] += fed.d2h_bytes_stats
      if fed.outstanding() > 1:
        fed.result()                                              # host consumes the energy of step k - 1
      if (k + 1) % epoch_len == 0 or k + 1 == n:
        w.epoch_end()
        d2h[0] += 32
    while fed.outstanding():
      fed.result()

  def e2e_timed(host_input):
    e2e_run(max(4, min(epoch_len, 8)), host_input)
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    d2h[0] = 0
    e0, e1 = ev(), ev()
    e0.record()
    e2e_run(args.steps, host_input)
    e1.record()
    torch.cuda.synchronize()
    return max_over_ranks(e0.elapsed_time(e1) * 1e-3, dev, world), d2h[0] / args.steps

  e2e_s, d2h_per_step = e2e_timed(host_cfg)           # the engine's own choice ('auto') of the upload form
  e2e_h2d_bytes = fed.h2d_bytes
  auto_pack = fed.host_pack
  fed.host_pack = not auto_pack                         # and the other form, for comparison
  e2e_other_s, _ = e2e_timed(host_cfg)
  fed.host_pack = auto_pack
  host_packed = w.state.packed.cpu().pin_memory()
  e2e_packed_s, _ = e2e_timed(host_packed)

  # ---- the other BASELINE configurations ------------------------------------------
  subs = {}
  for name in [c.strip() for c in args.configs.split(',') if c.strip()]:
    if name == 'C2' or name not in CONFIGS:
      continue
    cfg = CONFIGS[name]
    k = max(1, min(args.steps, cfg['max_steps']))
    cls = SupervisedWorkload if name == 'C4' else EnergyGradientWorkload
    try:
      sw = cls(name, cfg['walkers'], rank, world, dev)
      st = time_workload(sw, k, 3, flush, world, dev)
      subs[name] = result_for(sw, st, k, world, pk)
    except Exception as exc:        # a failing sub-configuration must not cost the headline line
      subs[name] = {'workload': cfg['desc'], 'error': '%s: %s' % (type(exc).__name__, exc)}
    del sw
    torch.cuda.empty_cache()

  parity = parity_selfcheck(rank, world, dev) if world > 1 else None

  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return

  # ---- the JSON line -------------------------------------------------------------
  walkers_total = B * world
  total_s = timing['total_s']
  roofline = main['roofline']
  traffic_path = os.path.join(REPO, 'profiles', 'dram_traffic.json')
  if os.path.exists(traffic_path):          # dram__bytes_read + write of one ncu --set full capture
    tr = json.load(open(traffic_path))
    roofline['traffic'] = tr.get('bytes_per_launch')
    roofline['traffic_source'] = tr.get('source')
  line = {
      'metric': 'walker_steps_per_sec', 'value': main['value'], 'unit': 'walker-steps/s',
      'eloc_evals_per_sec': main['eloc_evals_per_sec'],
      'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
      'ms_per_step': main['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': config_dict(B),
      'config_detail': {
          'n_params': P,
          'l2': ('flushed: %d MiB memset between launches (= epochs), outside the CUDA-event pairs; within an epoch '
                 'the walkers and ratio tables are SM-resident by design (registers / shared memory)'
                 if timing['per_epoch_launch'] else
                 'flushed: %d MiB memset between steps, outside the per-step CUDA-event pairs') % (L2_FLUSH_BYTES >> 20),
          'launch': ('one captured CUDA graph per EPOCH holding cgsvmc_batch_steps = ONE persistent cooperative '
                     'kernel running all batch iterations of the epoch (estimators + sweep per iteration, walkers '
                     'resident in registers, tables loaded once, one deterministic cross-CTA reduction); the '
                     'parameter tables are rebuilt at the start of the epoch after every Adam update'
                     if timing['per_epoch_launch'] else
                     'one captured CUDA graph per step holding cgsvmc_batch_step = ONE cooperative kernel '
                     '(estimators + sweep + deterministic cross-CTA reduction); the parameter tables are '
                     'rebuilt in the first step after every Adam update'),
          'timed_region': 'whole epochs of %d steps: every step plus the epoch end (float64 all-reduce of '
                          '[2P+4], gradient + Adam kernel, mean energy to the host, reset)' % epoch_len,
          'parallelism': 'walkers sharded, params replicated' + (
              ', one all-reduce of [2P+4] doubles per epoch' if world > 1 else '')},
      'step_ms': main['step_ms'], 'epoch_end_ms': main['epoch_end_ms'], 'allreduce_ms': main['allreduce_ms'],
      'collectives_in_timed_region': main['collectives_in_timed_region'], 'epoch_len': epoch_len,
      'mean_energy_per_site_last_epoch': (main['last_epoch_metric'] or 0.0) / N_SITES,
      'kernel_ms': {'split launch: rbm2::walker_kernel (accumulate) + reduce': t_acc * 1e3,
                    'split launch: rbm2::mc_kernel (36 Metropolis steps)': t_mc * 1e3},
      'kernel_rates': {'sampler_walker_steps_per_sec': B * SWEEP_STEPS / t_mc,
                       'accumulate_eloc_evals_per_sec': B / t_acc},
      'per_step_launch': per_step_launch,
      'roofline': roofline,
      'e2e': {'value': walkers_total * SWEEP_STEPS * args.steps / e2e_s, 'unit': 'walker-steps/s',
              'eloc_evals_per_sec': walkers_total * args.steps / e2e_s,
              'ms_per_step': e2e_s / args.steps * 1e3,
              'h2d_bytes_per_step': e2e_h2d_bytes, 'd2h_bytes_per_step': d2h_per_step,
              'd2h': 'the energy statistics (32 B) after every step and the all-reduced statistics at every '
                     'epoch end; the gradient never leaves the device (the Adam update runs there)',
              'input': 'float32 [B, N] +-1 configurations (the reference layout) in pinned host memory, every '
                       'step; ' + ('bit-packed by the host cores (cgsvmc_pack_configs_host, inside the timed '
                                   'region) and uploaded as uint64 words' if auto_pack else
                                   'uploaded as float32 and bit-packed by the walker kernel'),
              'host_pack': bool(auto_pack),
              'host_pack_choice': 'engine.HostFedBatchStep(host_pack="auto"): packs on the host unless the measured '
                                  'packing time exceeds the measured float32 upload + 60 us',
              'host_pack_probe': fed.host_pack_probe, 'host_pack_threads': fed.pack_threads,
              'other_upload_form': {'host_pack': not auto_pack,
                                    'value': walkers_total * SWEEP_STEPS * args.steps / e2e_other_s,
                                    'ms_per_step': e2e_other_s / args.steps * 1e3},
              'walkers': 'the swept walkers stay on the device like the reference\'s session-owned variable '
                         '(graph_builders.py:92-125); they are not copied back to the host',
              'packed_host_input': {
                  'value': walkers_total * SWEEP_STEPS * args.steps / e2e_packed_s,
                  'ms_per_step': e2e_packed_s / args.steps * 1e3,
                  'h2d_bytes_per_step': int(host_packed.numel() * 8),
                  'what': 'same loop with the host holding the walkers bit-packed (uint64 [B, ceil(N/64)])'}},
      'gpu_launches': timing['launches'],
      'clocks': timing['clocks'],
      'wall_s_timed_region': timing['wall_s'],
      'configs': subs,
  }
  if parity is not None:
    line['parity_ok'] = parity['parity_ok']
    line['parity'] = parity
  if world == 1 and not args.no_cpu_baseline:
    c = cpu_arm('C2', B, 3, 1)
    line['cpu_baseline'] = {
        'value': c['walker_steps_per_sec'], 'unit': 'walker-steps/s',
        'eloc_evals_per_sec': c['eloc_evals_per_sec'], 'cores': c['cores'], 'kind': 'port',
        'ms_per_step': c['ms_per_step'],
        'sample': '3 full steps (after 1 warm-up) of the same workload at the full %d walkers: '
                  'reference-equivalent torch-CPU float32 op sequence (TF1 not installable)' % B}
    if 'C1' in subs and 'error' not in subs['C1']:
      c1 = cpu_arm('C1', CONFIGS['C1']['walkers'], 3, 1)
      subs['C1']['cpu_baseline'] = {
          'value': c1['walker_steps_per_sec'], 'unit': 'walker-steps/s', 'cores': c1['cores'], 'kind': 'port',
          'ms_per_step': c1['ms_per_step'], 'sample': '3 full steps (after 1 warm-up) at the full 1024 walkers'}
  print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def _claim_stdout():
  """Returns a file object on the real stdout and points fd 1 at stderr, so
  that library banners (NCCL prints its version on stdout) cannot get in front
  of the one JSON line the driver parses."""
  sys.stdout.flush()
  real = os.fdopen(os.dup(1), 'w')
  os.dup2(2, 1)
  return real


def main():
  global print
  out = _claim_stdout()
  _print = print
  print = lambda *a, **k: (_print(*a, **dict(k, file=out)), out.flush())
  args = parse_args()
  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  if args.impl == 'reference':
    run_reference(args, rank)
  else:
    run_ours(args, rank, world, local_rank)


if __name__ == '__main__':
  main()
