"""ctypes binding of libcgsvmc.so (include/cgsvmc.h) for torch CUDA tensors.

torch is used for device memory and streams only; the signatures that cross
the boundary are plain pointers and sizes.
"""
import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# CGSVMC_LIBRARY selects another build of the same library (the phase-timing
# development build of profiles/run_rbm2_phases.py); never a different backend.
LIB_PATH = os.environ.get('CGSVMC_LIBRARY') or os.path.join(_HERE, 'libcgsvmc.so')

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED = 0, -1, -2, -3
ANSATZ_KINDS = {'fully_connected': 1, 'rbm': 2, 'conv_1d': 3, 'conv_2d': 4,
                'res_net_1d': 5, 'res_net_2d': 6}
ACTIVATIONS = {'relu': 0, 'tanh': 1, 'sigmoid': 2, 'identity': 3, 'cos': 4,
               'exp': 5, 'tan': 6, 'selu': 7}

EXPORTS = [
    'cgsvmc_version', 'cgsvmc_last_error', 'cgsvmc_ansatz_create',
    'cgsvmc_ansatz_destroy', 'cgsvmc_ansatz_num_params',
    'cgsvmc_ansatz_bind_params', 'cgsvmc_ansatz_track_params',
    'cgsvmc_ansatz_params_changed', 'cgsvmc_ham_create', 'cgsvmc_ham_destroy',
    'cgsvmc_pack_configs', 'cgsvmc_unpack_configs', 'cgsvmc_random_configs',
    'cgsvmc_log_amp', 'cgsvmc_mc_steps', 'cgsvmc_mc_steps_graph', 'cgsvmc_mc_step_replay',
    'cgsvmc_flip_enum', 'cgsvmc_local_energy', 'cgsvmc_weighted_grad_sum',
    'cgsvmc_energy_stats', 'cgsvmc_accumulate', 'cgsvmc_batch_step',
    'cgsvmc_propose_exchange', 'cgsvmc_accept_exchange', 'cgsvmc_local_energy_from_amps',
    'cgsvmc_swo_weights', 'cgsvmc_adam_step', 'cgsvmc_batch_step_fed', 'cgsvmc_batch_steps',
    'cgsvmc_epoch_end', 'cgsvmc_pack_configs_host', 'cgsvmc_upload_configs',
    'cgsvmc_conv_periodic', 'cgsvmc_log_amp_jvp',
]


class AnsatzDesc(ctypes.Structure):
  _fields_ = [(n, ctypes.c_int32) for n in (
      'kind', 'n_sites', 'num_layers', 'layer_size', 'num_filters',
      'kernel_size', 'size_x', 'size_y', 'nonlinearity')]


class NativeError(RuntimeError):
  pass


_lib = None


def load():
  """Loads the shared library (once).  Raises if it has not been built."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise NativeError(
        'libcgsvmc.so is missing (%s): run `python __graft_entry__.py` to '
        'build the CUDA library; there is no CPU fallback.' % LIB_PATH)
  lib = ctypes.CDLL(LIB_PATH)
  vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64
  lib.cgsvmc_version.restype = ctypes.c_int
  lib.cgsvmc_last_error.restype = ctypes.c_char_p
  lib.cgsvmc_ansatz_create.argtypes = [ctypes.POINTER(AnsatzDesc), ctypes.POINTER(vp)]
  lib.cgsvmc_ansatz_destroy.argtypes = [vp]
  lib.cgsvmc_ansatz_num_params.argtypes = [vp]
  lib.cgsvmc_ansatz_num_params.restype = i64
  lib.cgsvmc_ansatz_bind_params.argtypes = [vp, vp]
  lib.cgsvmc_ansatz_track_params.argtypes = [vp, ctypes.c_int]
  lib.cgsvmc_ansatz_params_changed.argtypes = [vp]
  lib.cgsvmc_ham_create.argtypes = [vp, vp, vp, i32, i32, ctypes.POINTER(vp)]
  lib.cgsvmc_ham_destroy.argtypes = [vp]
  lib.cgsvmc_pack_configs.argtypes = [vp, i64, i32, vp, vp]
  lib.cgsvmc_unpack_configs.argtypes = [vp, i64, i32, vp, vp]
  lib.cgsvmc_random_configs.argtypes = [vp, i64, i32, u64, u64, vp]
  lib.cgsvmc_log_amp.argtypes = [vp, vp, i64, vp, vp]
  lib.cgsvmc_mc_steps.argtypes = [vp, vp, i64, i32, u64, u64, u64, vp, vp, vp]
  lib.cgsvmc_mc_steps_graph.argtypes = [vp, vp, i64, i32, u64, u64, vp, vp, vp, vp]
  lib.cgsvmc_mc_step_replay.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp]
  lib.cgsvmc_flip_enum.argtypes = [vp, vp, i64, vp, vp, vp]
  lib.cgsvmc_local_energy.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, vp]
  lib.cgsvmc_weighted_grad_sum.argtypes = [vp, vp, vp, i64, i32, vp, vp]
  lib.cgsvmc_log_amp_jvp.argtypes = [vp, vp, i64, vp, vp, vp]
  lib.cgsvmc_energy_stats.argtypes = [vp, i64, vp, vp]
  lib.cgsvmc_accumulate.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, vp]
  lib.cgsvmc_batch_step.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, i32, u64, u64, u64, vp, vp, vp]
  lib.cgsvmc_propose_exchange.argtypes = [vp, i64, i32, u64, u64, u64, vp, vp, vp]
  lib.cgsvmc_accept_exchange.argtypes = [vp, vp, i64, i32, vp, vp, vp, vp, vp, vp, vp]
  lib.cgsvmc_local_energy_from_amps.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp]
  f32 = ctypes.c_float
  lib.cgsvmc_batch_steps.argtypes = [vp, vp, vp, i64, i32, vp, vp, vp, vp, i32, u64, u64, u64, vp, vp, vp]
  lib.cgsvmc_batch_step_fed.argtypes = [vp, vp, vp, vp, i64, vp, vp, vp, vp, i32, u64, u64, u64, vp, vp, vp, vp]
  lib.cgsvmc_swo_weights.argtypes = [vp, vp, vp, vp, i64, f32, f32, vp, vp, vp]
  lib.cgsvmc_adam_step.argtypes = [vp, vp, vp, i64, vp, vp, vp, f32, f32, vp, f32, f32, f32, u64, vp, vp]
  lib.cgsvmc_pack_configs_host.argtypes = [vp, i64, i32, vp, i32]
  lib.cgsvmc_upload_configs.argtypes = [vp, i64, i32, vp, vp, i32, vp]
  lib.cgsvmc_conv_periodic.argtypes = [vp, i64, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp]
  lib.cgsvmc_epoch_end.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp, vp, f32, f32, f32, f32, f32, u64, vp, vp, vp]
  for name in EXPORTS:
    fn = getattr(lib, name)
    if name not in ('cgsvmc_last_error', 'cgsvmc_ansatz_num_params'):
      fn.restype = ctypes.c_int
  _lib = lib
  return lib


def check(rc):
  """Maps a status code to the exception the reference raises for the same
  condition (ValueError for shape / registry errors)."""
  if rc == OK:
    return
  msg = load().cgsvmc_last_error().decode('utf-8', 'replace')
  if rc == ERR_INVALID:
    raise ValueError(msg)
  if rc == ERR_UNSUPPORTED:
    raise NotImplementedError(msg)
  raise NativeError('cgsvmc error %d: %s' % (rc, msg))


def require_cuda():
  if not torch.cuda.is_available():
    raise NativeError('no CUDA device: cgs_vmc_b200 has no CPU fallback')


def _ptr(t):
  return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
  return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def n_words(n_sites):
  return (n_sites + 63) // 64


def _want(t, dtype, shape=None, name='tensor'):
  if not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
    raise ValueError('%s must be a contiguous CUDA tensor of dtype %s' % (name, dtype))
  if shape is not None and tuple(t.shape) != tuple(shape):
    raise ValueError('%s has shape %s, expected %s' % (name, tuple(t.shape), tuple(shape)))


class Ansatz:
  """Owns a cgsvmc_ansatz handle and the flat float32 parameter buffer."""

  def __init__(self, kind, n_sites, num_layers=0, layer_size=0, num_filters=0,
               kernel_size=0, size_x=1, size_y=1, nonlinearity='relu',
               device='cuda'):
    require_cuda()
    lib = load()
    if kind not in ANSATZ_KINDS:
      raise ValueError('Provided wavefunction_type is not registered.')
    if nonlinearity not in ACTIVATIONS:
      raise ValueError('unknown nonlinearity %r' % (nonlinearity,))
    self.kind, self.n_sites = kind, n_sites
    self.device = torch.device(device)
    desc = AnsatzDesc(ANSATZ_KINDS[kind], n_sites, num_layers, layer_size,
                      num_filters, kernel_size, size_x, size_y,
                      ACTIVATIONS[nonlinearity])
    self.desc = desc
    handle = ctypes.c_void_p()
    with torch.cuda.device(self.device):
      check(lib.cgsvmc_ansatz_create(ctypes.byref(desc), ctypes.byref(handle)))
    self._handle = handle
    self.num_params = int(lib.cgsvmc_ansatz_num_params(handle))
    self.params = torch.zeros(self.num_params, dtype=torch.float32, device=self.device)
    check(lib.cgsvmc_ansatz_bind_params(handle, _ptr(self.params)))
    # derived tables are rebuilt only when torch reports an in-place change of
    # the parameter buffer (its version counter covers views as well)
    check(lib.cgsvmc_ansatz_track_params(handle, 1))
    self._seen_version = None

  def set_params(self, flat):
    """Copies a flat parameter vector (layout of include/cgsvmc.h) in place."""
    flat = torch.as_tensor(flat, dtype=torch.float32).reshape(-1)
    if flat.numel() != self.num_params:
      raise ValueError('expected %d parameters, got %d' % (self.num_params, flat.numel()))
    self.params.copy_(flat.to(self.device))

  def close(self):
    if getattr(self, '_handle', None) is not None and _lib is not None:
      _lib.cgsvmc_ansatz_destroy(self._handle)
      self._handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:   # interpreter shutdown
      pass

  def _sync_params(self):
    v = self.params._version
    if v != self._seen_version:
      check(load().cgsvmc_ansatz_params_changed(self._handle))
      self._seen_version = v

  # ---- compute entry points -------------------------------------------
  def log_amp(self, packed, out=None):
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    if out is None:
      out = torch.empty(b, dtype=torch.float32, device=packed.device)
    check(load().cgsvmc_log_amp(self._handle, _ptr(packed), b, _ptr(out), _stream()))
    return out

  def mc_steps(self, packed, n_steps, seed, walker_id0=0, step0=0,
               accept_count=None, log_amp_out=None):
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    if accept_count is not None:
      _want(accept_count, torch.int64, (1,), 'accept_count')
    if log_amp_out is not None:
      _want(log_amp_out, torch.float32, (b,), 'log_amp_out')
    check(load().cgsvmc_mc_steps(self._handle, _ptr(packed), b, int(n_steps),
                                 int(seed), int(walker_id0), int(step0),
                                 _ptr(accept_count), _ptr(log_amp_out), _stream()))

  def mc_steps_graph(self, packed, n_steps, seed, walker_id0, step_counter,
                     accept_count=None, log_amp_out=None):
    """mc_steps with the Philox step offset in device memory (int64 [1] tensor,
    advanced by n_steps on the stream): safe to capture in a CUDA graph."""
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    _want(step_counter, torch.int64, (1,), 'step_counter')
    if accept_count is not None:
      _want(accept_count, torch.int64, (1,), 'accept_count')
    check(load().cgsvmc_mc_steps_graph(self._handle, _ptr(packed), b, int(n_steps), int(seed),
                                       int(walker_id0), _ptr(step_counter), _ptr(accept_count),
                                       _ptr(log_amp_out), _stream()))

  def mc_step_replay(self, packed, u_sites, u_acc):
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    _want(u_sites, torch.float32, (b, self.n_sites), 'u_sites')
    _want(u_acc, torch.float32, (b,), 'u_acc')
    dev = packed.device
    down = torch.empty(b, dtype=torch.int32, device=dev)
    up = torch.empty(b, dtype=torch.int32, device=dev)
    log_ratio = torch.empty(b, dtype=torch.float32, device=dev)
    accept = torch.empty(b, dtype=torch.uint8, device=dev)
    check(load().cgsvmc_mc_step_replay(self._handle, _ptr(packed), b, _ptr(u_sites),
                                       _ptr(u_acc), _ptr(down), _ptr(up),
                                       _ptr(log_ratio), _ptr(accept), _stream()))
    return down, up, log_ratio, accept

  def local_energy(self, ham, packed, want_parts=False):
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    dev = packed.device
    e = torch.empty(b, dtype=torch.float32, device=dev)
    z = torch.empty(b, dtype=torch.float32, device=dev)
    diag = torch.empty(b, dtype=torch.float32, device=dev) if want_parts else None
    off = torch.empty(b, dtype=torch.float32, device=dev) if want_parts else None
    check(load().cgsvmc_local_energy(self._handle, ham._handle, _ptr(packed), b,
                                     _ptr(e), _ptr(z), _ptr(diag), _ptr(off), _stream()))
    return (e, z, diag, off) if want_parts else (e, z)

  def weighted_grad_sum(self, packed, weights, out=None):
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    if weights.dim() == 1:
      weights = weights.reshape(1, -1)
    k = weights.shape[0]
    _want(weights, torch.float32, (k, b), 'weights')
    if out is None:
      out = torch.zeros(k, self.num_params, dtype=torch.float32, device=packed.device)
    else:
      _want(out, torch.float32, (k, self.num_params), 'out')
    check(load().cgsvmc_weighted_grad_sum(self._handle, _ptr(packed), _ptr(weights),
                                          b, k, _ptr(out), _stream()))
    return out

  def log_amp_jvp(self, packed, tangent, out=None):
    """out[b] = sum_p d z_b / d params_p * tangent[p] (float32 [B]) for a
    tangent in the flat parameter layout: the forward counterpart of
    weighted_grad_sum (cgsvmc_log_amp_jvp; pure RBM only, NotImplementedError
    otherwise)."""
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    _want(tangent, torch.float32, (self.num_params,), 'tangent')
    if out is None:
      out = torch.empty(b, dtype=torch.float32, device=packed.device)
    else:
      _want(out, torch.float32, (b,), 'out')
    check(load().cgsvmc_log_amp_jvp(self._handle, _ptr(packed), b, _ptr(tangent), _ptr(out), _stream()))
    return out

  def accumulate(self, ham, packed, sums, stats, e_loc_out=None, log_amp_out=None):
    """One session.run(accumulate_gradients) (training.py:539-558): sums [2, P]
    += (sum_b O_b, sum_b E_b O_b), stats float64[4] += (sum E, sum E^2, B, 0)."""
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    _want(sums, torch.float32, (2, self.num_params), 'sums')
    _want(stats, torch.float64, (4,), 'stats')
    if e_loc_out is not None:
      _want(e_loc_out, torch.float32, (b,), 'e_loc_out')
    if log_amp_out is not None:
      _want(log_amp_out, torch.float32, (b,), 'log_amp_out')
    check(load().cgsvmc_accumulate(self._handle, ham._handle, _ptr(packed), b,
                                   _ptr(e_loc_out), _ptr(log_amp_out), _ptr(sums),
                                   _ptr(stats), _stream()))

  def batch_step(self, ham, packed, sums, stats, n_steps, seed, walker_id0=0, step0=0,
                 step_counter=None, accept_count=None, e_loc_out=None, log_amp_out=None):
    """accumulate() on the current configurations followed by n_steps
    Metropolis steps (one batch iteration of run_optimization_epoch,
    training.py:614-617); one kernel for the pure RBM.  With `step_counter`
    (int64 [1] device tensor) the Philox offset is read from and advanced on
    the device (CUDA-graph safe)."""
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    _want(sums, torch.float32, (2, self.num_params), 'sums')
    _want(stats, torch.float64, (4,), 'stats')
    if step_counter is not None:
      _want(step_counter, torch.int64, (1,), 'step_counter')
    if accept_count is not None:
      _want(accept_count, torch.int64, (1,), 'accept_count')
    if e_loc_out is not None:
      _want(e_loc_out, torch.float32, (b,), 'e_loc_out')
    if log_amp_out is not None:
      _want(log_amp_out, torch.float32, (b,), 'log_amp_out')
    check(load().cgsvmc_batch_step(self._handle, ham._handle, _ptr(packed), b, _ptr(e_loc_out),
                                   _ptr(log_amp_out), _ptr(sums), _ptr(stats), int(n_steps),
                                   int(seed), int(walker_id0), int(step0), _ptr(step_counter),
                                   _ptr(accept_count), _stream()))


  def batch_steps(self, ham, packed, n_batches, sums, stats, n_steps, seed, walker_id0=0, step0=0,
                  step_counter=None, accept_count=None, e_loc_out=None, log_amp_out=None):
    """n_batches consecutive batch iterations (the inner loop of
    run_optimization_epoch, training.py:614-617) in one call
    (cgsvmc_batch_steps): one persistent kernel for the pure RBM.  e_loc_out /
    log_amp_out: float32 [n_batches, B]."""
    self._sync_params()
    b = packed.shape[0]
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    _want(sums, torch.float32, (2, self.num_params), 'sums')
    _want(stats, torch.float64, (4,), 'stats')
    if step_counter is not None:
      _want(step_counter, torch.int64, (1,), 'step_counter')
    if accept_count is not None:
      _want(accept_count, torch.int64, (1,), 'accept_count')
    if e_loc_out is not None:
      _want(e_loc_out, torch.float32, (int(n_batches), b), 'e_loc_out')
    if log_amp_out is not None:
      _want(log_amp_out, torch.float32, (int(n_batches), b), 'log_amp_out')
    check(load().cgsvmc_batch_steps(self._handle, ham._handle, _ptr(packed), b, int(n_batches),
                                    _ptr(e_loc_out), _ptr(log_amp_out), _ptr(sums), _ptr(stats),
                                    int(n_steps), int(seed), int(walker_id0), int(step0),
                                    _ptr(step_counter), _ptr(accept_count), _stream()))

  def batch_step_fed(self, ham, configs_f32, packed_out, sums, stats, n_steps, seed, walker_id0,
                     step_counter, accept_count=None, e_loc_out=None, stats_out=None):
    """batch_step for a host-fed caller (cgsvmc_batch_step_fed): `configs_f32`
    (device float32 [B, N] of +-1, or None to step `packed_out` in place) is
    packed inside the walker kernel, `stats_out` (float64 [4]; a pinned host
    tensor is written directly from the device) receives the updated energy
    statistics.  CUDA-graph safe (device-side step counter)."""
    self._sync_params()
    b = packed_out.shape[0]
    _want(packed_out, torch.int64, (b, n_words(self.n_sites)), 'packed_out')
    if configs_f32 is not None:
      _want(configs_f32, torch.float32, (b, self.n_sites), 'configs_f32')
    _want(sums, torch.float32, (2, self.num_params), 'sums')
    _want(stats, torch.float64, (4,), 'stats')
    _want(step_counter, torch.int64, (1,), 'step_counter')
    if accept_count is not None:
      _want(accept_count, torch.int64, (1,), 'accept_count')
    if e_loc_out is not None:
      _want(e_loc_out, torch.float32, (b,), 'e_loc_out')
    if stats_out is not None:
      if stats_out.dtype != torch.float64 or stats_out.numel() != 4 or not stats_out.is_contiguous() or not (
          stats_out.is_cuda or stats_out.is_pinned()):
        raise ValueError('stats_out must be a contiguous float64 [4] tensor on the device or in pinned host memory')
    check(load().cgsvmc_batch_step_fed(self._handle, ham._handle, _ptr(configs_f32), _ptr(packed_out), b,
                                       _ptr(e_loc_out), None, _ptr(sums), _ptr(stats), int(n_steps),
                                       int(seed), int(walker_id0), 0, _ptr(step_counter),
                                       _ptr(accept_count), _ptr(stats_out), _stream()))


class Hamiltonian:
  """Owns a cgsvmc_ham handle (bond table on the device)."""

  def __init__(self, bonds_ij, jx, jz, n_sites, device='cuda'):
    require_cuda()
    lib = load()
    ij = np.ascontiguousarray(np.asarray(bonds_ij, dtype=np.int32).reshape(-1, 2))
    n_bonds = ij.shape[0]
    jx = np.ascontiguousarray(np.broadcast_to(np.asarray(jx, dtype=np.float32), (n_bonds,)))
    jz = np.ascontiguousarray(np.broadcast_to(np.asarray(jz, dtype=np.float32), (n_bonds,)))
    self.n_bonds, self.n_sites = n_bonds, n_sites
    self.bonds_ij, self.jx, self.jz = ij, jx, jz
    handle = ctypes.c_void_p()
    with torch.cuda.device(torch.device(device)):
      check(lib.cgsvmc_ham_create(ij.ctypes.data_as(ctypes.c_void_p),
                                  jx.ctypes.data_as(ctypes.c_void_p),
                                  jz.ctypes.data_as(ctypes.c_void_p),
                                  n_bonds, n_sites, ctypes.byref(handle)))
    self._handle = handle

  def close(self):
    if getattr(self, '_handle', None) is not None and _lib is not None:
      _lib.cgsvmc_ham_destroy(self._handle)
      self._handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  def flip_enum(self, packed, want_flipped=True):
    b, w = packed.shape
    _want(packed, torch.int64, (b, n_words(self.n_sites)), 'packed')
    dev = packed.device
    mask = torch.empty(b, (self.n_bonds + 31) // 32, dtype=torch.int32, device=dev)
    flipped = torch.empty(b, self.n_bonds, w, dtype=torch.int64, device=dev) \
        if want_flipped else None
    check(load().cgsvmc_flip_enum(self._handle, _ptr(packed), b, _ptr(flipped),
                                  _ptr(mask), _stream()))
    return mask, flipped


def pack_configs(configs, out=None):
  """float32 [B, N] of +-1 (CUDA) -> int64-viewed uint64 [B, W]."""
  require_cuda()
  b, n = configs.shape
  _want(configs, torch.float32, (b, n), 'configs')
  if out is None:
    packed = torch.empty(b, n_words(n), dtype=torch.int64, device=configs.device)
  else:
    _want(out, torch.int64, (b, n_words(n)), 'out')
    packed = out
  check(load().cgsvmc_pack_configs(_ptr(configs), b, n, _ptr(packed), _stream()))
  return packed


def pack_configs_host(configs, out, n_threads=0):
  """float32 [B, N] of +-1 in HOST memory -> int64-viewed uint64 [B, W] in host
  memory (normally a pinned staging buffer), on the host cores
  (cgsvmc_pack_configs_host)."""
  b, n = configs.shape
  if configs.is_cuda or configs.dtype != torch.float32 or not configs.is_contiguous():
    raise ValueError('configs must be a contiguous float32 host tensor')
  if out.is_cuda or out.dtype != torch.int64 or not out.is_contiguous() or tuple(out.shape) != (b, n_words(n)):
    raise ValueError('out must be a contiguous int64 host tensor of shape [B, ceil(N / 64)]')
  check(load().cgsvmc_pack_configs_host(_ptr(configs), b, n, _ptr(out), int(n_threads)))
  return out


def upload_configs(configs, dst, stream, staging=None, n_threads=0):
  """One float32 [B, N] host batch to the device on `stream` (a
  torch.cuda.Stream), as float32 into `dst` [B, N] or -- with a pinned
  `staging` buffer -- bit-packed on the host cores first, into `dst` [B, W]
  (cgsvmc_upload_configs).  No shape checks beyond the library's: the caller
  (engine.HostFedBatchStep) owns the buffers."""
  b, n = configs.shape
  check(load().cgsvmc_upload_configs(_ptr(configs), b, n, _ptr(staging), _ptr(dst), int(n_threads),
                                     ctypes.c_void_p(stream.cuda_stream)))


def conv_periodic(inputs, weights, bias=None):
  """layers.Conv1dPeriodic / Conv2dPeriodic (layers.py:24-160) on the device:
  inputs float32 [B, L, C_in] with weights [k, C_in, C_out], or [B, X, Y, C_in]
  with weights [k, k, C_in, C_out]; returns [B, ..., C_out]
  (cgsvmc_conv_periodic)."""
  require_cuda()
  rank = inputs.dim() - 2
  if rank not in (1, 2) or weights.dim() != rank + 2:
    raise ValueError('conv_periodic: inputs [B, L, C] / [B, X, Y, C] and weights [k, (k,) C_in, C_out] expected')
  k, c_in, c_out = weights.shape[0], weights.shape[-2], weights.shape[-1]
  if rank == 2 and weights.shape[1] != k:
    raise ValueError('conv_periodic: square kernels only')
  if inputs.shape[-1] != c_in:
    raise ValueError('conv_periodic: input channels do not match the weights')
  _want(inputs, torch.float32, None, 'inputs')
  _want(weights, torch.float32, None, 'weights')
  if bias is not None:
    _want(bias, torch.float32, (c_out,), 'bias')
  b, x = inputs.shape[0], inputs.shape[1]
  y = inputs.shape[2] if rank == 2 else 1
  out = torch.empty(tuple(inputs.shape[:-1]) + (c_out,), dtype=torch.float32, device=inputs.device)
  check(load().cgsvmc_conv_periodic(_ptr(inputs), b, x, y, c_in, c_out, k, rank, _ptr(weights), _ptr(bias),
                                    _ptr(out), _stream()))
  return out


def unpack_configs(packed, n_sites, out=None):
  require_cuda()
  b = packed.shape[0]
  _want(packed, torch.int64, (b, n_words(n_sites)), 'packed')
  if out is None:
    out = torch.empty(b, n_sites, dtype=torch.float32, device=packed.device)
  check(load().cgsvmc_unpack_configs(_ptr(packed), b, n_sites, _ptr(out), _stream()))
  return out


def random_configs(batch_size, n_sites, seed, walker_id0=0, device='cuda'):
  require_cuda()
  packed = torch.empty(batch_size, n_words(n_sites), dtype=torch.int64, device=device)
  check(load().cgsvmc_random_configs(_ptr(packed), batch_size, n_sites, int(seed),
                                     int(walker_id0), _stream()))
  return packed


def energy_stats(e_loc, stats=None):
  require_cuda()
  _want(e_loc, torch.float32, None, 'e_loc')
  if stats is None:
    stats = torch.zeros(4, dtype=torch.float64, device=e_loc.device)
  check(load().cgsvmc_energy_stats(_ptr(e_loc), e_loc.numel(), _ptr(stats), _stream()))
  return stats


def propose_exchange(packed, n_sites, seed, walker_id0, step):
  """One exchange proposal per walker (graph_builders.py:59-73) with the Philox
  convention of the fused samplers.  Returns (proposed packed, u_acc)."""
  require_cuda()
  b = packed.shape[0]
  _want(packed, torch.int64, (b, n_words(n_sites)), 'packed')
  proposed = torch.empty_like(packed)
  u_acc = torch.empty(b, dtype=torch.float32, device=packed.device)
  check(load().cgsvmc_propose_exchange(_ptr(packed), b, n_sites, int(seed), int(walker_id0), int(step),
                                       _ptr(proposed), _ptr(u_acc), _stream()))
  return proposed, u_acc


def accept_exchange(packed, proposed, n_sites, logabs, sign, logabs_new, sign_new, u_acc,
                    accept_count=None):
  """Metropolis accept / reject in the log domain (graph_builders.py:74-89);
  updates packed, logabs and sign in place."""
  b = packed.shape[0]
  _want(packed, torch.int64, (b, n_words(n_sites)), 'packed')
  _want(proposed, torch.int64, (b, n_words(n_sites)), 'proposed')
  for name, t in (('logabs', logabs), ('logabs_new', logabs_new), ('u_acc', u_acc)):
    _want(t, torch.float32, (b,), name)
  if sign is not None:
    _want(sign, torch.float32, (b,), 'sign')
    _want(sign_new, torch.float32, (b,), 'sign_new')
  if accept_count is not None:
    _want(accept_count, torch.int64, (1,), 'accept_count')
  check(load().cgsvmc_accept_exchange(_ptr(packed), _ptr(proposed), b, n_sites, _ptr(logabs), _ptr(sign),
                                      _ptr(logabs_new), _ptr(sign_new), _ptr(u_acc),
                                      _ptr(accept_count), _stream()))


def local_energy_from_amps(ham, packed, logabs, sign, flipped_logabs, flipped_sign, want_parts=False):
  """E_loc from externally evaluated amplitudes (operators.py:165-169, 241-259)."""
  b = packed.shape[0]
  _want(packed, torch.int64, (b, n_words(ham.n_sites)), 'packed')
  _want(logabs, torch.float32, (b,), 'logabs')
  _want(flipped_logabs, torch.float32, (b, ham.n_bonds), 'flipped_logabs')
  if sign is not None:
    _want(sign, torch.float32, (b,), 'sign')
  if flipped_sign is not None:
    _want(flipped_sign, torch.float32, (b, ham.n_bonds), 'flipped_sign')
  dev = packed.device
  e = torch.empty(b, dtype=torch.float32, device=dev)
  diag = torch.empty(b, dtype=torch.float32, device=dev) if want_parts else None
  off = torch.empty(b, dtype=torch.float32, device=dev) if want_parts else None
  check(load().cgsvmc_local_energy_from_amps(ham._handle, _ptr(packed), b, _ptr(logabs), _ptr(sign),
                                             _ptr(flipped_logabs), _ptr(flipped_sign), _ptr(e),
                                             _ptr(diag), _ptr(off), _stream()))
  return (e, diag, off) if want_parts else e



def swo_weights(log_amp, log_amp_target, log_norm, total, sign=None, sign_target=None, out=None,
                loss_acc=None):
  """Loss and gradient weights of SupervisedWavefunctionOptimizer
  (training.py:166-175) in one kernel: returns weights [1, B] = 2 (1 - r) / total
  with r = psi_target sqrt(2^N) / psi; loss_acc (float64 [2]) += (sum (1 - r)^2, B)."""
  b = log_amp.numel()
  for name, t in (('log_amp', log_amp), ('log_amp_target', log_amp_target)):
    _want(t, torch.float32, (b,), name)
  for name, t in (('sign', sign), ('sign_target', sign_target)):
    if t is not None:
      _want(t, torch.float32, (b,), name)
  if out is None:
    out = torch.empty(1, b, dtype=torch.float32, device=log_amp.device)
  _want(out, torch.float32, (1, b), 'out')
  if loss_acc is not None:
    _want(loss_acc, torch.float64, (2,), 'loss_acc')
  check(load().cgsvmc_swo_weights(_ptr(log_amp), _ptr(sign), _ptr(log_amp_target), _ptr(sign_target), b,
                                  float(log_norm), 1.0 / float(total), _ptr(out), _ptr(loss_acc),
                                  _stream()))
  return out


def epoch_end(params, m, v, local_sums, local_stats, ticket, total_sums=None, total_stats=None,
              total_payload=None, num_batches=1.0, lr=0.0, beta1=0.9, beta2=0.99, eps=1e-8, t=1,
              stats_out=None):
  """apply_gradients + metrics + reset_gradients of an EnergyGradientOptimizer
  epoch (training.py:618-622) in one kernel (cgsvmc_epoch_end): the Adam step on
  the energy gradient of the totals, the totals' statistics stored to
  `stats_out` (a pinned host tensor is written directly), the local
  accumulators zeroed.  Totals: (total_sums, total_stats), defaulting to the
  local accumulators, or the all-reduced float64 `total_payload` [2 P + 4]."""
  n = params.numel()
  for name, x in (('params', params), ('m', m), ('v', v)):
    _want(x, torch.float32, (n,), name)
  _want(local_sums, torch.float32, (2, n), 'local_sums')
  _want(local_stats, torch.float64, (4,), 'local_stats')
  _want(ticket, torch.int32, (1,), 'ticket')
  if total_payload is not None:
    _want(total_payload, torch.float64, (2 * n + 4,), 'total_payload')
    total_sums = total_stats = None
  else:
    total_sums = local_sums if total_sums is None else total_sums
    total_stats = local_stats if total_stats is None else total_stats
    _want(total_sums, torch.float32, (2, n), 'total_sums')
    _want(total_stats, torch.float64, (4,), 'total_stats')
  out_ptr = None
  if stats_out is not None:
    if stats_out.dtype != torch.float64 or stats_out.numel() != 4 or not stats_out.is_contiguous() or not (
        stats_out.is_cuda or stats_out.is_pinned()):
      raise ValueError('stats_out must be a contiguous float64 [4] tensor on the device or in pinned host memory')
    out_ptr = _ptr(stats_out)
  check(load().cgsvmc_epoch_end(_ptr(params), _ptr(m), _ptr(v), n, _ptr(total_sums), _ptr(total_payload),
                                _ptr(total_stats), _ptr(local_sums), _ptr(local_stats),
                                1.0 / float(num_batches), float(lr), float(beta1), float(beta2), float(eps),
                                int(t), out_ptr, _ptr(ticket), _stream()))
  torch.autograd.graph.increment_version(params)


def adam_step(params, m, v, grad=None, sums=None, stats=None, num_batches=1.0, lr=0.0, lr_dev=None,
              beta1=0.9, beta2=0.99, eps=1e-8, t=1, t_dev=None):
  """One tf.train.AdamOptimizer update of the flat parameter buffer in one
  kernel; the gradient is `grad` or the energy gradient of training.py:562-564
  formed from (sums [2, P], stats [4])."""
  n = params.numel()
  for name, x in (('params', params), ('m', m), ('v', v)):
    _want(x, torch.float32, (n,), name)
  if grad is not None:
    _want(grad, torch.float32, (n,), 'grad')
  if sums is not None:
    _want(sums, torch.float32, (2, n), 'sums')
    _want(stats, torch.float64, (4,), 'stats')
  if lr_dev is not None:
    _want(lr_dev, torch.float32, (1,), 'lr_dev')
  if t_dev is not None:
    _want(t_dev, torch.int64, (1,), 't_dev')
  check(load().cgsvmc_adam_step(_ptr(params), _ptr(m), _ptr(v), n, _ptr(grad), _ptr(sums), _ptr(stats),
                                1.0 / float(num_batches), float(lr), _ptr(lr_dev), float(beta1),
                                float(beta2), float(eps), int(t), _ptr(t_dev), _stream()))
  # the kernel wrote through the raw pointer: tell torch, so that the ansatz
  # handles notice the parameter change (Ansatz._sync_params)
  torch.autograd.graph.increment_version(params)
