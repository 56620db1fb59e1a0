"""Hyper-parameters and initial walker state (mirror of the reference's
utils.py).  `tf.contrib.training.HParams` does not exist here; `HParams` is a
small stand-in with the methods the drivers call (utils.py:87-166,
run_training.py:83-101)."""
import ast
import json

from . import _native


class HParams:
  def __init__(self, **kwargs):
    self._names = []
    for k, v in kwargs.items():
      self.add_hparam(k, v)

  def add_hparam(self, name, value):
    if name in self._names:
      raise ValueError('Hyperparameter name is reserved: %s' % name)
    self._names.append(name)
    setattr(self, name, value)

  def set_hparam(self, name, value):
    if name not in self._names:
      raise KeyError('Unknown hyperparameter: %s' % name)
    old = getattr(self, name)
    if isinstance(old, bool):
      value = value if isinstance(value, bool) else str(value).lower() in ('1', 'true')
    elif isinstance(old, int) and not isinstance(value, bool):
      value = int(value)
    elif isinstance(old, float):
      value = float(value)
    elif isinstance(old, (list, tuple)):
      # tf HParams keeps the list type of the default: a scalar override of a
      # list-valued hyper-parameter is an error there, as is a wrong length for
      # the fixed-size pairs (composite_wavefunction_types, ...)
      if not isinstance(value, (list, tuple)):
        raise ValueError('Must pass a list for multi-valued parameter: %s' % name)
      if isinstance(old, tuple) and len(value) != len(old):
        raise ValueError('Hyperparameter %s takes %d values, got %d' % (name, len(old), len(value)))
      value = type(old)(value)
    setattr(self, name, value)

  def override_from_dict(self, values):
    for k, v in values.items():
      self.set_hparam(k, v)
    return self

  def parse(self, text):
    """'a=1,b=relu,c=[1,2]' overrides (run_training.py:90)."""
    text = (text or '').strip()
    if not text:
      return self
    depth, start, items = 0, 0, []
    for pos, ch in enumerate(text):
      depth += ch in '[(' 
      depth -= ch in '])'
      if ch == ',' and depth == 0:
        items.append(text[start:pos]); start = pos + 1
    items.append(text[start:])
    for item in items:
      name, _, raw = item.partition('=')
      name, raw = name.strip(), raw.strip()
      self.set_hparam(name, self._parse_value(raw))
    return self

  @staticmethod
  def _parse_value(raw):
    """A number, a bare string, or a bracketed list of either
    (tf.contrib.training.HParams.parse takes `x=[rbm,fully_connected]` with
    unquoted strings)."""
    try:
      return ast.literal_eval(raw)
    except (ValueError, SyntaxError):
      pass
    if len(raw) >= 2 and raw[0] in '[(' and raw[-1] in '])':
      inner = raw[1:-1].strip()
      return [HParams._parse_value(item.strip()) for item in inner.split(',')] if inner else []
    return raw

  def values(self):
    return {k: getattr(self, k) for k in self._names}

  def to_json(self):
    return json.dumps(self.values(), indent=1, sort_keys=True)

  def __contains__(self, name):
    return name in self._names

  def __copy__(self):
    return HParams(**self.values())


def create_hparams(**kwargs):
  """Defaults of the reference, utils.py:87-150."""
  hparams = HParams(
      checkpoint_dir='', supervisor_dir='', basis_file_path='',
      wavefunction_type='', composite_wavefunction_types=('', ''),
      wavefunction_optimizer_type='',
      num_sites=40, size_x=1, size_y=1, size_z=1,
      num_fc_layers=3, fc_layer_size=80,
      num_conv_layers=5, conv_strides=1, kernel_size=5, num_conv_filters=16,
      num_resnet_blocks=2, bond_dimension=4,
      top_lin_table_file='', bot_lin_table_file='', ed_vector_file='',
      adjacency_list_path='',
      nonlinearity='relu', output_activation='exp',
      composite_output_activations=('', ''),
      num_equilibration_sweeps=100, num_monte_carlo_sweeps=1,
      num_epochs=500, batch_size=200, num_batches_per_epoch=50,
      time_evolution_beta=0.12,
      learning_rates=[1e-3, 1e-4, 2e-5, 1e-5], learning_rate_stops=[300, 600, 1000],
      optimizer='adam', beta2=0.99,
      num_evaluation_samples=100,
      # StochasticReconfiguration (not in the reference): shift on the identity,
      # conjugate-gradient iteration cap and relative residual target
      sr_diag_shift=0.01, sr_cg_max_iterations=100, sr_cg_tolerance=1e-4,
  )
  hparams.override_from_dict(kwargs)
  return hparams


def save_hparams(hparams, path):
  """The reference writes a text proto (run_training.py:100-101); TensorFlow's
  proto is unavailable, the same name=value content is written as JSON."""
  with open(path, 'w') as f:
    f.write(hparams.to_json())


def load_hparams(path):
  """utils.load_hparams (utils.py:153-166) for files written by save_hparams."""
  with open(path) as f:
    values = json.load(f)
  hparams = create_hparams()
  for k, v in values.items():
    if isinstance(getattr(hparams, k, None), tuple):
      v = tuple(v)
    if k in hparams:
      setattr(hparams, k, v)
    else:
      hparams.add_hparam(k, v)
  return hparams


def random_configurations(n_sites, batch_size=1, seed=0, walker_id0=0, device='cuda'):
  """utils.random_configurations (utils.py:169-192): float32 [B, N] of +-1
  with n_sites // 2 spins down, generated on the device."""
  packed = _native.random_configs(batch_size, n_sites, seed, walker_id0, device=device)
  return _native.unpack_configs(packed, n_sites)
