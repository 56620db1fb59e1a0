"""Mirror of the reference's evaluation.py: MonteCarloOperatorEvaluator
(evaluation.py:74-152).  VectorWavefunctionEvaluator is a file-dump utility
outside the hot path."""
import collections

import torch

from . import distributed, graph_builders, operators
from .session import Op

EvalOps = collections.namedtuple('EvaluationOps', [
    'value', 'mc_step', 'acceptance_rate', 'placeholder_input', 'wavefunction_value'])


class WavefunctionEvaluator:
  def build_eval_ops(self, wavefunction, operator, hparams, shared_resources):
    raise NotImplementedError

  def run_evaluation(self, eval_ops, session, hparams, epoch_num):
    raise NotImplementedError


class MonteCarloOperatorEvaluator(WavefunctionEvaluator):
  """Operator evaluation by MCMC."""

  def build_eval_ops(self, wavefunction, operator, hparams, shared_resources):
    """evaluation.py:77-110: value = mean of the local values.  An operator
    with a vector local value [B, K] (operators.HeisenbergBonds) gives the
    float64 numpy vector [K] of the per-column means; operators.RenyiSwap
    gives the means over walker pairs [R] (each rank pairs its own shard)."""
    n_sites = hparams.num_sites
    local_batch, walker_id0 = distributed.shard(hparams.batch_size)
    configs = graph_builders.get_configs(shared_resources, local_batch, n_sites,
                                         walker_id0=walker_id0)
    mc_step, acc_rate = graph_builders.get_monte_carlo_sampling(
        shared_resources, configs, wavefunction)

    def value():
      e = operator.local_value(wavefunction, configs)
      if isinstance(operator, operators.RenyiSwap):
        payload = torch.cat([e.double().sum(dim=0), e.new_full((1,), e.shape[0], dtype=torch.float64)])
        totals = distributed.allreduce_(payload).cpu().numpy()
        return totals[:-1] / totals[-1]
      if e.dim() == 2:
        totals = distributed.allreduce_(e.double().sum(dim=0))
        return totals.cpu().numpy() / hparams.batch_size
      total = distributed.allreduce_(e.double().sum())
      return float(total.item()) / hparams.batch_size

    return EvalOps(value=Op(value, 'mean_local_value'), mc_step=mc_step,
                   acceptance_rate=acc_rate, placeholder_input=None, wavefunction_value=None)

  def run_evaluation(self, eval_ops, session, hparams, epoch_num):
    """evaluation.py:113-152."""
    del epoch_num
    num_mc_steps = hparams.num_monte_carlo_sweeps * hparams.num_sites
    session.run(eval_ops.mc_step,
                n_steps=hparams.num_equilibration_sweeps * hparams.num_sites)
    values = []
    for _ in range(hparams.num_evaluation_samples):
      values.append(session.run(eval_ops.value))
      session.run(eval_ops.mc_step, n_steps=num_mc_steps)
    return values


class VectorWavefunctionEvaluator(WavefunctionEvaluator):
  def build_eval_ops(self, *args, **kwargs):
    raise NotImplementedError('VectorWavefunctionEvaluator dumps amplitudes on a basis file '
                              '(evaluation.py:155-246): outside the hot path')
