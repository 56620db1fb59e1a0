#!/usr/bin/env python
"""Energy evaluation driver: the reference's run_energy_evaluation.py
(lines 42-91) re-hosted on the B200 path."""
import os
import sys

import numpy as np
from absl import app
from absl import flags

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from cgs_vmc_b200 import checkpoint, drivers, evaluation, lattices, operators, utils, wavefunctions  # noqa: E402
from cgs_vmc_b200.session import Session  # noqa: E402

flags.DEFINE_float('heisenberg_jx', 1.0, 'Jx value in Heisenberg Hamiltonian.')
flags.DEFINE_string('checkpoint_dir', '', 'Full path to the checkpoint directory.')
flags.DEFINE_string('output_file', '', 'Optional file for the result.')
flags.DEFINE_string('hparams', '', 'Comma-separated name=value overrides.')
flags.DEFINE_string('correlations_file', '',
                    'Optional .npz for the spin-spin correlations <S_i . S_j> of all site pairs '
                    '(and the structure factor when the lattice geometry is known).')
flags.DEFINE_string('renyi_file', '',
                    'Optional .npz for the second Renyi entropy S2 of the prefix regions '
                    '(sites 0 .. l-1 for l = 1 .. N/2), by the replica-swap estimator.')
FLAGS = flags.FLAGS


def main(argv):
  del argv
  rank = drivers.init_distributed()
  hparams = utils.load_hparams(os.path.join(FLAGS.checkpoint_dir, 'hparams.pbtxt'))
  hparams.parse(FLAGS.hparams)
  bonds, j_x, j_z = drivers.load_bonds(FLAGS.checkpoint_dir, hparams.num_sites, FLAGS.heisenberg_jx)
  wavefunction = wavefunctions.build_wavefunction(hparams)
  hamiltonian = operators.HeisenbergHamiltonian(bonds, j_x, j_z)
  # before the energy run: a bond set without Marshall signs fails early
  signs = lattices.marshall_signs(hparams.num_sites, bonds, j_x, j_z) if FLAGS.correlations_file else None
  evaluator = evaluation.MonteCarloOperatorEvaluator()
  shared_resources = {}
  evaluation_ops = evaluator.build_eval_ops(
      wavefunction=wavefunction, operator=hamiltonian, hparams=hparams,
      shared_resources=shared_resources)
  session = Session()
  checkpoint.Saver(wavefunction).restore(
      session, checkpoint.latest_checkpoint(hparams.checkpoint_dir))
  data = evaluator.run_evaluation(evaluation_ops, session, hparams, epoch_num=0)
  mean_energy = np.mean(data)
  # the reference prints sqrt(std) / n (run_energy_evaluation.py:87, SURVEY.md
  # appendix B-11); the standard error of the mean is reported next to it
  reference_uncertainty = np.sqrt(np.std(data)) / len(data)
  stderr = np.std(data) / np.sqrt(len(data))
  if rank == 0:
    print('Energy: {} +/- {}'.format(mean_energy, reference_uncertainty))
    print('Standard error of the mean: {}'.format(stderr))
    if FLAGS.output_file:
      with open(FLAGS.output_file, 'w') as f:
        f.write('Energy mean: {}\nUncertainty: {}\nStderr: {}\n'.format(
            mean_energy, reference_uncertainty, stderr))
  if FLAGS.correlations_file:
    evaluate_correlations(evaluator, wavefunction, hparams, shared_resources, session, signs,
                          has_bond_file=os.path.exists(os.path.join(FLAGS.checkpoint_dir, 'J.txt')),
                          rank=rank)
  if FLAGS.renyi_file:
    evaluate_renyi(evaluator, wavefunction, hparams, shared_resources, session, rank=rank)


def evaluate_renyi(evaluator, wavefunction, hparams, shared_resources, session, rank):
  """S2 = -log Tr rho_A^2 of every prefix region from one more evaluation on
  the same walkers (replica swap of walker pairs).  The entropy and its error
  are NaN where the mean swap value is not positive."""
  regions = lattices.prefix_regions(hparams.num_sites)
  ops = evaluator.build_eval_ops(wavefunction=wavefunction, operator=operators.RenyiSwap(regions),
                                 hparams=hparams, shared_resources=shared_resources)
  samples = np.asarray(evaluator.run_evaluation(ops, session, hparams, epoch_num=0))
  if rank != 0:
    return
  mean = samples.mean(axis=0)
  stderr = samples.std(axis=0) / np.sqrt(len(samples))
  positive = mean > 0
  safe = np.where(positive, mean, 1.0)
  entropy = np.where(positive, -np.log(safe), np.nan)
  entropy_stderr = np.where(positive, stderr / safe, np.nan)
  with open(FLAGS.renyi_file, 'wb') as f:
    np.savez(f, regions=regions, swap_mean=mean, swap_stderr=stderr, entropy=entropy,
             entropy_stderr=entropy_stderr)


def evaluate_correlations(evaluator, wavefunction, hparams, shared_resources, session, signs, has_bond_file,
                          rank):
  """<S_i . S_j> of every site pair from a second evaluation on the same
  walkers, in the frame the Hamiltonian was written in (Marshall signs)."""
  n = hparams.num_sites
  pairs = np.asarray(lattices.all_pairs(n), dtype=np.int32)
  jx = (signs[pairs[:, 0]] * signs[pairs[:, 1]]).astype(np.float32)
  correlations = operators.HeisenbergBonds(pairs, jx, 1.0)
  ops = evaluator.build_eval_ops(wavefunction=wavefunction, operator=correlations, hparams=hparams,
                                 shared_resources=shared_resources)
  samples = np.asarray(evaluator.run_evaluation(ops, session, hparams, epoch_num=0))
  if rank != 0:
    return
  mean = samples.mean(axis=0)
  stderr = samples.std(axis=0) / np.sqrt(len(samples))
  matrix = np.full((n, n), 0.75)
  matrix[pairs[:, 0], pairs[:, 1]] = mean
  matrix[pairs[:, 1], pairs[:, 0]] = mean
  out = dict(pairs=pairs, signs=signs, mean=mean, stderr=stderr, matrix=matrix)
  # geometry: the default bonds are a periodic chain; a bond file is read as
  # the size_x x size_y square lattice when the sizes match, else S(q) is left out
  if not has_bond_file:
    out['structure_factor'] = lattices.structure_factor(matrix, n, 1)
  elif hparams.size_x * hparams.size_y == n:
    out['structure_factor'] = lattices.structure_factor(matrix, hparams.size_x, hparams.size_y)
  with open(FLAGS.correlations_file, 'wb') as f:
    np.savez(f, **out)


if __name__ == '__main__':
  app.run(main)
