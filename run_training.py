#!/usr/bin/env python
"""Ground-state optimisation driver: the reference's run_training.py
(run_training.py:73-160) re-hosted on the B200 path.  Same flags."""
import os
import sys

from absl import app
from absl import flags

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from cgs_vmc_b200 import checkpoint, drivers, operators, training, utils, wavefunctions  # noqa: E402
from cgs_vmc_b200.session import Session  # noqa: E402

flags.DEFINE_string('checkpoint_dir', '', 'Full path to the checkpoint directory.')
flags.DEFINE_integer('num_sites', 24, 'Number of sites in the system.')
flags.DEFINE_float('heisenberg_jx', 1.0, 'Jx value in Heisenberg Hamiltonian.')
flags.DEFINE_integer('num_epochs', 1000, 'Total of number of epochs to train on.')
flags.DEFINE_integer('checkpoint_frequency', 1, 'Number of epochs between checkpoints.')
flags.DEFINE_boolean('resume_training', False, 'Restore variables from the latest checkpoint.')
flags.DEFINE_string('wavefunction_type', '', 'Key of wavefunctions.WAVEFUNCTION_TYPES.')
flags.DEFINE_string('optimizer', 'EnergyGradient',
                    'Key of training.GROUND_STATE_OPTIMIZERS (the reference default ITSWO '
                    'crashes at graph build, training.py:812) or of '
                    'training.EXTRA_GROUND_STATE_OPTIMIZERS (StochasticReconfiguration).')
flags.DEFINE_boolean('generate_vectors', False, 'Not available on this path.')
flags.DEFINE_string('basis_file_path', '', 'Path to the basis file (unused).')
flags.DEFINE_string('hparams', '', 'Comma-separated name=value overrides.')
flags.DEFINE_boolean('override', True, 'Whether to override an existing hparams file.')
FLAGS = flags.FLAGS


def main(argv):
  del argv
  rank = drivers.init_distributed()
  hparams = utils.create_hparams()
  hparams.set_hparam('checkpoint_dir', FLAGS.checkpoint_dir)
  hparams.set_hparam('basis_file_path', FLAGS.basis_file_path)
  hparams.set_hparam('num_sites', FLAGS.num_sites)
  hparams.set_hparam('num_epochs', FLAGS.num_epochs)
  hparams.set_hparam('wavefunction_type', FLAGS.wavefunction_type)
  hparams.set_hparam('wavefunction_optimizer_type', FLAGS.optimizer)
  hparams.parse(FLAGS.hparams)
  hparams_path = os.path.join(hparams.checkpoint_dir, 'hparams.pbtxt')
  if rank == 0:
    os.makedirs(FLAGS.checkpoint_dir, exist_ok=True)
    if os.path.exists(hparams_path) and not FLAGS.override:
      print('Hparams file already exists')
      sys.exit()
    utils.save_hparams(hparams, hparams_path)

  bonds, j_x, j_z = drivers.load_bonds(FLAGS.checkpoint_dir, hparams.num_sites, FLAGS.heisenberg_jx)
  wavefunction = wavefunctions.build_wavefunction(hparams)
  hamiltonian = operators.HeisenbergHamiltonian(bonds, j_x, j_z)
  wavefunction_optimizer = training.ground_state_optimizer(FLAGS.optimizer)()
  shared_resources = {}
  train_ops = wavefunction_optimizer.build_opt_ops(
      wavefunction=wavefunction, hamiltonian=hamiltonian, hparams=hparams,
      shared_resources=shared_resources)

  session = Session()
  checkpoint_saver = checkpoint.Saver(wavefunction, max_to_keep=5)
  if FLAGS.resume_training:
    checkpoint_saver.restore(session, checkpoint.latest_checkpoint(hparams.checkpoint_dir))

  metrics_path = os.path.join(hparams.checkpoint_dir, 'metrics.txt')
  for epoch_number in range(FLAGS.num_epochs):
    if rank == 0:
      name = 'model_prior_{}_epochs'.format(epoch_number)
      checkpoint_saver.save(session, os.path.join(hparams.checkpoint_dir, name))
    metrics_record = wavefunction_optimizer.run_optimization_epoch(train_ops, session, hparams)
    if rank == 0:
      with open(metrics_path, 'a') as f:
        f.write('{}\n'.format(metrics_record))
  if FLAGS.generate_vectors:
    raise NotImplementedError('VectorWavefunctionEvaluator is outside the hot path')


if __name__ == '__main__':
  app.run(main)
