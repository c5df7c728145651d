#!/usr/bin/env python3
"""ttl_track.py -- generate a tractogram from a trained agent (reference: runners/ttl_track.py).

Same positional arguments and options as the reference's console script.  Underneath: volumes
are uploaded once, every step of every streamline runs on the GPU (tracktolearn_b200), seeds are
tracked by a streaming tracker that keeps --n_actor streamlines alive, and the tractogram is
written from packed arrays."""
import argparse
import json
import os
import random
from argparse import RawTextHelpFormatter
from os.path import join

import numpy as np
import torch

from tracktolearn_b200.algorithms.sac_auto import SACAuto
from tracktolearn_b200.environments import NoisyTrackingEnvironment
from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import detect_format
from tracktolearn_b200.tracking.tracker import Tracker

_ROOT = os.sep.join(os.path.normpath(os.path.dirname(__file__)).split(os.sep)[:-2])
# The reference defaults to its bundled agent (<repo>/models, runners/ttl_track.py:34).  The weights
# are not part of this repository: point TTL_MODEL_DIR at a directory in the reference's layout
# (last_model_state_actor.pth, last_model_state_critic.pth, hyperparameters.json) to get the same default.
DEFAULT_MODEL = os.environ.get('TTL_MODEL_DIR', os.path.join(_ROOT, 'models'))


class TrackToLearnTrack(object):
    """Reference: runners/ttl_track.py:37-186."""

    def __init__(self, track_dto):
        self.in_odf = track_dto['in_odf']
        self.in_seed = track_dto['in_seed']
        self.in_mask = track_dto['in_mask']
        self.input_wm = track_dto['input_wm']
        self.reference_file = track_dto['in_mask']
        self.out_tractogram = track_dto['out_tractogram']
        self.noise = track_dto['noise']
        self.noise_rng = track_dto.get('noise_rng', 'host')
        self.policy_prob = float(track_dto.get('policy_prob') or 0.0)
        self.binary_stopping_threshold = track_dto['binary_stopping_threshold']
        self.n_actor = track_dto['n_actor']
        self.npv = track_dto['npv']
        self.min_length = track_dto['min_length']
        self.max_length = track_dto['max_length']
        self.compress = track_dto['compress'] or 0.0
        self.sh_basis = track_dto['sh_basis']
        self.save_seeds = track_dto['save_seeds']
        self.oracle_checkpoint = track_dto.get('oracle_checkpoint')
        self.oracle_threshold = float(track_dto.get('oracle_threshold', 0.5))
        self.oracle_precision = track_dto.get('oracle_precision', 'fp16')
        self.save_oracle_scores = bool(track_dto.get('save_oracle_scores', False))
        self.compute_reward = False
        if not torch.cuda.is_available():
            raise SystemExit('ttl_track (tracktolearn_b200) needs a CUDA device; there is no CPU path')
        # one process per GPU under torchrun: NCCL for the final tractogram gather only
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        if self.world > 1:
            import torch.distributed as dist
            local = int(os.environ.get('LOCAL_RANK', '0'))
            torch.cuda.set_device(local)
            if not dist.is_initialized():
                dist.init_process_group('nccl', device_id=torch.device('cuda', local))
            self.device = torch.device('cuda', local)
        else:
            self.device = torch.device('cuda')
        self.fa_map = None      # the reference looks up the wrong key here (SURVEY F13): never set
        self.agent = track_dto['agent']
        self.hyperparameters = track_dto['hyperparameters']
        self.precision = track_dto.get('precision', 'fp16')
        with open(self.hyperparameters, 'r') as json_file:
            hyperparams = json.load(json_file)
            self.algorithm = hyperparams['algorithm']
            self.step_size = float(hyperparams['step_size'])
            self.voxel_size = hyperparams.get('voxel_size', 2.0)
            self.theta = hyperparams['max_angle']
            self.hidden_dims = hyperparams['hidden_dims']
            self.n_dirs = hyperparams['n_dirs']
            self.target_sh_order = hyperparams['target_sh_order']
        self.random_seed = track_dto['rng_seed']
        torch.manual_seed(self.random_seed)
        np.random.seed(self.random_seed)
        random.seed(self.random_seed)
        self.rng = np.random.RandomState(seed=self.random_seed)

    def get_tracking_env(self, step_size_mm):
        """Reference: experiment/experiment.py:89-204 (the env DTO) + env.py:311-347."""
        env_dto = {
            'fa_map': self.fa_map, 'n_dirs': self.n_dirs, 'step_size': step_size_mm, 'theta': self.theta,
            'min_length': self.min_length, 'max_length': self.max_length, 'noise': self.noise,
            'npv': self.npv, 'rng': self.rng, 'alignment_weighting': 0.0, 'oracle_bonus': 0.0,
            'oracle_validator': False, 'oracle_stopping_criterion': False, 'oracle_checkpoint': None,
            'scoring_data': None, 'tractometer_validator': False,
            'binary_stopping_threshold': self.binary_stopping_threshold, 'compute_reward': False,
            'device': self.device, 'target_sh_order': int(self.target_sh_order),
            'in_odf': self.in_odf, 'in_seed': self.in_seed, 'in_mask': self.in_mask,
            'sh_basis': self.sh_basis, 'input_wm': self.input_wm, 'reference': self.reference_file,
            'state_of_stopped': False, 'noise_rng': self.noise_rng, 'noise_seed': self.random_seed,
        }
        return NoisyTrackingEnvironment.from_files(env_dto)

    def run(self):
        ref_img = nifti.load(self.reference_file)
        tracking_voxel_size = ref_img.zooms[0]
        step_size_mm = self.step_size
        if abs(float(tracking_voxel_size) - float(self.voxel_size)) >= 0.1:
            step_size_mm = (float(tracking_voxel_size) / float(self.voxel_size)) * self.step_size
            print("Agent was trained on a voxel size of {}mm and a "
                  "step size of {}mm.".format(self.voxel_size, self.step_size))
            print("Subject has a voxel size of {}mm, setting step size to "
                  "{}mm.".format(tracking_voxel_size, step_size_mm))
        env = self.get_tracking_env(step_size_mm)
        self.input_size = env.get_state_size()
        self.action_size = env.get_action_size()
        algs = {'SACAuto': SACAuto}
        print('Tracking with {} agent.'.format(self.algorithm))
        alg = algs[self.algorithm](self.input_size, self.action_size, self.hidden_dims, n_actors=self.n_actor,
                                   rng=self.rng, device=self.device, precision=self.precision)
        alg.agent.load(self.agent, 'last_model_state')
        # --policy_prob > 0: the agent's stochastic policy, its draws keyed by --rng_seed (ttl_policy)
        tracker = Tracker(alg, self.n_actor, prob=self.policy_prob, compress=self.compress,
                          min_length=self.min_length, max_length=self.max_length, save_seeds=self.save_seeds,
                          policy_seed=self.random_seed if self.policy_prob > 0 else None)
        oracle = None
        if self.oracle_checkpoint:
            from tracktolearn_b200.oracles.oracle import OracleSingleton
            OracleSingleton.clear()
            oracle = OracleSingleton(self.oracle_checkpoint, self.device, precision=self.oracle_precision)
        n = tracker.track_to_file(env, self.out_tractogram, ref_img.shape[:3], ref_img.zooms[:3], oracle=oracle,
                                  oracle_threshold=self.oracle_threshold, save_scores=self.save_oracle_scores)
        if int(os.environ.get('RANK', '0')) == 0:
            print('Wrote {} streamlines to {}.'.format(n, self.out_tractogram))
        return n


def add_mandatory_options_tracking(p):
    p.add_argument('in_odf', help='File containing the orientation diffusion function \n'
                   'as spherical harmonics file (.nii.gz). Ex: ODF or fODF.\nCan be of any order and basis '
                   '(including "full" bases for\nasymmetric ODFs). See also --sh_basis.')
    p.add_argument('in_seed', help='Seeding mask (.nii.gz). Must be represent the WM/GM interface.')
    p.add_argument('in_mask', help='Tracking mask (.nii.gz).\nTracking will stop outside this mask.')
    p.add_argument('out_tractogram', help='Tractogram output file (must be .trk or .tck).')
    p.add_argument('--input_wm', action='store_true',
                   help='If set, append the WM mask to the input signal. The agent must have been trained '
                        'accordingly.')


def add_out_options(p):
    out_g = p.add_argument_group('Output options')
    out_g.add_argument('--compress', type=float, metavar='thresh',
                       help='If set, will compress streamlines. The parameter value is the \ndistance '
                            'threshold. [%(default)s]')
    out_g.add_argument('-f', dest='overwrite', action='store_true',
                       help='Force overwriting of the output files.')
    out_g.add_argument('--save_seeds', action='store_true',
                       help='If set, save the seeds used for the tracking \n in the data_per_streamline '
                            'property.')
    return out_g


def add_track_args(parser):
    add_mandatory_options_tracking(parser)
    basis_group = parser.add_argument_group('Basis options')
    basis_group.add_argument('--sh_basis', default='descoteaux07', choices=['descoteaux07', 'tournier07'],
                             help='Spherical harmonics basis used for the SH coefficients. [%(default)s]')
    add_out_options(parser)
    agent_group = parser.add_argument_group('Tracking agent options')
    agent_group.add_argument('--agent', type=str,
                             help='Path to the folder containing .pth files.\nIf not set, will default to '
                                  'the example models.\n[{}]'.format(DEFAULT_MODEL))
    agent_group.add_argument('--hyperparameters', type=str,
                             help='Path to the .json file containing the hyperparameters of your tracking '
                                  'agent. \nIf not set, will default to the example models.\n[{}]'.format(
                                      DEFAULT_MODEL))
    agent_group.add_argument('--n_actor', type=int, default=10000, metavar='N',
                             help='Number of streamlines to track simultaneously.\n[%(default)s]')
    agent_group.add_argument('--precision', default='fp16', choices=['fp16', 'tf32', 'bf16', 'fp32'],
                             help='Actor arithmetic.  fp16 / tf32: tcgen05 tensor cores, outputs within 1e-3 of the '
                                  'fp32 reference (fp16 at full rate within +-65504 -- tracking aborts with a '
                                  'message if a value saturates; tf32 at half rate with fp32 range); bf16: tensor '
                                  'cores, ~4e-3; fp32: CUDA cores, the reference arithmetic. [%(default)s]')
    seed_group = parser.add_argument_group('Seeding options')
    seed_group.add_argument('--npv', type=int, default=1, help='Number of seeds per voxel [%(default)s].')
    track_g = parser.add_argument_group('Tracking options')
    track_g.add_argument('--min_length', type=float, default=10., metavar='m',
                         help='Minimum length of a streamline in mm. [%(default)s]')
    track_g.add_argument('--max_length', type=float, default=300., metavar='M',
                         help='Maximum length of a streamline in mm. [%(default)s]')
    track_g.add_argument('--noise', default=0.0, type=float, metavar='sigma',
                         help='Add noise ~ N (0, `noise`) to the agent\'s\noutput to make tracking more '
                              'probabilistic.\nShould be between 0.0 and 0.1.[%(default)s]')
    track_g.add_argument('--noise_rng', default='host', choices=['host', 'device'],
                         help='Where the `--noise` draws come from.\nhost: the reference\'s numpy RandomState '
                              'stream, drawn on the CPU every step;\nthe tractogram then depends on --n_actor and '
                              'on the number of GPUs.\ndevice: drawn inside the GPU step from --rng_seed, the seed\'s '
                              'index and the step;\nthe tractogram is the same for every --n_actor and GPU count, and '
                              'no host work is added per step.\nNeither reproduces the reference\'s random '
                              'stream. [%(default)s]')
    track_g.add_argument('--policy_prob', default=0.0, type=float, metavar='P',
                         help='Sample the agent\'s stochastic policy, its std scaled by P:\n'
                              'a = tanh(mu + P * std * eps).  0 tracks with the mean action.\n'
                              'eps is drawn on the GPU from --rng_seed, the seed\'s index and the step, so the\n'
                              'tractogram is the same for every --n_actor and GPU count. [%(default)s]')
    track_g.add_argument('--fa_map', type=str, default=None,
                         help='Scale the added noise (see `--noise`) according\nto the provided FA map '
                              '(.nii.gz). Optional.')
    track_g.add_argument('--binary_stopping_threshold', type=float, default=0.1,
                         help='Lower limit for interpolation of tracking mask value.\nTracking will stop '
                              'below this threshold.')
    parser.add_argument('--rng_seed', default=1337, type=int, help='Random number generator seed [%(default)s].')
    oracle_g = parser.add_argument_group('Oracle filtering')
    oracle_g.add_argument('--oracle_checkpoint', type=str, default=None, metavar='CKPT',
                          help='TractOracle-Net checkpoint.  If set, every streamline that passes the length\n'
                               'filter is scored on the GPU and kept only when its score is\n'
                               '>= --oracle_threshold.  Scores are taken before --compress.')
    oracle_g.add_argument('--oracle_threshold', type=float, default=0.5, metavar='T',
                          help='Keep streamlines whose oracle score is >= T, in [0, 1]. [%(default)s]')
    oracle_g.add_argument('--oracle_precision', default='fp16', choices=['fp16', 'fp32'],
                          help='Oracle arithmetic.  fp16: tcgen05 tensor cores, the reference\'s autocast\n'
                               'arithmetic; fp32: CUDA cores. [%(default)s]')
    oracle_g.add_argument('--save_oracle_scores', action='store_true',
                          help='Save each kept streamline\'s score as the per-streamline\nproperty '
                               '"oracle_score" (.trk only).')


def verify_agent_option(parser, args):
    if (args.agent is not None and args.hyperparameters is None) or \
       (args.agent is None and args.hyperparameters is not None):
        parser.error('You must specify both --agent and --hyperparameters arguments or use the default model.')
    if args.agent is None:
        if not os.path.exists(join(DEFAULT_MODEL, 'last_model_state_actor.pth')):
            parser.error('no agent given and no default agent at %s (the reference\'s bundled weights are not '
                         'shipped here): pass --agent and --hyperparameters, or set TTL_MODEL_DIR' % DEFAULT_MODEL)
        args.agent = DEFAULT_MODEL
        args.hyperparameters = join(DEFAULT_MODEL, 'hyperparameters.json')


def parse_args(argv=None):
    """ Generate a tractogram from a trained model. """
    parser = argparse.ArgumentParser(description=parse_args.__doc__, formatter_class=RawTextHelpFormatter)
    add_track_args(parser)
    args = parser.parse_args(argv)
    if not 0 <= args.policy_prob < float('inf'):
        parser.error('--policy_prob must be a finite number >= 0, not %r' % args.policy_prob)
    for f in (args.in_odf, args.in_seed, args.in_mask):
        if not os.path.isfile(f):
            parser.error('Input file {} does not exist'.format(f))
    if os.path.isfile(args.out_tractogram) and not args.overwrite:
        parser.error('Output file {} exists. Use -f to force overwriting'.format(args.out_tractogram))
    try:
        detect_format(args.out_tractogram)
    except ValueError as e:
        parser.error(str(e))
    if args.min_length < 0 or args.max_length < args.min_length:
        parser.error('Invalid streamline length options')
    if args.compress is not None and args.compress < 0.001:
        parser.error('--compress should be at least 0.001')
    if not 0.0 <= args.oracle_threshold <= 1.0:
        parser.error('--oracle_threshold must be in [0, 1], not %r' % args.oracle_threshold)
    if args.save_oracle_scores and not args.oracle_checkpoint:
        parser.error('--save_oracle_scores needs --oracle_checkpoint')
    if args.save_oracle_scores and detect_format(args.out_tractogram) != 'trk':
        parser.error('--save_oracle_scores needs a .trk output: .tck files cannot hold per-streamline data')
    if args.oracle_checkpoint and not os.path.isfile(args.oracle_checkpoint):
        parser.error('Oracle checkpoint {} does not exist'.format(args.oracle_checkpoint))
    verify_agent_option(parser, args)
    return args


def main(argv=None):
    """ Main tracking script """
    args = parse_args(argv)
    try:
        TrackToLearnTrack(vars(args)).run()
    finally:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and int(os.environ.get('WORLD_SIZE', '1')) > 1:
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
