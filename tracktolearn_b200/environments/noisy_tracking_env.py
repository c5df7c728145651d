"""NoisyTrackingEnvironment (reference: environments/noisy_tracking_env.py:9-77).

Every ``ttl_track`` run uses this class, even with ``--noise 0`` (SURVEY.md F7): the float64
``rng.normal`` array added to the float32 actions makes the whole direction arithmetic
float64, which the step kernel reproduces with ``dir_f64 = 1``.

Where the noise comes from (``env_dto['noise_rng']``):
  * ``'host'`` (default, the reference's protocol): ``rng.normal(0, noise, (n_alive, 3))`` on the host
    every step, copied to the device; draw k goes to the streamline at alive-list position k.
  * ``'device'``: the step kernel draws it from a counter-based generator keyed by
    ``env_dto['noise_seed']`` (ttl_noise in include/ttl_b200.h): a streamline's noise at each step is a
    function of (seed, its index in the seed list, its point count) only, so the tractogram does not
    depend on ``n_actor``, refill, the slot order, CUDA-graph replay or the number of GPUs.
    No host work per step, and the fused actor head and graph replay stay available.
Neither is the reference's random stream: at noise > 0 no tractogram matches the reference's bit for bit.
"""
import numpy as np
import torch

from tracktolearn_b200 import _lib
from tracktolearn_b200.environments.tracking_env import TrackingEnvironment

NOISE_RNGS = ('host', 'device')


class NoisyTrackingEnvironment(TrackingEnvironment):

    def __init__(self, dataset_file, split_id, env_dto):
        self.noise = env_dto['noise']
        self.fa_map = None
        if env_dto.get('fa_map'):
            # The reference parses --fa_map but never reaches this branch (ttl_track.py:86 looks
            # for the wrong key, SURVEY.md F13); FA-scaled noise is dead code there and absent here.
            raise NotImplementedError('FA-scaled noise is dead code in the reference (F13)')
        self.noise_rng = env_dto.get('noise_rng', 'host')
        if self.noise_rng not in NOISE_RNGS:
            raise ValueError('noise_rng must be one of %s, not %r' % (NOISE_RNGS, self.noise_rng))
        self.noise_seed = env_dto.get('noise_seed')
        if self.noise_rng == 'device':
            if self.noise_seed is None:
                raise ValueError("noise_rng='device' needs env_dto['noise_seed'] (an int >= 0)")
            self.noise_seed = int(self.noise_seed)
            if not 0 <= self.noise_seed < 1 << 64:
                raise ValueError('noise_seed must be in [0, 2**64), not %d' % self.noise_seed)
        self.max_action = 1.
        self._float64_directions = True
        super().__init__(dataset_file, split_id, env_dto)

    def load_subject(self):
        super().load_subject()
        self._params.dir_f64 = 1

    # Device noise is keyed by g = row_base + batch row, with seed_offset / row_base kept by
    # TrackingEnvironment (reset, reset_streaming, nreset), which keys the stochastic policy the same way.

    def _device_noise(self):
        if self.noise_rng != 'device':
            return None
        return _lib.Noise(sigma=float(self.noise), seed=self.noise_seed, row_base=self._row_base)

    def _draw_noise(self, shape):
        """noisy_tracking_env.py:74: host RandomState draw, float64; None when sigma == 0
        (adding an all-zero float64 array only changes the dtype, which dir_f64 covers)."""
        if self.noise > 0. and self.noise_rng == 'host':
            noise = self.rng.normal(0., self.noise, size=shape)
            return torch.from_numpy(noise).to(self.device)
        return None

    def step(self, actions):
        """Reference: noisy_tracking_env.py:38-77."""
        actions = self._host_actions(actions)
        return self._step(actions, self._draw_noise((self._n_alive_host, 3)))

    def step_device(self, actions=None, noise=None, head=None, policy=None):
        if noise is None and head is None:
            noise = self._draw_noise((self._n_alive_host, 3))
        return super().step_device(actions, noise, head, policy)
