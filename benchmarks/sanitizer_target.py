#!/usr/bin/env python
"""Small end-to-end run for compute-sanitizer (scripts/sanitize.sh): reset + 20 steps of the reference
protocol (fp32 state rows, host actions), a streaming device-mode episode in every tensor-core tier (fused
multi-layer actor launch with its inter-layer flags, stop bookkeeping across the two env kernels, slot
refill), TractOracle-Net scoring, and the tractogram pack.  Sizes are tiny: the sanitizer slows kernels
down by one to two orders of magnitude."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    from tracktolearn_b200 import synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    from tracktolearn_b200.datasets.utils import MRIDataVolume
    from tracktolearn_b200.environments import NoisyTrackingEnvironment
    from tracktolearn_b200.oracles.oracle import OracleSingleton
    dev = torch.device('cuda:0')
    shape = (24, 26, 22)
    sub = synthetic.make_subject(shape, seed=3)
    rs = np.random.RandomState(1)
    seeds = synthetic.seeds_from_mask(synthetic.ellipsoid_mask(shape, frac=0.3).numpy(), 1, rs)
    rs.shuffle(seeds)
    seeds = seeds[:300]
    affine = np.eye(4)
    subject = (MRIDataVolume(sub['sh'], affine), MRIDataVolume(sub['mask'], affine),
               MRIDataVolume(sub['mask'], affine), None, affine)
    dto = {'n_dirs': 100, 'theta': 30.0, 'npv': 1, 'binary_stopping_threshold': 0.1, 'step_size': 0.75,
           'min_length': 1.0, 'max_length': 22.5, 'oracle_checkpoint': None, 'oracle_stopping_criterion': False,
           'scoring_data': None, 'compute_reward': False, 'alignment_weighting': 0.0, 'oracle_bonus': 0.0,
           'rng': np.random.RandomState(0), 'device': dev, 'target_sh_order': 8, 'noise': 0.0, 'fa_map': None}
    env = NoisyTrackingEnvironment(subject, 'testing', dto)
    env.seeds = seeds
    sd = synthetic.actor_state_dict(615, '256-256-256', seed=9, kind='tracking')
    # reference protocol: reset + 20 steps with host actions
    alg32 = SACAuto(615, 3, '256-256-256', n_actors=300, device=dev, precision='fp32')
    alg32.agent.actor.load_state_dict(sd)
    state = env.reset(0, len(seeds))
    for _ in range(20):
        if len(env.continue_idx) == 0:
            break
        a = alg32.agent.select_action(state, 0.0).cpu().numpy()
        env.step(a)
        state, _ = env.harvest()
    n_done_api = int(env.dones.sum())
    # device mode, every tensor-core tier
    counts = {}
    for prec in ('fp16', 'tf32', 'bf16'):
        alg = SACAuto(615, 3, '256-256-256', n_actors=300, device=dev, precision=prec)
        alg.agent.actor.load_state_dict(sd)
        env.reset_streaming(0, len(seeds), 128, fp32_state=False, operand=prec)
        alg.validation_episode(None, env, 0.0)
        counts[prec] = int(env.streamline_steps())
        tr = env.get_streamlines()
        assert len(tr) == len(seeds)
    # TractOracle-Net, both tiers
    ck = synthetic.oracle_checkpoint(n_head=4, n_layers=2, seed=7)
    for prec in ('fp16', 'fp32'):
        OracleSingleton.clear()
        scores = OracleSingleton(ck, dev, precision=prec).predict(tr.streamlines[:64])
        assert np.isfinite(scores).all()
    OracleSingleton.clear()
    torch.cuda.synchronize()
    print('sanitizer target ok: api dones %d, streamline-steps %s' % (n_done_api, counts))


if __name__ == '__main__':
    main()
