#!/usr/bin/env python
"""Cost of sampling the stochastic policy: the configs[1] workload of bench.py (145x174x145 1.25 mm, tracking-like
actor, fp16 tier, streaming over 50 000 slots, operand-only state rows) in one process, three legs alternated and
repeated:

    prob 0             the deterministic path bench.py times (fused head)
    prob 1 torch eps   torch.randn per step, actor head_finish_kernel, then the env step: the route without a
                       policy seed, here streamed like the others so that the comparison is like for like
    prob 1 device eps  eps drawn inside propagate_policy_kernel (ttl_env_step with a ttl_policy): fused head stays on

    python benchmarks/policy_probe.py [--repeats 3] [--steps 200] [--burn-in 384] [--out profiles/policy_probe.json]

Every leg: reset, BURN_IN untimed steps, REST_S idle, K steps timed with CUDA events, then 20 steps with
per-kernel CUDA events (ttl_prof) in a separate segment.  Reports streamline-steps/s (spread over the repeats),
the propagate kernel's time, every library kernel's time, library kernels per step, the alive count at the end
of the timed window (the synthetic actor's log_std is about 0, so at prob 1 streamlines are short and the seed
list drains sooner), and the card's name and power limit read in the same call."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402
from benchmarks.noise_probe import card  # noqa: E402

LEGS = (('prob 0', 0.0, None), ('prob 1 torch eps', 1.0, None), ('prob 1 device eps', 1.0, 1337))
PROF_STEPS = 20


def run_leg(env, actor, prob, policy_seed, steps, burn_in, lib, dev):
    import torch
    from tracktolearn_b200 import _lib
    from tracktolearn_b200.algorithms.rl import StepRunner
    torch.manual_seed(1337)
    env.reset_streaming(0, len(env.seeds), B.N_ACTOR, fp32_state=False, operand='fp16')
    runner = StepRunner(env, actor, prob, use_graph=False, policy_seed=policy_seed)
    for _ in range(burn_in):
        runner.step()
    env.n_alive()
    time.sleep(B.REST_S)
    stream = torch.cuda.current_stream(dev)
    s0, n0 = env.streamline_steps(), lib.ttl_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        runner.step()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    launches = lib.ttl_launch_count() - n0
    env.n_alive()
    units = env.streamline_steps() - s0
    alive_end = int(env._batch.ctrl_host[env._cur])
    lib.ttl_prof_enable(1)
    for _ in range(PROF_STEPS):
        runner.step()
    torch.cuda.synchronize(dev)
    prof = _lib.prof_report()
    lib.ttl_prof_enable(0)
    k1 = prof.get('propagate_policy_kernel' if runner.policy_seed is not None else 'propagate_stop_kernel', (0, 0.0))
    return {'ms': ms, 'us_per_step': 1000.0 * ms / steps, 'streamline_steps': units,
            'streamline_steps_per_s': units / (ms * 1e-3), 'alive_end': alive_end,
            'kernels_per_step': launches / float(steps), 'fuse_head': bool(runner.fuse_head),
            'propagate_us': 1000.0 * k1[1] / max(k1[0], 1),
            'kernels_us': {k: round(1000.0 * t / c, 2) for k, (c, t) in sorted(prof.items())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--burn-in', type=int, default=B.BURN_IN,
                    help='untimed steps per leg (short prob-1 streamlines drain the seed list sooner)')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'policy_probe.json'))
    a = ap.parse_args()
    import numpy as np
    import torch
    from tracktolearn_b200 import _lib, synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    if not torch.cuda.is_available():
        raise SystemExit('policy_probe.py needs a CUDA device')
    dev = torch.device('cuda:0')
    lib = _lib.load()
    env, sub = B.make_env(B.SHAPE, B.VOXEL_MM, dev)
    env.seeds = B.sharded_seed_list(sub['seed_mask'].cpu().numpy(), 1, 0)
    alg = SACAuto(B.STATE_SIZE, 3, B.HIDDEN, n_actors=B.N_ACTOR, device=dev, precision='fp16')
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(B.STATE_SIZE, B.HIDDEN, seed=1111, kind='tracking'))
    runs = {name: [] for name, _, _ in LEGS}
    for rep in range(a.repeats):
        for name, prob, seed in LEGS:
            r = run_leg(env, alg.agent.actor, prob, seed, a.steps, a.burn_in, lib, dev)
            runs[name].append(r)
            print('rep %d  %-17s %8.1f us/step  %6.1f M streamline-steps/s  propagate %6.1f us  '
                  '%.2f kernels/step  alive at end %d' % (rep, name, r['us_per_step'], r['streamline_steps_per_s'] / 1e6,
                                                          r['propagate_us'], r['kernels_per_step'], r['alive_end']),
                  flush=True)
    summary = {}
    for name, _, _ in LEGS:
        rates = np.asarray([r['streamline_steps_per_s'] for r in runs[name]])
        summary[name] = {'streamline_steps_per_s_median': float(np.median(rates)),
                         'streamline_steps_per_s_min': float(rates.min()),
                         'streamline_steps_per_s_max': float(rates.max()),
                         'propagate_us_median': float(np.median([r['propagate_us'] for r in runs[name]])),
                         'kernels_per_step': runs[name][-1]['kernels_per_step'],
                         'kernels_us': runs[name][-1]['kernels_us'],
                         'alive_end': [r['alive_end'] for r in runs[name]]}
    base = summary['prob 0']['streamline_steps_per_s_median']
    for name in summary:
        summary[name]['vs_prob_0'] = summary[name]['streamline_steps_per_s_median'] / base
    out = {'workload': B.WORKLOAD + ', fp16 tier, operand-only rows, streaming, no graph replay', 'steps': a.steps,
           'repeats': a.repeats, 'burn_in': a.burn_in, 'card': card(0), 'summary': summary, 'runs': runs}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({'card': out['card'], 'summary': summary}, indent=1))


if __name__ == '__main__':
    main()
