#!/usr/bin/env python
"""Cost of tracking noise: the configs[1] workload of bench.py (145x174x145 1.25 mm, tracking-like actor,
fp16 tier, streaming over 50 000 slots, operand-only state rows) in one process, three legs alternated and
repeated:

    noise 0            the deterministic path bench.py times
    noise 0.1 host     rng.normal on the host every step + H2D copy; the fused head and graph replay are off
    noise 0.1 device   drawn inside propagate_stop_kernel (ttl_env_step with a ttl_noise): fused head stays on

    python benchmarks/noise_probe.py [--repeats 3] [--steps 200] [--out profiles/noise_probe.json]

Every leg: reset, BURN_IN untimed steps (the alive set reaches its steady-state mix), REST_S idle, K steps timed
with CUDA events, then 20 steps with per-kernel CUDA events (ttl_prof) in a separate segment.  Reports
streamline-steps/s (spread over the repeats), the propagate_stop_kernel time, library kernels per step, and the
card's name and power limit read in the same call."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402

LEGS = (('noise 0', 0.0, 'host'), ('noise 0.1 host', 0.1, 'host'), ('noise 0.1 device', 0.1, 'device'))
PROF_STEPS = 20


def card(dev_index):
    import torch
    info = {'name': torch.cuda.get_device_name(dev_index), 'power_limit_w': None, 'sm_max_mhz': None}
    try:
        out = subprocess.run(['nvidia-smi', '-i', str(dev_index), '--query-gpu=power.limit,clocks.max.sm',
                              '--format=csv,noheader,nounits'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                             timeout=30).stdout.decode().strip().split(',')
        info['power_limit_w'], info['sm_max_mhz'] = float(out[0]), float(out[1])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        pass
    return info


def run_leg(env, actor, sigma, rng, steps, lib, dev):
    import torch
    from tracktolearn_b200 import _lib
    from tracktolearn_b200.algorithms.rl import StepRunner
    env.noise, env.noise_rng, env.noise_seed = sigma, rng, 1337
    env.reset_streaming(0, len(env.seeds), B.N_ACTOR, fp32_state=False, operand='fp16')
    runner = StepRunner(env, actor, 0.0, use_graph=False)
    for _ in range(B.BURN_IN):
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
    k1 = prof.get('propagate_stop_kernel', (0, 0.0))
    return {'ms': ms, 'us_per_step': 1000.0 * ms / steps, 'streamline_steps': units,
            'streamline_steps_per_s': units / (ms * 1e-3), 'alive_end': alive_end,
            'kernels_per_step': launches / float(steps), 'fuse_head': bool(runner.fuse_head),
            'propagate_stop_us': 1000.0 * k1[1] / max(k1[0], 1),
            'kernels_us': {k: round(1000.0 * t / c, 2) for k, (c, t) in sorted(prof.items())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'noise_probe.json'))
    a = ap.parse_args()
    import numpy as np
    import torch
    from tracktolearn_b200 import _lib, synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    if not torch.cuda.is_available():
        raise SystemExit('noise_probe.py needs a CUDA device')
    dev = torch.device('cuda:0')
    lib = _lib.load()
    env, sub = B.make_env(B.SHAPE, B.VOXEL_MM, dev)
    env.seeds = B.sharded_seed_list(sub['seed_mask'].cpu().numpy(), 1, 0)
    alg = SACAuto(B.STATE_SIZE, 3, B.HIDDEN, n_actors=B.N_ACTOR, device=dev, precision='fp16')
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(B.STATE_SIZE, B.HIDDEN, seed=1111, kind='tracking'))
    runs = {name: [] for name, _, _ in LEGS}
    for rep in range(a.repeats):
        for name, sigma, rng in LEGS:
            r = run_leg(env, alg.agent.actor, sigma, rng, a.steps, lib, dev)
            runs[name].append(r)
            print('rep %d  %-17s %8.1f us/step  %6.1f M streamline-steps/s  propagate_stop %6.1f us  '
                  '%.2f kernels/step' % (rep, name, r['us_per_step'], r['streamline_steps_per_s'] / 1e6,
                                         r['propagate_stop_us'], r['kernels_per_step']), flush=True)
    summary = {}
    for name, _, _ in LEGS:
        rates = np.asarray([r['streamline_steps_per_s'] for r in runs[name]])
        summary[name] = {'streamline_steps_per_s_median': float(np.median(rates)),
                         'streamline_steps_per_s_min': float(rates.min()),
                         'streamline_steps_per_s_max': float(rates.max()),
                         'propagate_stop_us_median': float(np.median([r['propagate_stop_us'] for r in runs[name]])),
                         'kernels_per_step': runs[name][-1]['kernels_per_step']}
    base = summary['noise 0']['streamline_steps_per_s_median']
    for name in summary:
        summary[name]['vs_noise_0'] = summary[name]['streamline_steps_per_s_median'] / base
    out = {'workload': B.WORKLOAD + ', fp16 tier, operand-only rows, no graph replay', 'steps': a.steps,
           'repeats': a.repeats, 'burn_in': B.BURN_IN, 'card': card(0), 'summary': summary, 'runs': runs}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({'card': out['card'], 'summary': summary}, indent=1))


if __name__ == '__main__':
    main()
