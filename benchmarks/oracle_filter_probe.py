"""Cost of filtering a tractogram by TractOracle-Net score inside Tracker.track_to_file.

Workload: BASELINE.json configs[1] (bench.py's volume, 800 000 seeds, n_actor 50 000, the 615-1024^3-6
actor in bf16), written to a .trk in a temporary directory -- without and with the oracle (a synthetic
4-layer TransformerOracle, fp16 tier, threshold 0.5), alternating in one process after one warm-up run
of each.  Reports the wall time of each variant, the oracle scoring time alone (CUDA events around
predict_device) and the streamlines kept after the length filter and after the oracle filter, with the
GPU's name and power limit.

    python benchmarks/oracle_filter_probe.py [--reps 3] [--seeds 800000]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402


class TimedOracle(object):
    """Forwards predict_device and accumulates its device time and the streamlines it scored."""

    def __init__(self, oracle):
        self.oracle, self.device = oracle, oracle.device
        self.events, self.scored = [], 0

    def predict_device(self, points, offsets, distributed=True):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        scores = self.oracle.predict_device(points, offsets, distributed=distributed)
        e1.record()
        self.events.append((e0, e1))
        self.scored += int(offsets.shape[0]) - 1
        return scores

    def take(self):
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in self.events)
        out = (ms, self.scored)
        self.events, self.scored = [], 0
        return out


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(',')]
    except Exception:
        name, power = torch.cuda.get_device_name(0), 'unknown'
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--seeds', type=int, default=800000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('oracle_filter_probe measures the GPU path: no CUDA device')
    from tracktolearn_b200 import synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    from tracktolearn_b200.oracles.oracle import OracleSingleton
    from tracktolearn_b200.tracking.tracker import Tracker
    dev = torch.device('cuda:0')
    env, sub = bench.make_env(bench.SHAPE, bench.VOXEL_MM, dev)
    seeds = bench.draw_seeds(sub['seed_mask'].cpu().numpy(), 0)[:args.seeds]
    alg = SACAuto(bench.STATE_SIZE, 3, bench.HIDDEN, n_actors=bench.N_ACTOR, device=dev, precision='bf16')
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(bench.STATE_SIZE, bench.HIDDEN, seed=1111,
                                                               kind='tracking'))
    oracle = TimedOracle(OracleSingleton(synthetic.oracle_checkpoint(seed=78), dev, precision='fp16'))
    tracker = Tracker(alg, bench.N_ACTOR, min_length=10.0, max_length=bench.MAX_LENGTH_MM)
    name, power = gpu_info()
    res = {'gpu': name, 'power_limit': power, 'seeds': len(seeds), 'n_actor': bench.N_ACTOR,
           'plain_s': [], 'oracle_s': [], 'scoring_ms': [], 'length_kept': None, 'oracle_kept': None}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'out.trk')

        def run(with_oracle):
            env.seeds = seeds.copy()
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = tracker.track_to_file(env, path, bench.SHAPE, (bench.VOXEL_MM,) * 3,
                                      oracle=oracle if with_oracle else None)
            torch.cuda.synchronize()
            return time.perf_counter() - t0, n
        for with_oracle in (False, True):          # warm-up
            run(with_oracle)
            oracle.take()
        for _ in range(args.reps):
            t, n = run(False)
            res['plain_s'].append(t)
            res['length_kept'] = n
            t, n = run(True)
            ms, scored = oracle.take()
            res['oracle_s'].append(t)
            res['scoring_ms'].append(ms)
            res['oracle_kept'] = n
            assert scored == res['length_kept'], (scored, res['length_kept'])
    res['plain_median_s'] = float(np.median(res['plain_s']))
    res['oracle_median_s'] = float(np.median(res['oracle_s']))
    res['scoring_median_ms'] = float(np.median(res['scoring_ms']))
    res['scoring_rate_M_per_s'] = res['length_kept'] / res['scoring_median_ms'] / 1e3
    print(json.dumps(res))


if __name__ == '__main__':
    main()
