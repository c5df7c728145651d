"""Cost of the streamline density and endpoint maps inside Tracker.track_to_file.

Workload: BASELINE.json configs[1] (bench.py's volume, 800 000 seeds, n_actor 50 000, the 615-1024^3-6
actor in bf16), written to a .trk in a temporary directory -- without and with both maps, alternating in one
process after one warm-up run of each.  Reports the wall time of each variant (medians), the map kernel
alone on the length-kept streamlines of the run (CUDA events over repeated launches), the numpy restatement
of tests/maps_oracle.py over the same streamlines (host time, with a check that both give the same maps),
the time to download both maps and write them as .nii files, and the GPU's name and power limit read in
the same run.

    python benchmarks/density_probe.py [--reps 3] [--seeds 800000]
"""
import argparse
import json
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from benchmarks.oracle_filter_probe import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--seeds', type=int, default=800000)
    ap.add_argument('--kernel_reps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('density_probe measures the GPU path: no CUDA device')
    from tests import maps_oracle
    from tracktolearn_b200 import _lib, synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.tracking.postprocess import lengths_packed, select_packed
    from tracktolearn_b200.tracking.tracker import Tracker
    dev = torch.device('cuda:0')
    env, sub = bench.make_env(bench.SHAPE, bench.VOXEL_MM, dev)
    seeds = bench.draw_seeds(sub['seed_mask'].cpu().numpy(), 0)[:args.seeds]
    alg = SACAuto(bench.STATE_SIZE, 3, bench.HIDDEN, n_actors=bench.N_ACTOR, device=dev, precision='bf16')
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(bench.STATE_SIZE, bench.HIDDEN, seed=1111,
                                                               kind='tracking'))
    min_mm = 10.0
    tracker = Tracker(alg, bench.N_ACTOR, min_length=min_mm, max_length=bench.MAX_LENGTH_MM)
    name, power = gpu_info()
    dims = (env._volume.X, env._volume.Y, env._volume.Z)
    res = {'gpu': name, 'power_limit': power, 'seeds': len(seeds), 'n_actor': bench.N_ACTOR, 'dims': dims,
           'plain_s': [], 'maps_s': [], 'kept': None, 'skipped': None}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'out.trk')
        maps = dict(density_path=os.path.join(d, 'density.nii'), endpoints_path=os.path.join(d, 'endpoints.nii'))

        def run(with_maps):
            env.seeds = seeds.copy()
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = tracker.track_to_file(env, path, bench.SHAPE, (bench.VOXEL_MM,) * 3, **(maps if with_maps else {}))
            torch.cuda.synchronize()
            return time.perf_counter() - t0, n
        for with_maps in (False, True):          # warm-up
            run(with_maps)
        for _ in range(args.reps):
            t, n = run(False)
            res['plain_s'].append(t)
            t, n_maps = run(True)
            res['maps_s'].append(t)
            assert n_maps == n, (n_maps, n)
            res['kept'], res['skipped'] = n, tracker.maps_skipped
        file_maps = [nifti.load(maps[k]).data for k in ('density_path', 'endpoints_path')]

    # the kernel alone, on the length-kept streamlines of the last pass (one pass at these sizes)
    pts, offsets = env.get_streamlines_device()
    vox_size = float(np.mean(np.abs(np.asarray(env.affine_vox2rasmm))[np.diag_indices(4)][:3]))
    lens = lengths_packed(pts, offsets)
    data, off, _ = select_packed(pts, offsets, keep=(lens >= min_mm / vox_size) & (lens <= bench.MAX_LENGTH_MM / vox_size))
    m = int(off.shape[0]) - 1
    res['pass_kept'], res['points'] = m, int(data.shape[0])
    lib = _lib.load()
    density = torch.zeros(dims, dtype=torch.int32, device=dev)
    endpoints = torch.zeros(dims, dtype=torch.int32, device=dev)
    skipped = torch.zeros((1,), dtype=torch.int64, device=dev)
    sp = _lib.stream_ptr(dev)

    def launch():
        _lib.check(lib.ttl_tract_maps(_lib.ptr(data), _lib.ptr(off), m, *dims, _lib.ptr(density), _lib.ptr(endpoints),
                                      _lib.ptr(skipped), sp), 'ttl_tract_maps')
    launch()                                   # warm-up
    torch.cuda.synchronize()
    times = []
    for _ in range(args.kernel_reps):
        density.zero_()
        endpoints.zero_()
        skipped.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    res['kernel_ms'] = times
    res['kernel_median_ms'] = float(np.median(times))
    dev_maps = (density.cpu().numpy(), endpoints.cpu().numpy(), int(skipped.item()))
    # what track_to_file adds after the last pass: both maps to the host and into .nii files
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        for k, t in enumerate((density, endpoints)):
            nifti.save(os.path.join(d, '%d.nii' % k), t.cpu().numpy(), env.affine_vox2rasmm)
        res['download_and_write_s'] = time.perf_counter() - t0

    # the numpy restatement over the same streamlines, on the host
    h_data, h_off = data.cpu().numpy(), off.cpu().numpy()
    t0 = time.perf_counter()
    host_maps = maps_oracle.tract_maps_fast(h_data, h_off, dims)
    res['host_numpy_s'] = time.perf_counter() - t0
    res['device_equals_host'] = bool(all(np.array_equal(a, b) for a, b in zip(dev_maps[:2], host_maps[:2]))
                                     and dev_maps[2] == host_maps[2])
    res['file_maps_equal_kernel_maps'] = bool(all(np.array_equal(a, b) for a, b in zip(file_maps, dev_maps[:2])))
    res['plain_median_s'] = float(np.median(res['plain_s']))
    res['maps_median_s'] = float(np.median(res['maps_s']))
    res['overhead_median_s'] = res['maps_median_s'] - res['plain_median_s']
    print(json.dumps(res))


if __name__ == '__main__':
    main()
