"""Cost of the connectivity matrix inside Tracker.track_to_file, and of its kernel alone.

Workload: BASELINE.json configs[1] (bench.py's volume, 800 000 seeds, n_actor 50 000, the 615-1024^3-6 actor in
bf16), written to a .trk in a temporary directory, with a synthetic parcellation: 200 labels, each voxel of a
shell around the tracking mask (two voxels outside it, one inside its border) taking the label of the nearest
of 200 centres drawn in the shell.  An agent seeded at the interface ends on or near that shell, as it would
near a cortical parcellation.

Reports, with the GPU's name and power limit read in the same run:
  * track_to_file without and with --out_connectivity at R = 0 and R = 4 mm, alternating in one process after
    one warm-up run of each (medians of --reps);
  * ttl_connectome alone on the length-kept streamlines at radii of 0, 2, 4 and 8 voxels (CUDA events, median
    of --kernel_reps launches, matrix only, as track_to_file calls it);
  * the worst contention case: an all-zero label volume, every streamline adding to [0][0];
  * the numpy restatement of tests/connectome_oracle.py over the same streamlines at R = 4 mm (host time), with
    a check that it gives the kernel's matrix.

    python benchmarks/connectome_probe.py [--reps 3] [--seeds 800000]
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


def shell_parcellation(mask, n_labels=200, seed=0):
    from scipy import ndimage
    from scipy.spatial import cKDTree
    inside = np.asarray(mask) > 0.5
    shell = ndimage.binary_dilation(inside, iterations=2) & ~ndimage.binary_erosion(inside, iterations=1)
    idx = np.argwhere(shell)
    rng = np.random.RandomState(seed)
    centres = idx[rng.choice(len(idx), n_labels, replace=False)]
    lab = np.zeros(inside.shape, np.int32)
    lab[shell] = cKDTree(centres).query(idx)[1] + 1
    return lab


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--seeds', type=int, default=800000)
    ap.add_argument('--kernel_reps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('connectome_probe measures the GPU path: no CUDA device')
    from tests import connectome_oracle
    from tracktolearn_b200 import _lib, synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    from tracktolearn_b200.tracking.postprocess import lengths_packed, radius_voxels, select_packed
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
    lab = shell_parcellation(sub['mask'].cpu().numpy())
    labels = torch.from_numpy(lab).to(dev)
    K = int(lab.max()) + 1
    res = {'gpu': name, 'power_limit': power, 'seeds': len(seeds), 'n_actor': bench.N_ACTOR, 'dims': dims,
           'labels': K - 1, 'labelled_voxels': int((lab > 0).sum()), 'plain_s': [], 'r0_s': [], 'r4mm_s': [],
           'kept': None, 'unlabelled_endpoints': {}}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'out.trk')
        variants = {'plain_s': {}, 'r0_s': dict(labels=labels, connectivity_path=os.path.join(d, 'c0.npy')),
                    'r4mm_s': dict(labels=labels, connectivity_path=os.path.join(d, 'c4.npy'),
                                   connectivity_radius=4.0)}

        def run(key):
            env.seeds = seeds.copy()
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = tracker.track_to_file(env, path, bench.SHAPE, (bench.VOXEL_MM,) * 3, **variants[key])
            torch.cuda.synchronize()
            if key != 'plain_s':
                res['unlabelled_endpoints'][key[:-2]] = tracker.connectome_unlabelled
            return time.perf_counter() - t0, n
        for key in variants:                     # warm-up
            run(key)
        for _ in range(args.reps):
            for key in variants:
                t, n = run(key)
                res[key].append(t)
                assert res['kept'] in (None, n), (res['kept'], n)
                res['kept'] = n
        file_r4 = np.load(variants['r4mm_s']['connectivity_path'])

    # the kernel alone, on the length-kept streamlines of the last pass (one pass at these sizes)
    pts, offsets = env.get_streamlines_device()
    vox_size = float(np.mean(np.abs(np.asarray(env.affine_vox2rasmm))[np.diag_indices(4)][:3]))
    lens = lengths_packed(pts, offsets)
    data, off, _ = select_packed(pts, offsets, keep=(lens >= min_mm / vox_size) & (lens <= bench.MAX_LENGTH_MM / vox_size))
    m = int(off.shape[0]) - 1
    res['pass_kept'], res['points'] = m, int(data.shape[0])
    lib = _lib.load()
    matrix = torch.zeros((K, K), dtype=torch.int32, device=dev)
    zeros = torch.zeros_like(labels)
    sp = _lib.stream_ptr(dev)

    def time_kernel(vol, r):
        def launch():
            _lib.check(lib.ttl_connectome(_lib.ptr(data), _lib.ptr(off), m, _lib.ptr(vol), *dims, K, float(r),
                                          _lib.ptr(matrix), None, sp), 'ttl_connectome')
        matrix.zero_()
        launch()                                # warm-up
        torch.cuda.synchronize()
        times = []
        for _ in range(args.kernel_reps):
            matrix.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        return times
    res['kernel_ms'] = {}
    for r in (0, 2, 4, 8):
        res['kernel_ms'][str(r)] = time_kernel(labels, r)
    r4 = radius_voxels(4.0, env.affine_vox2rasmm)
    res['r4mm_vox'] = r4
    res['kernel_ms']['r4mm'] = time_kernel(labels, r4)
    dev_r4 = matrix.cpu().numpy()
    res['contention_ms'] = time_kernel(zeros, 0)
    res['contention_exact'] = bool(int(matrix[0, 0]) == int((off[1:] > off[:-1]).sum()) == int(matrix.sum()))
    res['kernel_median_ms'] = {k: float(np.median(v)) for k, v in res['kernel_ms'].items()}
    res['contention_median_ms'] = float(np.median(res['contention_ms']))

    # the numpy restatement over the same streamlines, on the host
    h_data, h_off = data.cpu().numpy(), off.cpu().numpy()
    t0 = time.perf_counter()
    host_r4 = connectome_oracle.connectome_fast(h_data, h_off, lab, r4)[0]
    res['host_numpy_r4mm_s'] = time.perf_counter() - t0
    res['device_equals_host_r4mm'] = bool(np.array_equal(dev_r4, host_r4))
    res['file_equals_kernel_r4mm'] = bool(np.array_equal(file_r4, dev_r4))
    for key in ('plain_s', 'r0_s', 'r4mm_s'):
        res[key[:-2] + '_median_s'] = float(np.median(res[key]))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
