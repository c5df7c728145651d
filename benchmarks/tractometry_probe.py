"""Cost of tractometry inside Tracker.track_to_file, and of its two kernels alone.

Workload: BASELINE.json configs[1] (bench.py's volume, 800 000 seeds, n_actor 50 000, the 615-1024^3-6 actor in
bf16), written to a .trk in a temporary directory, with connectome_probe's synthetic 200-label shell parcellation
and two synthetic metric volumes on the tracking grid: a smooth field in [0, 1] (FA-like) and one around 1e-3
(MD-like), both with voxel noise, so that the trilinear weights and the corner values vary along every streamline.

Reports, with the GPU's name and power limit read in the same run:
  * track_to_file without and with tractometry (2 metrics, per-streamline means in the .trk, the labels, and the
    mean-metric and mean-length matrices), alternating in one process after one warm-up run of each (medians of
    --reps, with every run's time);
  * ttl_sample_metrics alone on the length-kept streamlines for C = 1, 2, 4 and 8 (CUDA events, median of
    --kernel_reps launches), and ttl_connectome_sums alone on their end labels and (2 metrics + length) values,
    and in the worst contention case, every value landing in [0][0];
  * the numpy restatement of tests/tractometry_oracle.py over the same streamlines for C = 2 (host time), with
    its largest difference from the kernel in float32 ulps.

    python benchmarks/tractometry_probe.py [--reps 5] [--seeds 800000]
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
from benchmarks.connectome_probe import shell_parcellation  # noqa: E402
from benchmarks.oracle_filter_probe import gpu_info  # noqa: E402


def metric_volumes(dims, seed=0):
    from scipy import ndimage
    rng = np.random.RandomState(seed)
    smooth = ndimage.gaussian_filter(rng.rand(*dims), 3.0)
    smooth = (smooth - smooth.min()) / (smooth.max() - smooth.min())
    fa = np.clip(smooth + rng.randn(*dims) * 0.05, 0.0, 1.0)
    md = 1e-3 * (1.5 - smooth) + rng.randn(*dims) * 5e-5
    return np.stack([fa, md], -1).astype(np.float32)


def event_ms(launch, reps, before=None):
    if before is not None:
        before()
    launch()                                    # warm-up
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        if before is not None:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--seeds', type=int, default=800000)
    ap.add_argument('--kernel_reps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('tractometry_probe measures the GPU path: no CUDA device')
    from tests import tractometry_oracle
    from tracktolearn_b200 import _lib, synthetic
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    from tracktolearn_b200.tracking.postprocess import (connectome_packed, lengths_packed, metric_shift,
                                                        select_packed)
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
    vol = metric_volumes(dims)
    metrics = torch.from_numpy(vol).to(dev)
    res = {'gpu': name, 'power_limit': power, 'seeds': len(seeds), 'n_actor': bench.N_ACTOR, 'dims': dims,
           'labels': K - 1, 'metrics': 2, 'plain_s': [], 'tractometry_s': [], 'kept': None}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'out.trk')
        variants = {'plain_s': {},
                    'tractometry_s': dict(labels=labels, metrics=metrics, metric_names=['FA', 'MD'],
                                          save_metric_means=True, metric_connectivity_prefix=os.path.join(d, 'w_'),
                                          length_connectivity_path=os.path.join(d, 'len.npy'))}

        def run(key):
            env.seeds = seeds.copy()
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = tracker.track_to_file(env, path, bench.SHAPE, (bench.VOXEL_MM,) * 3, **variants[key])
            torch.cuda.synchronize()
            if key != 'plain_s':
                res['unsampled_streamlines'] = tracker.metrics_unsampled
            return time.perf_counter() - t0, n
        for key in variants:                     # warm-up
            run(key)
        for _ in range(args.reps):
            for key in variants:
                t, n = run(key)
                res[key].append(t)
                assert res['kept'] in (None, n), (res['kept'], n)
                res['kept'] = n

    # the kernels alone, on the length-kept streamlines of the last pass (one pass at these sizes)
    pts, offsets = env.get_streamlines_device()
    vox_size = float(np.mean(np.abs(np.asarray(env.affine_vox2rasmm))[np.diag_indices(4)][:3]))
    lens = lengths_packed(pts, offsets)
    data, off, index = select_packed(pts, offsets,
                                     keep=(lens >= min_mm / vox_size) & (lens <= bench.MAX_LENGTH_MM / vox_size))
    m = int(off.shape[0]) - 1
    res['pass_kept'], res['points'] = m, int(data.shape[0])
    lib = _lib.load()
    sp = _lib.stream_ptr(dev)
    skipped = torch.zeros((1,), dtype=torch.int64, device=dev)
    res['sample_ms'] = {}
    means2 = None
    for C in (1, 2, 4, 8):
        v = metrics[..., [c % 2 for c in range(C)]].contiguous()
        out = torch.empty((m, C), dtype=torch.float32, device=dev)

        def launch():
            _lib.check(lib.ttl_sample_metrics(_lib.ptr(data), _lib.ptr(off), m, _lib.ptr(v), C, *dims, _lib.ptr(out),
                                              _lib.ptr(skipped), sp), 'ttl_sample_metrics')
        res['sample_ms'][str(C)] = event_ms(launch, args.kernel_reps)
        if C == 2:
            means2 = out.clone()
    res['sample_median_ms'] = {k: float(np.median(t)) for k, t in res['sample_ms'].items()}
    pairs = connectome_packed(data, off, labels, None, 0.0, pairs=True)
    values = torch.cat([means2, (lens[index] * vox_size).to(torch.float32).reshape(-1, 1)], 1).contiguous()
    shifts = np.asarray([metric_shift(float(b)) for b in np.abs(vol).reshape(-1, 2).max(0)]
                        + [metric_shift(bench.MAX_LENGTH_MM * 1.001)], dtype=np.int32)
    sums = torch.zeros((3, K, K), dtype=torch.int64, device=dev)
    counts = torch.zeros((3, K, K), dtype=torch.int32, device=dev)
    zero_pairs = torch.zeros_like(pairs)

    def clear():
        sums.zero_()
        counts.zero_()

    def sums_launch(p):
        def launch():
            _lib.check(lib.ttl_connectome_sums(_lib.ptr(p), m, _lib.ptr(values), 3, K, shifts.ctypes.data,
                                               _lib.ptr(sums), _lib.ptr(counts), sp), 'ttl_connectome_sums')
        return launch
    res['sums_ms'] = event_ms(sums_launch(pairs), args.kernel_reps, clear)
    h_pairs, h_values = pairs.cpu().numpy(), values.cpu().numpy()
    want = tractometry_oracle.edge_sums(h_pairs, h_values, shifts, K)
    res['sums_exact'] = bool(np.array_equal(sums.cpu().numpy(), want[0]) and np.array_equal(counts.cpu().numpy(), want[1]))
    res['contention_ms'] = event_ms(sums_launch(zero_pairs), args.kernel_reps, clear)
    finite = np.isfinite(h_values)
    q = np.where(finite, np.rint(np.ldexp(np.where(finite, h_values, 0).astype(np.float64), shifts)), 0).astype(np.int64)
    res['contention_exact'] = bool(sums[:, 0, 0].cpu().tolist() == q.sum(0).tolist()
                                   and counts[:, 0, 0].cpu().tolist() == finite.sum(0).tolist())
    res['sums_median_ms'] = float(np.median(res['sums_ms']))
    res['contention_median_ms'] = float(np.median(res['contention_ms']))

    # the numpy restatement over the same streamlines, on the host
    h_data, h_off = data.cpu().numpy(), off.cpu().numpy()
    t0 = time.perf_counter()
    host, _ = tractometry_oracle.sample_means(h_data, h_off, vol)
    res['host_numpy_c2_s'] = time.perf_counter() - t0
    dev2 = means2.cpu().numpy()
    ok = ~np.isnan(host)
    res['device_nan_equals_host'] = bool(np.array_equal(np.isnan(dev2), np.isnan(host)))
    res['device_max_ulp_from_host'] = int(np.abs(dev2[ok].view(np.int32).astype(np.int64)
                                                 - host[ok].view(np.int32).astype(np.int64)).max(initial=0))
    for key in ('plain_s', 'tractometry_s'):
        res[key[:-2] + '_median_s'] = float(np.median(res[key]))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
