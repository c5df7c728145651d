#!/usr/bin/env python3
"""ttl_tractometry.py -- per-streamline means of scalar maps along an existing tractogram, on the GPU.

Reads a .trk or .tck file, moves its points back to voxel space (``ttl_oracle_filter.voxel_points``: the
inverse of what ``ttl_track.py`` writes) and samples every --in_metric at its points with
``postprocess.sample_metrics_packed`` -- the means ``ttl_track.py --save_metric_means`` computes while tracking.
The first metric is the grid and the vox -> RAS mm affine.  Writes the float32 means [n, C] in file order with
``np.save`` (NaN for a streamline with no point in the grid).  One process, one GPU.

The means are taken over the points the file holds: a file written with --compress has fewer points, spread
unevenly, and gives different means than ``ttl_track.py`` takes before compressing."""
import argparse
import os
from argparse import RawTextHelpFormatter

import numpy as np
import torch

from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import detect_format, read_tck, read_trk
from tracktolearn_b200.runners.ttl_connectivity import add_metric_arg, check_metric_names, load_metrics
from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
from tracktolearn_b200.runners.ttl_tract_maps import _trk_grid


def tractometry(in_path, metrics, affine, device='cuda'):
    """The float32 [n, C] per-streamline means (numpy) of the tractogram ``in_path`` over ``metrics``, the
    (volume, names, bounds) of ``load_metrics`` on the grid of ``affine``, and the number of points outside the
    grid."""
    from tracktolearn_b200.tracking.postprocess import sample_metrics_packed
    device = torch.device(device)
    fmt = detect_format(in_path)
    data, offsets, hdr = (read_trk if fmt == 'trk' else read_tck)(in_path)
    vox = voxel_points(data, fmt, hdr.get('voxel_sizes'), affine)
    means, skipped = sample_metrics_packed(torch.from_numpy(vox).to(device), torch.from_numpy(offsets).to(device),
                                           metrics[0].to(device))
    return means.cpu().numpy(), skipped


def parse_args(argv=None):
    """ Per-streamline means of scalar maps (FA, MD, ...) along a tractogram. """
    p = argparse.ArgumentParser(description=parse_args.__doc__, formatter_class=RawTextHelpFormatter)
    p.add_argument('in_tractogram', help='Input tractogram (.trk or .tck).')
    p.add_argument('out_means', help='Output (.npy, float32 [n, C]): the mean of each metric over every\n'
                                     'streamline\'s points, in file order and --in_metric order.')
    add_metric_arg(p)
    p.add_argument('-f', dest='overwrite', action='store_true', help='Force overwriting of the output file.')
    args = p.parse_args(argv)
    try:
        fmt = detect_format(args.in_tractogram)
    except ValueError as e:
        p.error(str(e))
    metrics = args.in_metric or []
    if not metrics:
        p.error('give at least one --in_metric NAME FILE')
    try:
        check_metric_names([n for n, _ in metrics])
    except ValueError as e:
        p.error('--in_metric: {}'.format(e))
    inputs = [args.in_tractogram] + [path for _, path in metrics]
    for f in inputs:
        if not os.path.isfile(f):
            p.error('Input file {} does not exist'.format(f))
    if not args.out_means.endswith('.npy'):
        p.error('the output must be a .npy file, not {}'.format(args.out_means))
    if os.path.isfile(args.out_means) and not args.overwrite:
        p.error('Output file {} exists. Use -f to force overwriting'.format(args.out_means))
    if os.path.abspath(args.out_means) in [os.path.abspath(f) for f in inputs]:
        p.error('the output {} is also an input'.format(args.out_means))
    try:
        ref = nifti.load(metrics[0][1])
    except (OSError, ValueError) as e:
        p.error('Cannot read the metric volume {}: {}'.format(metrics[0][1], e))
    try:
        args.metrics = load_metrics(metrics, ref.shape, ref.affine, device='cpu')
    except ValueError as e:
        p.error(str(e))
    if fmt == 'trk':
        try:
            dims, sizes = _trk_grid(args.in_tractogram)
        except ValueError as e:
            p.error(str(e))
        if tuple(dims) != tuple(ref.shape[:3]) or not np.allclose(sizes, ref.zooms[:3], rtol=1e-5, atol=0.0):
            p.error('{} has dimensions {} and voxel sizes {}; the metrics have {} and {}'.format(
                args.in_tractogram, tuple(dims), tuple(sizes), tuple(ref.shape[:3]), tuple(ref.zooms[:3])))
    args.affine = ref.affine
    return args


def main(argv=None):
    args = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit('ttl_tractometry (tracktolearn_b200) needs a CUDA device; there is no CPU path')
    means, _ = tractometry(args.in_tractogram, args.metrics, args.affine)
    np.save(args.out_means, means)
    print('Wrote the means of {} metrics ({}) over {} streamlines to {}.'.format(
        means.shape[1], ', '.join(args.metrics[1]), means.shape[0], args.out_means))
    unsampled = int(np.isnan(means[:, 0]).sum()) if means.size else 0
    if unsampled:
        print('{} streamlines have no point inside the grid: their means are NaN.'.format(unsampled))
    return means


if __name__ == '__main__':
    main()
