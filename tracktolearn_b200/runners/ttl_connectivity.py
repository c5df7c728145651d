#!/usr/bin/env python3
"""ttl_connectivity.py -- structural connectivity matrix of an existing tractogram over a parcellation, on the GPU.

Reads a .trk or .tck file, moves its points back to voxel space (``ttl_oracle_filter.voxel_points``: the
inverse of what ``ttl_track.py`` writes) and labels both ends of every streamline from the label image with
``postprocess.connectome_packed`` -- the matrix ``ttl_track.py --in_labels --out_connectivity`` computes while
tracking.  The label image is the grid and the vox -> RAS mm affine.  Writes the int32 matrix [K, K],
K = max label + 1, with ``np.save``.  With --in_metric / --out_metrics / --out_length it also writes the mean
metric and mean length (mm) of the streamlines of every edge, float64 [K, K] (NaN where no streamline), the
matrices ``ttl_track.py --out_connectivity_metrics / --out_connectivity_length`` computes.  One process, one GPU.

``load_labels`` is the check of a label volume that ``ttl_track.py --in_labels`` uses too, and
``load_metrics`` the check of metric volumes that ``ttl_track.py`` and ``ttl_tractometry.py`` use."""
import argparse
import os
import re
from argparse import RawTextHelpFormatter

import numpy as np
import torch

from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import detect_format, read_tck, read_trk
from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
from tracktolearn_b200.runners.ttl_tract_maps import _trk_grid
from tracktolearn_b200.tracking.postprocess import (CONNECTOME_MAX_LABEL, SAMPLE_MAX_METRICS, metric_shift,
                                                    radius_voxels, unlabelled_endpoints)


def label_volume(img, dims, affine, name='labels'):
    """The values of the NIfTI image ``img`` as an int32 numpy volume [X, Y, Z] (C order) and K = max + 1.
    Raises ValueError unless the shape is ``dims``, the affine is ``affine`` within 1e-4 and every value is an
    integer in [0, 16383] (any integer dtype, or a float dtype holding integral values only)."""
    dims = tuple(int(d) for d in dims)
    if tuple(img.shape) != dims:
        raise ValueError('{} has shape {}; the tracking volume\'s grid is {}'.format(name, tuple(img.shape), dims))
    if not np.allclose(img.affine, np.asarray(affine, dtype=np.float64), rtol=0.0, atol=1e-4):
        raise ValueError('{} has the affine\n{}\nand the tracking volume\n{}'.format(
            name, np.asarray(img.affine), np.asarray(affine)))
    data = np.asarray(img.data)
    if np.issubdtype(data.dtype, np.floating):
        if not np.all(np.isfinite(data)) or not np.all(data == np.floor(data)):
            raise ValueError('{} holds non-integral values: labels must be integers'.format(name))
    elif not np.issubdtype(data.dtype, np.integer):
        raise ValueError('{} has the data type {}: labels must be integers'.format(name, data.dtype))
    lo, hi = (data.min(), data.max()) if data.size else (0, 0)
    if lo < 0 or hi > CONNECTOME_MAX_LABEL:
        raise ValueError('{} has values in [{}, {}]: labels must lie in [0, {}]'.format(
            name, lo, hi, CONNECTOME_MAX_LABEL))
    return np.ascontiguousarray(data, dtype=np.int32), int(hi) + 1


def load_labels(path, dims, affine, device='cuda'):
    """Reads the label volume ``path`` (NIfTI) on the tracking grid: ``label_volume``'s checks, then returns
    (int32 volume [X, Y, Z] on ``device``, K)."""
    try:
        img = nifti.load(path)
    except (OSError, ValueError) as e:
        raise ValueError('Cannot read the label volume {}: {}'.format(path, e))
    vol, K = label_volume(img, dims, affine, name=str(path))
    return torch.from_numpy(vol).to(device), K


def check_metric_names(names):
    """Raises ValueError unless there are 1 to 8 names, each matching [A-Za-z][A-Za-z0-9_]{0,13} (so that
    ``mean_NAME`` fits a .trk property name) and all distinct."""
    names = list(names)
    if not 1 <= len(names) <= SAMPLE_MAX_METRICS:
        raise ValueError('between 1 and %d metrics can be sampled, not %d' % (SAMPLE_MAX_METRICS, len(names)))
    for name in names:
        if not METRIC_NAME.fullmatch(name):
            raise ValueError('the metric name %r must be a letter followed by at most 13 letters, digits or '
                             'underscores' % name)
    if len(set(names)) != len(names):
        raise ValueError('the metric names %s are not distinct' % ', '.join(names))


METRIC_NAME = re.compile(r'[A-Za-z][A-Za-z0-9_]{0,13}')


def metric_outputs(prefix, names):
    """The files of the mean-weighted matrices: PREFIX + NAME + '.npy' per metric ([] without a prefix)."""
    return [] if prefix is None else [prefix + name + '.npy' for name in names]


def add_metric_arg(p):
    p.add_argument('--in_metric', nargs=2, action='append', metavar=('NAME', 'FILE'), default=None,
                   help='A scalar map (.nii / .nii.gz, any numeric type, finite) on the grid, and its\n'
                        'name ([A-Za-z][A-Za-z0-9_]{0,13}).  Repeat for up to 8 metrics.')


def load_metrics(metrics, dims, affine, device='cuda'):
    """Reads the metric volumes ``metrics`` [(NAME, path), ...] (NIfTI) on the grid ``dims`` / ``affine``.  Each
    must be 3-D of shape ``dims``, with ``affine`` within 1e-4, of a numeric dtype (converted to float32) and
    finite everywhere; the names pass ``check_metric_names``.  Returns (float32 tensor (X, Y, Z, C) on
    ``device``, the C names, the C bounds: the largest |value| of each volume).  Raises ValueError."""
    metrics = [(str(n), str(p)) for n, p in metrics]
    check_metric_names([n for n, _ in metrics])
    dims = tuple(int(d) for d in dims)
    vols, bounds = [], []
    for name, path in metrics:
        try:
            img = nifti.load(path)
        except (OSError, ValueError) as e:
            raise ValueError('Cannot read the metric volume {}: {}'.format(path, e))
        if tuple(img.shape) != dims:
            raise ValueError('the metric {} ({}) has shape {}; the grid is {}'.format(name, path, tuple(img.shape), dims))
        if not np.allclose(img.affine, np.asarray(affine, dtype=np.float64), rtol=0.0, atol=1e-4):
            raise ValueError('the metric {} ({}) has the affine\n{}\nand the grid\n{}'.format(
                name, path, np.asarray(img.affine), np.asarray(affine)))
        data = np.asarray(img.data)
        if not (np.issubdtype(data.dtype, np.integer) or np.issubdtype(data.dtype, np.floating)
                or data.dtype == np.bool_):
            raise ValueError('the metric {} ({}) has the data type {}: it must be numeric'.format(name, path, data.dtype))
        vol = np.ascontiguousarray(data, dtype=np.float32)
        if not np.all(np.isfinite(vol)):
            raise ValueError('the metric {} ({}) holds NaN or infinite values (in float32)'.format(name, path))
        bound = float(np.abs(vol).max()) if vol.size else 0.0
        try:
            metric_shift(bound)
        except ValueError as e:
            raise ValueError('the metric {} ({}): {}'.format(name, path, e))
        vols.append(vol)
        bounds.append(bound)
    vol = torch.from_numpy(np.ascontiguousarray(np.stack(vols, axis=-1))).to(device)
    return vol, [n for n, _ in metrics], bounds


def connectivity(in_path, labels_img, radius_mm=0.0, device='cuda'):
    """The int32 connectivity matrix [K, K] (numpy) of the tractogram ``in_path`` over ``labels_img`` (a
    ``nifti.NiftiImage``, which is also the grid and affine)."""
    return connectivity_matrices(in_path, labels_img, radius_mm, device=device)[0]


def connectivity_matrices(in_path, labels_img, radius_mm=0.0, metrics=None, length=False, device='cuda'):
    """``connectivity`` and, from the same end labels, the mean-weighted matrices: ``metrics`` is
    ``load_metrics``' (volume, names, bounds) on the label image's grid, ``length`` asks for the mean length in mm
    (the lengths of the points in the label grid's voxels times the mean |diagonal| of its affine).  Returns (the
    int32 count matrix, float64 [C, K, K] metric means or None, float64 [K, K] mean lengths or None), numpy."""
    from tracktolearn_b200.tracking.postprocess import (connectome_packed, connectome_sums_packed, edge_means,
                                                        lengths_packed, sample_metrics_packed)
    device = torch.device(device)
    vol, K = label_volume(labels_img, labels_img.shape, labels_img.affine)
    labels = torch.from_numpy(vol).to(device)
    r = radius_voxels(radius_mm, labels_img.affine)
    fmt = detect_format(in_path)
    data, offsets, hdr = (read_trk if fmt == 'trk' else read_tck)(in_path)
    vox = voxel_points(data, fmt, hdr.get('voxel_sizes'), labels_img.affine)
    d, o = torch.from_numpy(vox).to(device), torch.from_numpy(offsets).to(device)
    matrix = torch.zeros((K, K), dtype=torch.int32, device=device)
    weighted = metrics is not None or length
    pairs = connectome_packed(d, o, labels, matrix, r, pairs=weighted)
    if not weighted:
        return matrix.cpu().numpy(), None, None
    cols, shifts = [], []
    if metrics is not None:
        means, _ = sample_metrics_packed(d, o, metrics[0])
        cols.append(means)
        shifts += [metric_shift(b) for b in metrics[2]]
    if length:
        vox_size = float(np.mean(np.abs(np.asarray(labels_img.affine, dtype=np.float64))[np.diag_indices(4)][:3]))
        mm = (lengths_packed(d, o) * vox_size).to(torch.float32)
        cols.append(mm.reshape(-1, 1))
        shifts.append(metric_shift(float(mm.max().item()) if mm.numel() else 0.0))
    values = torch.cat(cols, 1).contiguous()
    sums = torch.zeros((values.shape[1], K, K), dtype=torch.int64, device=device)
    counts = torch.zeros((values.shape[1], K, K), dtype=torch.int32, device=device)
    connectome_sums_packed(pairs, values, shifts, sums, counts)
    mean = edge_means(sums, counts, shifts)
    n_metrics = len(shifts) - int(length)
    return matrix.cpu().numpy(), (mean[:n_metrics] if metrics is not None else None), (mean[-1] if length else None)


def parse_args(argv=None):
    """ Structural connectivity matrix of a tractogram over a parcellation (streamline counts between the
    labels of its two ends). """
    p = argparse.ArgumentParser(description=parse_args.__doc__, formatter_class=RawTextHelpFormatter)
    p.add_argument('in_tractogram', help='Input tractogram (.trk or .tck).')
    p.add_argument('in_labels', help='Label volume (.nii / .nii.gz, integers in [0, 16383], 0 = no region): the\n'
                                     'grid and affine.  For .tck its affine also maps voxels to the\n'
                                     'tractogram\'s RAS mm space; a .trk header must have its dimensions\n'
                                     'and voxel sizes.')
    p.add_argument('out_connectivity', help='Output matrix (.npy, int32 [K, K], K = max label + 1).')
    p.add_argument('--radius', type=float, default=0.0, metavar='MM',
                   help='An endpoint whose own voxel is unlabelled takes the label of the nearest\n'
                        'labelled voxel within MM (at most 8 voxels). 0: its own voxel only. [%(default)s]')
    add_metric_arg(p)
    p.add_argument('--out_metrics', metavar='PREFIX', default=None,
                   help='Write the mean of each --in_metric over the streamlines of every edge to\n'
                        'PREFIX + NAME + ".npy" (float64 [K, K], NaN where no streamline).')
    p.add_argument('--out_length', metavar='FILE', default=None,
                   help='Mean length in mm of the streamlines of every edge (.npy, float64 [K, K]).')
    p.add_argument('-f', dest='overwrite', action='store_true', help='Force overwriting of the output file.')
    args = p.parse_args(argv)
    try:
        fmt = detect_format(args.in_tractogram)
    except ValueError as e:
        p.error(str(e))
    metrics = args.in_metric or []
    for f in [args.in_tractogram, args.in_labels] + [path for _, path in metrics]:
        if not os.path.isfile(f):
            p.error('Input file {} does not exist'.format(f))
    if bool(metrics) != (args.out_metrics is not None):
        p.error('--in_metric needs --out_metrics, and --out_metrics needs --in_metric')
    try:
        if metrics:
            check_metric_names([n for n, _ in metrics])
    except ValueError as e:
        p.error('--in_metric: {}'.format(e))
    outs = [args.out_connectivity] + metric_outputs(args.out_metrics, [n for n, _ in metrics]) + \
        ([args.out_length] if args.out_length is not None else [])
    taken = [os.path.abspath(f) for f in [args.in_tractogram, args.in_labels] + [path for _, path in metrics]]
    for out in outs:
        if not out.endswith('.npy'):
            p.error('the output must be a .npy file, not {}'.format(out))
        if os.path.isfile(out) and not args.overwrite:
            p.error('Output file {} exists. Use -f to force overwriting'.format(out))
        if os.path.abspath(out) in taken:
            p.error('the output {} is also an input or another output'.format(out))
        taken.append(os.path.abspath(out))
    try:
        img = nifti.load(args.in_labels)
    except (OSError, ValueError) as e:
        p.error('Cannot read the label volume {}: {}'.format(args.in_labels, e))
    try:
        label_volume(img, img.shape, img.affine, name=args.in_labels)
    except ValueError as e:
        p.error(str(e))
    try:
        radius_voxels(args.radius, img.affine)
    except ValueError as e:
        p.error('--radius: {}'.format(e))
    if fmt == 'trk':
        try:
            dims, sizes = _trk_grid(args.in_tractogram)
        except ValueError as e:
            p.error(str(e))
        if tuple(dims) != tuple(img.shape[:3]) or not np.allclose(sizes, img.zooms[:3], rtol=1e-5, atol=0.0):
            p.error('{} has dimensions {} and voxel sizes {}; the label volume has {} and {}'.format(
                args.in_tractogram, tuple(dims), tuple(sizes), tuple(img.shape[:3]), tuple(img.zooms[:3])))
    args.labels_image = img
    args.metrics = None
    if metrics:
        try:
            args.metrics = load_metrics(metrics, img.shape, img.affine, device='cpu')
        except ValueError as e:
            p.error(str(e))
    return args


def main(argv=None):
    args = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit('ttl_connectivity (tracktolearn_b200) needs a CUDA device; there is no CPU path')
    metrics = None
    if args.metrics is not None:
        vol, names, bounds = args.metrics
        metrics = (vol.to('cuda'), names, bounds)
    try:
        matrix, metric_means, length_means = connectivity_matrices(
            args.in_tractogram, args.labels_image, args.radius, metrics=metrics, length=args.out_length is not None)
    except ValueError as e:
        raise SystemExit(str(e))
    np.save(args.out_connectivity, matrix)
    print('Wrote the {0}x{0} connectivity matrix to {1}.'.format(matrix.shape[0], args.out_connectivity))
    print('{} streamline endpoints have no label.'.format(unlabelled_endpoints(matrix)))
    if metric_means is not None:
        for path, m in zip(metric_outputs(args.out_metrics, metrics[1]), metric_means):
            np.save(path, m)
            print('Wrote {}.'.format(path))
    if length_means is not None:
        np.save(args.out_length, length_means)
        print('Wrote {}.'.format(args.out_length))
    return matrix


if __name__ == '__main__':
    main()
