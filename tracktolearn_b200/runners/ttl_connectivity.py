#!/usr/bin/env python3
"""ttl_connectivity.py -- structural connectivity matrix of an existing tractogram over a parcellation, on the GPU.

Reads a .trk or .tck file, moves its points back to voxel space (``ttl_oracle_filter.voxel_points``: the
inverse of what ``ttl_track.py`` writes) and labels both ends of every streamline from the label image with
``postprocess.connectome_packed`` -- the matrix ``ttl_track.py --in_labels --out_connectivity`` computes while
tracking.  The label image is the grid and the vox -> RAS mm affine.  Writes the int32 matrix [K, K],
K = max label + 1, with ``np.save``.  One process, one GPU.

``load_labels`` is the check of a label volume that ``ttl_track.py --in_labels`` uses too."""
import argparse
import os
from argparse import RawTextHelpFormatter

import numpy as np
import torch

from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import detect_format, read_tck, read_trk
from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
from tracktolearn_b200.runners.ttl_tract_maps import _trk_grid
from tracktolearn_b200.tracking.postprocess import CONNECTOME_MAX_LABEL, radius_voxels, unlabelled_endpoints


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


def connectivity(in_path, labels_img, radius_mm=0.0, device='cuda'):
    """The int32 connectivity matrix [K, K] (numpy) of the tractogram ``in_path`` over ``labels_img`` (a
    ``nifti.NiftiImage``, which is also the grid and affine)."""
    from tracktolearn_b200.tracking.postprocess import connectome_packed
    device = torch.device(device)
    vol, K = label_volume(labels_img, labels_img.shape, labels_img.affine)
    labels = torch.from_numpy(vol).to(device)
    r = radius_voxels(radius_mm, labels_img.affine)
    fmt = detect_format(in_path)
    data, offsets, hdr = (read_trk if fmt == 'trk' else read_tck)(in_path)
    vox = voxel_points(data, fmt, hdr.get('voxel_sizes'), labels_img.affine)
    matrix = torch.zeros((K, K), dtype=torch.int32, device=device)
    connectome_packed(torch.from_numpy(vox).to(device), torch.from_numpy(offsets).to(device), labels, matrix, r)
    return matrix.cpu().numpy()


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
    p.add_argument('-f', dest='overwrite', action='store_true', help='Force overwriting of the output file.')
    args = p.parse_args(argv)
    try:
        fmt = detect_format(args.in_tractogram)
    except ValueError as e:
        p.error(str(e))
    for f in (args.in_tractogram, args.in_labels):
        if not os.path.isfile(f):
            p.error('Input file {} does not exist'.format(f))
    if not args.out_connectivity.endswith('.npy'):
        p.error('the output must be a .npy file, not {}'.format(args.out_connectivity))
    if os.path.isfile(args.out_connectivity) and not args.overwrite:
        p.error('Output file {} exists. Use -f to force overwriting'.format(args.out_connectivity))
    if os.path.abspath(args.out_connectivity) in (os.path.abspath(args.in_tractogram), os.path.abspath(args.in_labels)):
        p.error('the output {} is also an input'.format(args.out_connectivity))
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
    return args


def main(argv=None):
    args = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit('ttl_connectivity (tracktolearn_b200) needs a CUDA device; there is no CPU path')
    try:
        matrix = connectivity(args.in_tractogram, args.labels_image, args.radius)
    except ValueError as e:
        raise SystemExit(str(e))
    np.save(args.out_connectivity, matrix)
    print('Wrote the {0}x{0} connectivity matrix to {1}.'.format(matrix.shape[0], args.out_connectivity))
    print('{} streamline endpoints have no label.'.format(unlabelled_endpoints(matrix)))
    return matrix


if __name__ == '__main__':
    main()
