#!/usr/bin/env python3
"""ttl_tract_maps.py -- streamline density and endpoint maps of an existing tractogram, on the GPU.

Reads a .trk or .tck file, moves its points back to voxel space (``ttl_oracle_filter.voxel_points``: the
inverse of what ``ttl_track.py`` writes) and counts them on the voxel grid of --reference with
``postprocess.tract_maps_packed`` -- the maps ``ttl_track.py --out_density / --out_endpoints`` computes while
tracking.  Writes int32 NIfTI files with the reference's affine.  One process, one GPU."""
import argparse
import os
import struct
from argparse import RawTextHelpFormatter

import numpy as np
import torch

from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import detect_format, read_tck, read_trk
from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
from tracktolearn_b200.runners.ttl_track import add_map_args, check_map_args


def _trk_grid(path):
    """(dims, voxel_sizes) of a .trk header."""
    with open(path, 'rb') as f:
        raw = f.read(24)
    if len(raw) < 24 or raw[:5] != b'TRACK':
        raise ValueError('{} is not a .trk file'.format(path))
    return struct.unpack('<3h', raw[6:12]), struct.unpack('<3f', raw[12:24])


def tract_maps(in_path, reference, density=True, endpoints=True, device='cuda'):
    """Maps of the tractogram `in_path` on the grid of `reference` (a ``nifti.NiftiImage``).  Returns
    (density or None, endpoints or None, skipped) as int32 numpy arrays [X, Y, Z] and the number of points
    outside the grid."""
    from tracktolearn_b200.tracking.postprocess import tract_maps_packed
    fmt = detect_format(in_path)
    data, offsets, hdr = (read_trk if fmt == 'trk' else read_tck)(in_path)
    vox = voxel_points(data, fmt, hdr.get('voxel_sizes'), reference.affine)
    dims = tuple(int(d) for d in reference.shape[:3])
    device = torch.device(device)
    maps = [torch.zeros(dims, dtype=torch.int32, device=device) if want else None for want in (density, endpoints)]
    skipped = tract_maps_packed(torch.from_numpy(vox).to(device), torch.from_numpy(offsets).to(device), dims,
                                *maps)
    return tuple(None if m is None else m.cpu().numpy() for m in maps) + (skipped,)


def parse_args(argv=None):
    """ Streamline density and endpoint maps of a tractogram, on the voxel grid of a reference image. """
    p = argparse.ArgumentParser(description=parse_args.__doc__, formatter_class=RawTextHelpFormatter)
    p.add_argument('in_tractogram', help='Input tractogram (.trk or .tck).')
    p.add_argument('--reference', required=True, metavar='REF',
                   help='Reference image (.nii / .nii.gz): the maps\' grid and affine.  For .tck its affine\n'
                        'also maps voxels to the tractogram\'s RAS mm space; a .trk header must have its\n'
                        'dimensions and voxel sizes.')
    add_map_args(p)
    p.add_argument('-f', dest='overwrite', action='store_true', help='Force overwriting of the output files.')
    args = p.parse_args(argv)
    try:
        fmt = detect_format(args.in_tractogram)
    except ValueError as e:
        p.error(str(e))
    for f in (args.in_tractogram, args.reference):
        if not os.path.isfile(f):
            p.error('Input file {} does not exist'.format(f))
    if args.out_density is None and args.out_endpoints is None:
        p.error('Nothing to do: give --out_density, --out_endpoints or both')
    check_map_args(p, args, [args.in_tractogram, args.reference])
    try:
        ref = nifti.load(args.reference)
    except (OSError, ValueError) as e:
        p.error('Cannot read the reference {}: {}'.format(args.reference, e))
    if fmt == 'trk':
        try:
            dims, sizes = _trk_grid(args.in_tractogram)
        except ValueError as e:
            p.error(str(e))
        if tuple(dims) != tuple(ref.shape[:3]) or not np.allclose(sizes, ref.zooms[:3], rtol=1e-5, atol=0.0):
            p.error('{} has dimensions {} and voxel sizes {}; the reference has {} and {}'.format(
                args.in_tractogram, tuple(dims), tuple(sizes), tuple(ref.shape[:3]), tuple(ref.zooms[:3])))
    args.reference_image = ref
    return args


def main(argv=None):
    args = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit('ttl_tract_maps (tracktolearn_b200) needs a CUDA device; there is no CPU path')
    ref = args.reference_image
    density, endpoints, skipped = tract_maps(args.in_tractogram, ref, args.out_density is not None,
                                             args.out_endpoints is not None)
    for path, m in ((args.out_density, density), (args.out_endpoints, endpoints)):
        if m is not None:
            nifti.save(path, m, ref.affine)
            print('Wrote {}.'.format(path))
    if skipped:
        print('{} points lie outside the reference\'s grid and are not counted in the maps.'.format(skipped))
    return density, endpoints, skipped


if __name__ == '__main__':
    main()
