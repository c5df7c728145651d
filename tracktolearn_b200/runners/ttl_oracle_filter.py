#!/usr/bin/env python3
"""ttl_oracle_filter.py -- keep the streamlines of a tractogram that TractOracle-Net judges plausible.

Reads a .trk or .tck file, scores every streamline on the GPU (``OracleSingleton.predict_device``) on
its voxel-space points, and writes the streamlines whose score is >= --threshold to a file of the same
format.  Kept records are copied byte for byte from the input (points, per-point scalars, existing
properties); --save_scores (.trk) appends the score as one more per-streamline property.

Under torchrun every rank reads the file, the ranks share the scoring and rank 0 writes."""
import argparse
import os
import struct
from argparse import RawTextHelpFormatter

import numpy as np
import torch

from tracktolearn_b200.io.streamlines import detect_format, read_tck, read_trk

TRK_MAX_PROPERTIES = 10


def voxel_points(data, fmt, voxel_sizes=None, reference_affine=None):
    """File-space points -> float32 voxel coordinates, the space the tracker scores in.  .trk: the inverse
    of TrkWriter's (voxel + 0.5) * voxel size; .tck: the inverse of the reference's vox -> RAS mm affine."""
    d = np.asarray(data, dtype=np.float64)
    if fmt == 'trk':
        return (d / np.asarray(voxel_sizes, dtype=np.float64) - 0.5).astype(np.float32)
    inv = np.linalg.inv(np.asarray(reference_affine, dtype=np.float64))
    return (d @ inv[:3, :3].T + inv[:3, 3]).astype(np.float32)


def _tck_header(head, count):
    """The header lines of an input .tck with the count replaced and the data offset recomputed."""
    lines = [ln for ln in head.split('\n') if ln and not ln.startswith(('file:', 'count:'))]
    lines.insert(1 if lines else 0, 'count: %010d' % count)
    prefix = '\n'.join(lines) + '\n'
    offset = len(prefix) + len('file: . ') + len('\nEND\n')
    while True:
        text = prefix + 'file: . %d' % offset + '\nEND\n'
        if len(text) == offset:
            return text.encode()
        offset = len(text)


def filter_tractogram(in_path, out_path, oracle, threshold=0.5, reference_affine=None, save_scores=False):
    """Scores the streamlines of `in_path` and writes those with score >= threshold (compared in float32)
    to `out_path` (rank 0 only under torch.distributed).  Returns (keep mask, scores) as numpy arrays."""
    import torch.distributed as dist
    fmt = detect_format(in_path)
    if detect_format(out_path) != fmt:
        raise ValueError('input and output must have the same format (.trk or .tck)')
    if save_scores and fmt != 'trk':
        raise ValueError('.tck files cannot hold per-streamline data: --save_scores needs .trk')
    if fmt == 'tck' and reference_affine is None:
        raise ValueError('a .tck file needs a reference image to be moved to voxel space')
    data, offsets, hdr, (starts, ends) = (read_trk if fmt == 'trk' else read_tck)(in_path, spans=True)
    if save_scores and hdr['n_properties'] >= TRK_MAX_PROPERTIES:
        raise ValueError('%s already has %d per-streamline properties, the .trk maximum'
                         % (in_path, hdr['n_properties']))
    vox = voxel_points(data, fmt, hdr.get('voxel_sizes'), reference_affine)
    pts = torch.from_numpy(vox).to(oracle.device)
    off = torch.from_numpy(offsets).to(oracle.device)
    scores = oracle.predict_device(pts, off, distributed=True).cpu().numpy()
    keep = scores >= np.float32(threshold)
    if dist.is_initialized() and dist.get_rank() != 0:
        return keep, scores
    with open(in_path, 'rb') as f:
        raw = f.read()
    kept = np.nonzero(keep)[0]
    if fmt == 'trk':
        head = bytearray(raw[:1000])
        struct.pack_into('<i', head, 988, len(kept))
        if save_scores:
            n_prop = hdr['n_properties']
            struct.pack_into('<h', head, 238, n_prop + 1)
            head[240 + 20 * n_prop:260 + 20 * n_prop] = b'oracle_score'.ljust(20, b'\x00')
            body = b''.join(raw[starts[i]:ends[i]] + scores[i:i + 1].astype('<f4').tobytes() for i in kept)
        else:
            body = b''.join(raw[starts[i]:ends[i]] for i in kept)
        out = bytes(head) + body
    else:
        head = raw[:raw.index(b'END\n')].decode()
        out = (_tck_header(head, len(kept)) + b''.join(raw[starts[i]:ends[i]] for i in kept)
               + np.full((1, 3), np.inf, dtype='<f4').tobytes())
    with open(out_path, 'wb') as f:
        f.write(out)
    return keep, scores


def parse_args(argv=None):
    """ Keep the streamlines of a tractogram that TractOracle-Net scores at or above a threshold. """
    p = argparse.ArgumentParser(description=parse_args.__doc__, formatter_class=RawTextHelpFormatter)
    p.add_argument('in_tractogram', help='Input tractogram (.trk or .tck).')
    p.add_argument('out_tractogram', help='Output tractogram, same format as the input.')
    oracle_g = p.add_argument_group('Oracle filtering')
    oracle_g.add_argument('--oracle_checkpoint', required=True, metavar='CKPT', help='TractOracle-Net checkpoint.')
    oracle_g.add_argument('--reference', metavar='REF',
                          help='Reference image (.nii / .nii.gz) whose affine maps voxels to the\n'
                               'tractogram\'s RAS mm space.  Required for .tck.')
    oracle_g.add_argument('--threshold', type=float, default=0.5, metavar='T',
                          help='Keep streamlines whose score is >= T, in [0, 1]. [%(default)s]')
    oracle_g.add_argument('--precision', default='fp16', choices=['fp16', 'fp32'],
                          help='Oracle arithmetic.  fp16: tcgen05 tensor cores, the reference\'s autocast\n'
                               'arithmetic; fp32: CUDA cores. [%(default)s]')
    oracle_g.add_argument('--save_scores', action='store_true',
                          help='Append each kept streamline\'s score as the per-streamline\nproperty '
                               '"oracle_score" (.trk only).')
    p.add_argument('-f', dest='overwrite', action='store_true', help='Force overwriting of the output file.')
    args = p.parse_args(argv)
    try:
        fmt_in, fmt_out = detect_format(args.in_tractogram), detect_format(args.out_tractogram)
    except ValueError as e:
        p.error(str(e))
    if fmt_in != fmt_out:
        p.error('Input and output must have the same format (.trk or .tck); conversion is not supported')
    for f in (args.in_tractogram, args.oracle_checkpoint):
        if not os.path.isfile(f):
            p.error('Input file {} does not exist'.format(f))
    if os.path.isfile(args.out_tractogram) and not args.overwrite:
        p.error('Output file {} exists. Use -f to force overwriting'.format(args.out_tractogram))
    if not 0.0 <= args.threshold <= 1.0:
        p.error('--threshold must be in [0, 1], not %r' % args.threshold)
    if args.save_scores and fmt_in != 'trk':
        p.error('--save_scores needs .trk: .tck files cannot hold per-streamline data')
    if fmt_in == 'tck' and args.reference is None:
        p.error('--reference is required for .tck input')
    if args.reference is not None and not os.path.isfile(args.reference):
        p.error('Reference file {} does not exist'.format(args.reference))
    return args


def main(argv=None):
    args = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit('ttl_oracle_filter (tracktolearn_b200) needs a CUDA device; there is no CPU path')
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    device = torch.device('cuda')
    if world > 1:
        local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            dist.init_process_group('nccl', device_id=torch.device('cuda', local))
        device = torch.device('cuda', local)
    try:
        from tracktolearn_b200.oracles.oracle import OracleSingleton
        affine = None
        if args.reference is not None:
            from tracktolearn_b200.io import nifti
            affine = nifti.load(args.reference).affine
        OracleSingleton.clear()
        oracle = OracleSingleton(args.oracle_checkpoint, device, precision=args.precision)
        keep, _ = filter_tractogram(args.in_tractogram, args.out_tractogram, oracle, threshold=args.threshold,
                                    reference_affine=affine, save_scores=args.save_scores)
        if int(os.environ.get('RANK', '0')) == 0:
            print('Kept {} of {} streamlines in {}.'.format(int(keep.sum()), len(keep), args.out_tractogram))
        return int(keep.sum())
    finally:
        if world > 1 and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
