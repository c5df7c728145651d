"""Tractometry without a GPU: the restatement of tests/tractometry_oracle.py against scipy's order-1 interpolation
and the maps' in-grid rule, the fixed-point shift and order-free edge sums, the C ABI of ttl_sample_metrics and
ttl_connectome_sums and their argument checks, the kernels' stack frames, the metric volume checks, the argument
checks of ttl_track.py's Tractometry options, of ttl_connectivity.py and of ttl_tractometry.py, the mean_NAME
properties of a .trk file, and the world-2 gloo reduction of the int64 / int32 planes and gather of the means."""
import json
import math
import os
import re
import shutil
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy import ndimage

from tests import maps_oracle as M
from tests import tractometry_oracle as T
from tracktolearn_b200 import _lib, build, parallel
from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import TrkWriter, read_trk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def _pack(streamlines):
    lens = [len(s) for s in streamlines]
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = np.concatenate([np.asarray(s, dtype=F32).reshape(-1, 3) for s in streamlines]) if streamlines else \
        np.zeros((0, 3), F32)
    return data.astype(F32), offsets


# ------------------------------------------------------------------------------------ the restatement

def test_trilinear_is_scipy_order_one_inside_the_grid():
    rng = np.random.RandomState(0)
    dims = (7, 9, 6)
    vol = rng.randn(*dims, 3).astype(F32)
    inner = (rng.rand(4000, 3) * (np.asarray(dims) - 1)).astype(F32)
    faces = []                                        # on voxel faces and centres, and on the grid's last index
    for k in range(3):
        p = (rng.rand(300, 3) * (np.asarray(dims) - 1)).astype(F32)
        p[:, k] = rng.randint(0, dims[k] * 2 - 1, size=300) / F32(2.0)
        faces.append(p)
    pts = np.concatenate([inner] + faces + [np.asarray([[0, 0, 0], np.asarray(dims) - 1], F32)])
    got = T.trilinear(pts, vol)
    for c in range(3):
        want = ndimage.map_coordinates(vol[..., c].astype(np.float64), pts.T.astype(np.float64), order=1)
        np.testing.assert_allclose(got[:, c], want, rtol=1e-12, atol=1e-12)


def test_trilinear_replicates_the_edge_in_the_outer_half_voxel_rim():
    rng = np.random.RandomState(1)
    dims = (5, 4, 6)
    vol = rng.rand(*dims).astype(F32)
    pts = (rng.rand(3000, 3) * (np.asarray(dims) + 1) - 1.0).astype(F32)
    pts = pts[T.sampled(pts, dims)]                   # in [-0.5, n - 0.5): some in the rim on every side
    assert ((pts < 0) | (pts > np.asarray(dims) - 1)).any(axis=1).sum() > 300
    padded = np.pad(vol.astype(np.float64), 1, mode='edge')
    want = ndimage.map_coordinates(padded, pts.T.astype(np.float64) + 1.0, order=1)
    np.testing.assert_allclose(T.trilinear(pts, vol)[:, 0], want, rtol=1e-12, atol=1e-12)


def test_sampled_points_are_the_maps_in_grid_points():
    dims = (4, 3, 5)
    edge = [np.nan, np.inf, -np.inf, -0.5, -0.51, np.nextafter(F32(-0.5), F32(0)), 3.5, 3.49, 4.5, 0.0, 1e30,
            -1e30]
    vals = np.asarray(edge + [1.0, 2.2], dtype=F32)
    pts = np.stack(np.meshgrid(vals, vals, vals, indexing='ij'), -1).reshape(-1, 3)
    want = np.asarray([M.voxel_of(p, dims) is not None for p in pts])
    np.testing.assert_array_equal(T.sampled(pts, dims), want)
    offsets = np.asarray([0, 10, 10, len(pts)], np.int64)
    means, skipped = T.sample_means(pts, offsets, np.ones(dims, F32))
    assert skipped == M.tract_maps(pts, offsets, dims)[2] == int((~want).sum())
    assert np.isnan(means[1, 0])                      # empty
    assert means[2, 0] == 1.0


def _simple_means(data, offsets, vol):
    """Per streamline, lane by lane in a Python loop, then the tree: the order the kernel sums in."""
    out = []
    vol = vol[..., None] if vol.ndim == 3 else vol
    for i in range(len(offsets) - 1):
        s = data[offsets[i]:offsets[i + 1]]
        ok = T.sampled(s, vol.shape[:3])
        acc = np.zeros((1, 32, vol.shape[3]))
        for j in np.nonzero(ok)[0]:
            acc[0, j % 32] = acc[0, j % 32] + T.trilinear(s[j:j + 1], vol)[0]
        total = T._tree(acc)[0]
        out.append(np.full(vol.shape[3], np.nan, F32) if ok.sum() == 0 else (total / ok.sum()).astype(F32))
    return np.asarray(out).reshape(-1, vol.shape[3])


def _walks(rng, n, dims, lo, hi, junk=0.05):
    out = []
    for _ in range(n):
        L = int(rng.randint(lo, hi))
        s = np.cumsum(rng.randn(L, 3) * 0.8, axis=0) + rng.rand(3) * (np.asarray(dims) + 2) - 1
        if junk and L:
            hit = rng.rand(L) < junk
            s[hit, rng.randint(0, 3)] = rng.choice([np.nan, np.inf, -np.inf, -0.5, -0.51, dims[0] - 0.5, -3.0])
        out.append(s.astype(F32))
    return out


def test_vectorised_means_follow_the_lane_order_and_are_the_arithmetic_mean():
    rng = np.random.RandomState(2)
    dims = (9, 8, 7)
    vol = (rng.rand(*dims, 4) * 3 - 1).astype(F32)
    sl = _walks(rng, 150, dims, 0, 120) + [np.zeros((0, 3), F32)]
    data, offsets = _pack(sl)
    means, skipped = T.sample_means(data, offsets, vol, chunk=37)
    np.testing.assert_array_equal(means, _simple_means(data, offsets, vol))
    assert skipped == M.tract_maps_fast(data, offsets, dims)[2]
    for i, s in enumerate(sl):
        ok = T.sampled(s, dims)
        if ok.any():
            np.testing.assert_allclose(means[i], T.trilinear(s[ok], vol).mean(0), rtol=1e-6)
        else:
            assert np.isnan(means[i]).all()


# ------------------------------------------------------------------------------------ fixed point

def test_metric_shift_keeps_every_value_within_2_to_the_31():
    from tracktolearn_b200.tracking.postprocess import metric_shift
    bounds = [0.0, 5e-324, 1e-30, 0.7, 1.0, 3.0, 2.0 ** 30, 2.0 ** 31 - 1, 2.0 ** 31 - 2 ** -22]
    for k in range(-70, 31):
        bounds += [2.0 ** k, np.nextafter(2.0 ** k, 0.0)]
    for b in bounds:
        S = metric_shift(b)
        assert S == T.metric_shift(b) and 0 <= S <= 62
        assert abs(np.rint(np.ldexp(b, S))) <= 2.0 ** 31, (b, S)
        if 0 < S < 62:
            assert np.ldexp(b, S + 1) >= 2.0 ** 31 or b == 0.0, (b, S)    # the largest shift that fits
    assert metric_shift(0.0) == 31
    for bad in (2.0 ** 31, 1e300, math.inf, math.nan, -1.0):
        with pytest.raises(ValueError):
            metric_shift(bad)


def test_fixed_point_edge_sums_do_not_depend_on_order_or_batches():
    from tracktolearn_b200.tracking.postprocess import edge_means
    rng = np.random.RandomState(3)
    n, K = 5000, 13
    pairs = rng.randint(-2, K + 3, size=(n, 2)).astype(np.int32)
    values = np.stack([(rng.rand(n) * 0.9).astype(F32), (rng.randn(n) * 300).astype(F32)], 1)
    values[rng.rand(n) < 0.05, 0] = np.nan
    values[:3, 1] = [np.inf, -np.inf, np.nan]
    shifts = [T.metric_shift(0.9), T.metric_shift(np.abs(values[3:, 1]).max())]
    whole = T.edge_sums(pairs, values, shifts, K)
    perm = rng.permutation(n)
    shuffled = T.edge_sums(pairs[perm], values[perm], shifts, K)
    parts = [T.edge_sums(pairs[c], values[c], shifts, K) for c in np.array_split(perm, 7)]
    for got in (shuffled, (sum(p[0] for p in parts), sum(p[1] for p in parts))):
        assert got[0].tobytes() == whole[0].tobytes() and got[1].tobytes() == whole[1].tobytes()
    mean = edge_means(*whole, shifts)
    a, b = (np.where((pairs[:, k] > 0) & (pairs[:, k] < K), pairs[:, k], 0) for k in range(2))
    for c in range(2):
        want = np.full((K, K), np.nan)
        for x in range(K):
            for y in range(K):
                sel = ((a == x) & (b == y)) | ((a == y) & (b == x))
                v = values[sel, c].astype(np.float64)
                v = v[np.isfinite(v)]
                if len(v):
                    want[x, y] = v.mean()
        np.testing.assert_allclose(mean[c], want, rtol=1e-7, atol=2.0 ** -shifts[c])
        assert np.array_equal(np.isnan(mean[c]), whole[1][c] == 0)


# ------------------------------------------------------------------------------------ C ABI

_ARGS_PROBE = r'''
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from tracktolearn_b200 import _lib
lib = _lib.load()
fake = iter(range(1 << 20, 1 << 30, 1 << 16))          # distinct aligned addresses, never dereferenced
pts, off, vol, means, skipped, pairs, vals, sums, counts = (ctypes.c_void_p(next(fake)) for _ in range(9))


def sample(n=10, C=3, dims=(4, 5, 6), points=pts, offsets=off, volumes=vol, out=means, sk=skipped):
    return lib.ttl_sample_metrics(points, offsets, n, volumes, C, *dims, out, sk, None)


def shifts_of(*s):
    return (ctypes.c_int32 * len(s))(*s)


good = shifts_of(0, 31, 62, 5, 5, 5, 5, 5, 5)


def esums(n=10, C=3, K=7, shifts=good, p=pairs, v=vals, s=sums, c=counts):
    return lib.ttl_connectome_sums(p, n, v, C, K, shifts, s, c, None)


bad = {
    'n < 0': sample(n=-1), 'C = 0': sample(C=0), 'C = 9': sample(C=9), 'C < 0': sample(C=-1),
    'zero x': sample(dims=(0, 5, 6)), 'zero y': sample(dims=(4, 0, 6)), 'zero z': sample(dims=(4, 5, 0)),
    'negative dim': sample(dims=(4, -5, 6)),
    'grid * C = 2^31': sample(C=2, dims=(1 << 10, 1 << 10, 1 << 10)),
    'grid * C above 2^31': sample(C=8, dims=(1 << 9, 1 << 9, 1 << 10)),
    'no volumes': sample(volumes=None), 'no means': sample(out=None), 'no skipped': sample(sk=None),
    'no volumes, n = 0': sample(n=0, volumes=None),
    'no points': sample(points=None), 'no offsets': sample(offsets=None),
    'sums n < 0': esums(n=-1), 'sums C = 0': esums(C=0), 'sums C = 10': esums(C=10), 'sums K = 0': esums(K=0),
    'sums K = 16385': esums(K=16385), 'no shifts': esums(shifts=None), 'shift < 0': esums(shifts=shifts_of(0, -1, 0)),
    'shift 63': esums(shifts=shifts_of(0, 63, 0)), 'no sums': esums(s=None), 'no counts': esums(c=None),
    'no sums, n = 0': esums(n=0, s=None), 'no pairs': esums(p=None), 'no values': esums(v=None),
}
ok = {'n = 0': sample(n=0), 'n = 0 without points': sample(n=0, points=None, offsets=None),
      'sums n = 0': esums(n=0), 'sums n = 0 without inputs': esums(n=0, p=None, v=None)}
accepted = [sample(), sample(C=1), sample(C=8), sample(C=1, dims=(1 << 11, 1 << 10, (1 << 10) - 1)),
            esums(), esums(C=9), esums(K=1), esums(K=16384)]
print(json.dumps({'bad': bad, 'ok': ok, 'accepted': accepted}))
'''


def test_exports_are_bound_and_reject_bad_arguments():
    """Every bad argument is refused with TTL_ERR_BAD_ARG before any CUDA call.  No device is visible to the
    probe: an accepted call gets past every check and fails at its launch instead of running on the fake
    pointers."""
    build.build()
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'ttl_b200.h')).read()
    for name in ('ttl_sample_metrics', 'ttl_connectome_sums'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
        assert re.search(r'\b%s\(' % name, header)
    assert lib.ttl_abi_version() == _lib.ABI_VERSION == 5
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, '-c', _ARGS_PROBE, ROOT], env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT)
    assert out.returncode == 0, out.stdout.decode()
    res = json.loads(out.stdout.decode().strip().splitlines()[-1])
    assert len(res['bad']) == 29 and all(c == -1 for c in res['bad'].values()), res['bad']
    assert all(c == 0 for c in res['ok'].values()), res['ok']
    assert all(c > 0 for c in res['accepted']), res['accepted']


def test_tractometry_kernels_have_no_stack_frame():
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    build.build()
    out = subprocess.run([tool, '-res-usage', _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()
    found = re.findall(r'Function (\S*(?:sample_metrics_kernel|connectome_sums_kernel)\S*):\s*\n\s*REG:(\d+) '
                       r'STACK:(\d+).*LOCAL:(\d+)', out)
    assert len(found) == 9, found                    # C = 1..8 and the sums
    for name, reg, stack, local in found:
        assert int(stack) == 0 and int(local) == 0, name


# ------------------------------------------------------------------------------------ metric volumes

AFFINE = np.array([[1.25, 0, 0, -5.0], [0, 1.25, 0, 3.0], [0, 0, 1.25, 1.0], [0, 0, 0, 1]])
DIMS = (6, 7, 5)


def _nii(tmp_path, data, name, affine=AFFINE):
    path = str(tmp_path / name)
    nifti.save(path, data, affine)
    return path


@pytest.mark.parametrize('dtype', [np.uint8, np.int16, np.int32, np.float32, np.float64])
def test_load_metrics_accepts_numeric_volumes(tmp_path, dtype):
    from tracktolearn_b200.runners.ttl_connectivity import load_metrics
    rng = np.random.RandomState(4)
    a = (rng.rand(*DIMS) * 100).astype(dtype)
    b = -(rng.rand(*DIMS) * 7).astype(np.float32)
    vol, names, bounds = load_metrics([('FA', _nii(tmp_path, a, 'a.nii.gz')), ('md_1', _nii(tmp_path, b, 'b.nii'))],
                                      DIMS, AFFINE + 3e-5, device='cpu')
    assert vol.dtype == torch.float32 and tuple(vol.shape) == DIMS + (2,) and vol.is_contiguous()
    np.testing.assert_array_equal(vol[..., 0].numpy(), a.astype(F32))
    np.testing.assert_array_equal(vol[..., 1].numpy(), b)
    assert names == ['FA', 'md_1'] and bounds == [float(np.abs(a.astype(F32)).max()), float(np.abs(b).max())]


def test_load_metrics_refuses_what_is_not_a_metric_of_the_grid(tmp_path):
    from tracktolearn_b200.runners.ttl_connectivity import load_metrics
    good = _nii(tmp_path, np.ones(DIMS, F32), 'good.nii')
    nan = np.ones(DIMS, F32)
    nan[1, 1, 1] = np.nan
    inf = np.ones(DIMS, np.float64)
    inf[0, 0, 0] = 1e300                              # finite in float64, inf in float32
    huge = np.ones(DIMS, F32)
    huge[0, 0, 0] = 2.0 ** 31
    shifted = AFFINE.copy()
    shifted[1, 3] += 2e-4
    cases = [[('FA', _nii(tmp_path, nan, 'nan.nii'))], [('FA', _nii(tmp_path, inf, 'inf.nii'))],
             [('FA', _nii(tmp_path, huge, 'huge.nii'))],
             [('FA', _nii(tmp_path, np.ones((6, 7, 4), F32), 'shape.nii'))],
             [('FA', _nii(tmp_path, np.ones(DIMS + (2,), F32), '4d.nii'))],
             [('FA', _nii(tmp_path, np.ones(DIMS, F32), 'aff.nii', shifted))],
             [('FA', str(tmp_path / 'missing.nii'))], [('FA', good), ('FA', good)], [('1FA', good)],
             [('fa-x', good)], [('a' * 15, good)], [('', good)], [('m%d' % i, good) for i in range(9)], []]
    for metrics in cases:
        with pytest.raises(ValueError):
            load_metrics(metrics, DIMS, AFFINE, device='cpu')
    load_metrics([('a' * 14, good)] + [('m%d' % i, good) for i in range(7)], DIMS, AFFINE, device='cpu')


# ------------------------------------------------------------------------------------ command lines

def _touch(path):
    open(path, 'wb').close()
    return str(path)


def _track_argv(tmp_path, out, *extra):
    ins = [_touch(tmp_path / n) for n in ('fodf.nii.gz', 'seed.nii.gz', 'mask.nii.gz')]
    return ins + [str(tmp_path / out), '--agent', str(tmp_path), '--hyperparameters', _touch(tmp_path / 'hp.json')] \
        + list(extra)


def test_ttl_track_tractometry_options(tmp_path):
    from tracktolearn_b200.runners.ttl_track import parse_args
    args = parse_args(_track_argv(tmp_path, 'out.trk'))
    assert args.in_metric is None and not args.save_metric_means
    assert args.out_connectivity_metrics is None and args.out_connectivity_length is None
    fa, md, lab = (_touch(tmp_path / n) for n in ('fa.nii.gz', 'md.nii.gz', 'aparc.nii.gz'))
    pre = str(tmp_path / 'conn_')
    args = parse_args(_track_argv(tmp_path, 'out.trk', '--in_metric', 'FA', fa, '--in_metric', 'MD', md,
                                  '--save_metric_means', '--in_labels', lab, '--out_connectivity_metrics', pre,
                                  '--out_connectivity_length', str(tmp_path / 'len.npy')))
    assert args.in_metric == [['FA', fa], ['MD', md]] and args.save_metric_means
    parse_args(_track_argv(tmp_path, 'out.tck', '--in_labels', lab, '--out_connectivity_length',
                           str(tmp_path / 'len.npy')))
    parse_args(_track_argv(tmp_path, 'out.tck', '--in_metric', 'FA', fa, '--in_labels', lab,
                           '--out_connectivity_metrics', pre))
    ten = ['--in_metric', 'FA', fa, '--in_metric', 'MD', md, '--in_metric', 'RD', md, '--in_metric', 'AD', md,
           '--in_metric', 'FW', md, '--save_metric_means', '--save_seeds', '--save_connectivity_labels', '--in_labels', lab]
    parse_args(_track_argv(tmp_path, 'out.trk', *ten))                      # 5 + 3 + 2 = 10 properties
    _touch(tmp_path / 'conn_FA.npy')
    parse_args(_track_argv(tmp_path, 'out.trk', '--in_metric', 'FA', fa, '--in_labels', lab,
                           '--out_connectivity_metrics', pre, '-f'))
    eight = [a for i in range(8) for a in ('--in_metric', 'm%d' % i, fa)]
    bad = [('--in_metric', 'FA', fa),                                                       # no output
           ('--save_metric_means',), ('--in_labels', lab, '--out_connectivity_metrics', pre),  # no metric
           ('--in_metric', 'FA', fa, '--out_connectivity_metrics', pre),                   # no labels
           ('--out_connectivity_length', str(tmp_path / 'len.npy')),                       # no labels
           ('--in_metric', 'FA', str(tmp_path / 'missing.nii'), '--save_metric_means'),
           ('--in_metric', '2FA', fa, '--save_metric_means'), ('--in_metric', 'F-A', fa, '--save_metric_means'),
           ('--in_metric', 'abcdefghijklmno', fa, '--save_metric_means'),
           ('--in_metric', 'FA', fa, '--in_metric', 'FA', md, '--save_metric_means'),
           tuple(eight) + ('--in_metric', 'm8', fa, '--save_metric_means'),                 # 9 metrics
           tuple(ten) + ('--save_oracle_scores', '--oracle_checkpoint', fa),               # 11 properties
           tuple(ten) + ('--in_metric', 'XX', fa),                                         # 11 properties
           ('--in_metric', 'FA', fa, '--in_labels', lab, '--out_connectivity_metrics', pre),  # exists, no -f
           ('--in_labels', lab, '--out_connectivity_length', str(tmp_path / 'len.csv')),   # not .npy
           ('--in_labels', lab, '--out_connectivity_length', str(tmp_path / 'c.npy'), '--out_connectivity',
            str(tmp_path / 'c.npy')),                                                      # collide
           ('--in_metric', 'FA', fa, '--in_labels', lab, '--out_connectivity_metrics', str(tmp_path / 'x'),
            '--out_connectivity_length', str(tmp_path / 'xFA.npy'))]                       # collide
    for extra in bad:
        with pytest.raises(SystemExit):
            parse_args(_track_argv(tmp_path, 'out.trk', *extra))
    with pytest.raises(SystemExit):                                                         # .tck holds no means
        parse_args(_track_argv(tmp_path, 'out.tck', '--in_metric', 'FA', fa, '--save_metric_means'))


def _trk(tmp_path, name, dims, zooms):
    path = str(tmp_path / name)
    w = TrkWriter(path, dims, zooms, np.eye(4))
    w.write(np.zeros((2, 3), F32), np.array([0, 2], np.int64))
    w.close()
    return path


def test_ttl_connectivity_metric_options(tmp_path):
    from tracktolearn_b200.runners.ttl_connectivity import parse_args
    lab = _nii(tmp_path, np.arange(np.prod(DIMS)).reshape(DIMS) % 5, 'lab.nii.gz')
    fa = _nii(tmp_path, np.random.RandomState(5).rand(*DIMS).astype(F32), 'fa.nii.gz')
    trk = _trk(tmp_path, 'in.trk', DIMS, (1.25, 1.25, 1.25))
    out = str(tmp_path / 'c.npy')
    args = parse_args([trk, lab, out, '--in_metric', 'FA', fa, '--out_metrics', str(tmp_path / 'w_'),
                       '--out_length', str(tmp_path / 'len.npy')])
    vol, names, bounds = args.metrics
    assert names == ['FA'] and tuple(vol.shape) == DIMS + (1,)
    assert parse_args([trk, lab, out]).metrics is None
    other = _nii(tmp_path, np.ones((6, 7, 6), F32), 'other.nii')
    _touch(tmp_path / 'w_FA.npy')
    bad = [[trk, lab, out, '--in_metric', 'FA', fa],                                         # no --out_metrics
           [trk, lab, out, '--out_metrics', str(tmp_path / 'v_')],                          # no --in_metric
           [trk, lab, out, '--in_metric', 'FA', other, '--out_metrics', str(tmp_path / 'v_')],   # off the grid
           [trk, lab, out, '--in_metric', 'FA', fa, '--out_metrics', str(tmp_path / 'w_')],  # exists, no -f
           [trk, lab, out, '--in_metric', 'F A', fa, '--out_metrics', str(tmp_path / 'v_')],
           [trk, lab, out, '--out_length', str(tmp_path / 'len.txt')],
           [trk, lab, out, '--out_length', out],                                            # collides
           [trk, lab, out, '--out_length', lab, '-f'],
           [trk, lab, out, '--in_metric', 'FA', str(tmp_path / 'missing.nii'), '--out_metrics', str(tmp_path / 'v')]]
    for argv in bad:
        with pytest.raises(SystemExit):
            parse_args(argv)


def test_ttl_tractometry_options(tmp_path):
    from tracktolearn_b200.runners.ttl_tractometry import parse_args
    fa = _nii(tmp_path, np.random.RandomState(6).rand(*DIMS).astype(F32), 'fa.nii.gz')
    md = _nii(tmp_path, np.random.RandomState(7).rand(*DIMS).astype(np.float64), 'md.nii')
    trk = _trk(tmp_path, 'in.trk', DIMS, (1.25, 1.25, 1.25))
    tck = _touch(tmp_path / 'in.tck')
    out = str(tmp_path / 'm.npy')
    args = parse_args([trk, out, '--in_metric', 'FA', fa, '--in_metric', 'MD', md])
    assert args.metrics[1] == ['FA', 'MD'] and np.allclose(args.affine, AFFINE)
    parse_args([tck, out, '--in_metric', 'FA', fa])
    _touch(tmp_path / 'm.npy')
    parse_args([trk, out, '--in_metric', 'FA', fa, '-f'])
    other = _nii(tmp_path, np.ones(DIMS, F32), 'other.nii', np.diag([1.25, 1.25, 1.5, 1]))
    bad = [[trk, out, '--in_metric', 'FA', fa],                                             # exists
           [trk, str(tmp_path / 'x.npy')],                                                  # no metric
           [trk, str(tmp_path / 'x.txt'), '--in_metric', 'FA', fa],
           [trk, fa, '--in_metric', 'FA', fa, '-f'],
           [trk, str(tmp_path / 'x.npy'), '--in_metric', 'FA', fa, '--in_metric', 'FA', md],
           [trk, str(tmp_path / 'x.npy'), '--in_metric', 'FA', fa, '--in_metric', 'B', other],
           [trk, str(tmp_path / 'x.npy'), '--in_metric', '_FA', fa],
           [str(tmp_path / 'in.vtk'), str(tmp_path / 'x.npy'), '--in_metric', 'FA', fa],
           [str(tmp_path / 'missing.trk'), str(tmp_path / 'x.npy'), '--in_metric', 'FA', fa],
           [_trk(tmp_path, 'dims.trk', (6, 7, 6), (1.25, 1.25, 1.25)), str(tmp_path / 'x.npy'), '--in_metric', 'FA', fa],
           [_trk(tmp_path, 'vox.trk', DIMS, (1.25, 1.5, 1.25)), str(tmp_path / 'x.npy'), '--in_metric', 'FA', fa]]
    for argv in bad:
        with pytest.raises(SystemExit):
            parse_args(argv)


def test_help_lists_the_tractometry_options():
    for script, flags in (('ttl_track.py', ('Tractometry', '--in_metric', '--save_metric_means',
                                            '--out_connectivity_metrics', '--out_connectivity_length')),
                          ('ttl_connectivity.py', ('--in_metric', '--out_metrics', '--out_length')),
                          ('ttl_tractometry.py', ('in_tractogram', 'out_means', '--in_metric'))):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', script), '--help'],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        for flag in flags:
            assert flag in out.stdout, (script, flag)


# ------------------------------------------------------------------------------------ .trk properties

@pytest.mark.parametrize('save_seeds', [False, True])
@pytest.mark.parametrize('save_scores', [False, True])
@pytest.mark.parametrize('save_labels', [False, True])
def test_trk_metric_means_round_trip(tmp_path, save_seeds, save_scores, save_labels):
    rng = np.random.RandomState(8)
    names = ['FA', 'MD', 'a' * 14][:10 - 3 * save_seeds - save_scores - 2 * save_labels]
    path = str(tmp_path / 'a.trk')
    w = TrkWriter(path, (10, 11, 12), (1.25, 1.25, 1.25), np.eye(4), save_seeds=save_seeds, save_scores=save_scores,
                  save_labels=save_labels, metric_names=names)
    batches = []
    for n in (9, 0, 25):
        lens = rng.randint(1, 30, size=n)
        offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
        data = rng.randn(int(offsets[-1]), 3).astype(F32)
        seeds, scores = rng.randn(n, 3), rng.rand(n).astype(F32)
        labels = rng.randint(0, 16384, size=(n, 2)).astype(np.int32)
        means = rng.randn(n, len(names)).astype(F32)
        means[:2, 0] = np.nan
        w.write(data, offsets, seeds if save_seeds else None, scores if save_scores else None,
                labels if save_labels else None, means)
        batches.append((data, offsets, seeds, scores, labels, means))
    w.close()
    data, offsets, hdr = read_trk(path)
    want = ['seeds_x', 'seeds_y', 'seeds_z'] * save_seeds + ['oracle_score'] * save_scores + \
        ['start_label', 'end_label'] * save_labels + ['mean_' + m for m in names]
    assert hdr['property_names'] == want and hdr['n_count'] == 34
    np.testing.assert_array_equal(data, np.concatenate([b[0] for b in batches]))
    props = hdr['properties']
    C = len(names)
    np.testing.assert_array_equal(props[:, -C:], np.concatenate([b[5] for b in batches]))
    if save_labels:
        np.testing.assert_array_equal(props[:, -C - 2:-C].astype(np.int32), np.concatenate([b[4] for b in batches]))
    if save_scores:
        np.testing.assert_array_equal(props[:, -C - 1 - 2 * save_labels], np.concatenate([b[3] for b in batches]))
    if save_seeds:
        np.testing.assert_array_equal(props[:, :3], np.concatenate([b[2] for b in batches]).astype(F32))


def test_trk_bytes_unchanged_without_metrics_and_at_most_ten_properties(tmp_path):
    rng = np.random.RandomState(9)
    lens = rng.randint(1, 30, size=12)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = rng.randn(int(offsets[-1]), 3).astype(F32)
    seeds, scores, labels = rng.randn(12, 3), rng.rand(12), rng.randint(0, 9, size=(12, 2))
    outs = []
    for kw in ({}, {'metric_names': ()}):
        path = str(tmp_path / ('%d.trk' % len(outs)))
        w = TrkWriter(path, (10, 11, 12), (2.0, 2.0, 2.0), np.eye(4), True, save_scores=True, save_labels=True, **kw)
        w.write(data, offsets, seeds, scores, labels)
        w.close()
        outs.append(open(path, 'rb').read())
    assert outs[0] == outs[1]
    with pytest.raises(ValueError):
        TrkWriter(str(tmp_path / 'x.trk'), (1, 1, 1), (1, 1, 1), np.eye(4), True, save_scores=True, save_labels=True,
                  metric_names=['a', 'b', 'c', 'd', 'e'])
    assert not os.path.exists(str(tmp_path / 'x.trk'))


# ------------------------------------------------------------------------------------ ranks

def _rank_part(rank):
    rng = np.random.RandomState(40 + rank)
    n, K = 30 + 11 * rank, 6
    pairs = rng.randint(0, K, size=(n, 2)).astype(np.int32)
    values = rng.randn(n, 3).astype(F32)
    values[::7, 1] = np.nan
    data, offsets = _pack(_walks(rng, n, (5, 5, 5), 1, 20))
    return pairs, values, data, offsets


SHIFTS = [29, 29, 29]


def _worker(rank, world, port, via, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    pairs, values, data, offsets = _rank_part(rank)
    sums, counts = (torch.from_numpy(x) for x in T.edge_sums(pairs, values, SHIFTS, 6))
    unsampled = torch.tensor([rank + 1], dtype=torch.int64)
    total = parallel.reduce_maps([None, sums, counts, unsampled], 3 + rank)
    n = len(offsets) - 1
    merged = parallel.gather_packed(torch.from_numpy(data), torch.from_numpy(np.diff(offsets)),
                                    torch.zeros((n, 3), dtype=torch.float64), torch.zeros((n,), dtype=torch.int64),
                                    via=via, labels=torch.from_numpy(pairs), means=torch.from_numpy(values))
    if rank == 0:
        q.put((sums.numpy().copy(), counts.numpy().copy(), int(unsampled), total, dict(merged.data_per_streamline)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('via', ['nccl', 'host'])
def test_two_rank_reduce_sums_the_planes_and_gather_carries_the_means(via):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, via, q)) for r in range(2)]
    for p in procs:
        p.start()
    sums, counts, unsampled, total, per = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    parts = [_rank_part(r) for r in range(2)]
    pairs = np.concatenate([p[0] for p in parts])
    values = np.concatenate([p[1] for p in parts])
    want = T.edge_sums(pairs, values, SHIFTS, 6)
    assert sums.dtype == np.int64 and sums.tobytes() == want[0].tobytes()
    assert counts.dtype == np.int32 and counts.tobytes() == want[1].tobytes()
    assert unsampled == 3 and total == 7
    assert per['metric_means'].dtype == np.float32 and per['metric_means'].shape == values.shape
    assert per['metric_means'].tobytes() == values.tobytes()
    np.testing.assert_array_equal(np.stack((per['start_label'], per['end_label']), 1), pairs)
