"""Connectivity matrix without a GPU: the restatement of tests/connectome_oracle.py on hand-made cases and against
dipy's end-voxel rule, the C ABI of ttl_connectome and its argument checks, the kernel's stack frame, the label
volume checks, the argument checks of ttl_track.py's Connectivity options and of ttl_connectivity.py, the world-2
gloo reduction of per-rank matrices and gather of per-streamline labels, and the start_label / end_label
properties of a .trk file."""
import json
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

from tests import connectome_oracle as C
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


def _both(data, offsets, labels, r, K=None):
    """The loop and the vectorised restatement, asserted equal."""
    want = C.connectome(data, offsets, labels, r, K)
    got = C.connectome_fast(data, offsets, labels, r, K)
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1], want[1])
    return want


# ------------------------------------------------------------------------------------ the rule, by hand

def test_own_voxel_wins_over_a_nearer_looking_neighbour():
    lab = np.zeros((4, 4, 4), np.int32)
    lab[1, 1, 1] = 3
    lab[2, 1, 1] = 5
    p = (F32(1.49), F32(1.0), F32(1.0))              # own voxel (1,1,1); (2,1,1) is 0.51 away
    assert C.end_label(p, lab, 4.0) == 3
    lab[1, 1, 1] = 0                                  # unlabelled own voxel: the search finds (2,1,1)
    assert C.end_label(p, lab, 0.51) == 5
    assert C.end_label(p, lab, 0.5) == 0              # 0.51 away, r = 0.5: nothing
    assert C.end_label(p, lab, 0.0) == 0


def test_exact_distance_tie_goes_to_the_lower_linear_index():
    lab = np.zeros((5, 5, 5), np.int32)
    lab[1, 2, 2] = 7                                  # linear index (1*5+2)*5+2 = 37
    lab[3, 2, 2] = 4                                  # 87, at the same distance 1 from (2,2,2)
    assert C.end_label((2, 2, 2), lab, 1.0) == 7
    lab[2, 2, 1] = 9                                  # 61 < 87 but > 37
    assert C.end_label((2, 2, 2), lab, 1.0) == 7
    lab[2, 1, 2] = 2                                  # 57
    assert C.end_label((2, 2, 2), lab, 1.0) == 7
    lab[1, 2, 2] = 0
    assert C.end_label((2, 2, 2), lab, 1.0) == 2
    lab[2, 2, 3] = 6                                  # 63 at the same distance: 57 still wins
    assert C.end_label((2, 2, 2), lab, 1.0) == 2
    lab[2, 2, 2] = 0
    lab[2, 3, 3] = 1                                  # sqrt(2) away: farther, loses whatever its index
    assert C.end_label((2, 2, 2), lab, 1.5) == 2


def test_voxel_at_exactly_the_radius_is_included():
    lab = np.zeros((8, 3, 3), np.int32)
    lab[5, 1, 1] = 11
    p = (F32(2.0), F32(1.0), F32(1.0))               # d2 = 9.0 exactly
    assert C.end_label(p, lab, 3.0) == 11
    assert C.end_label(p, lab, np.nextafter(3.0, 0.0)) == 0
    lab[5, 1, 1], lab[4, 2, 2] = 0, 12                # d2 = 4 + 1 + 1 = 6, compared with r*r as rounded
    r = np.sqrt(6.0)
    assert C.end_label(p, lab, r) == (12 if 6.0 <= r * r else 0)
    assert C.end_label(p, lab, np.nextafter(r, 3.0)) == 12


@pytest.mark.parametrize('bad', [np.nan, np.inf, -np.inf])
def test_non_finite_endpoints_get_label_zero(bad):
    lab = np.ones((3, 3, 3), np.int32)
    for axis in range(3):
        p = [F32(1.0)] * 3
        p[axis] = F32(bad)
        assert C.end_label(p, lab, 8.0) == 0
    data, offsets = _pack([[(1, 1, 1), (F32(bad), 1, 1)]])
    m, pairs = _both(data, offsets, lab, 8.0)
    assert pairs.tolist() == [[1, 0]] and m[0, 1] == m[1, 0] == 1 and m.sum() == 2


def test_off_grid_endpoint_whose_box_reaches_the_grid():
    lab = np.zeros((4, 5, 6), np.int32)
    lab[0, 2, 3] = 8
    assert C.end_label((F32(-1.7), F32(2.0), F32(3.0)), lab, 2.0) == 8          # 1.7 away
    assert C.end_label((F32(-1.7), F32(2.0), F32(3.0)), lab, 1.6) == 0
    lab[3, 4, 5] = 2
    assert C.end_label((F32(4.5), F32(5.5), F32(6.5)), lab, 2.0) == 0           # sqrt(3 * 1.5^2) = 2.6 > 2
    assert C.end_label((F32(4.5), F32(5.5), F32(6.5)), lab, 2.6) == 2
    assert C.end_label((F32(3.9), F32(4.9), F32(5.9)), lab, 0.0) == 0           # own voxel off the grid
    assert C.end_label((F32(1e30), F32(0), F32(0)), lab, 8.0) == 0
    assert C.end_label((F32(-1e30), F32(0), F32(0)), lab, 8.0) == 0


def test_one_point_streamline_both_ends_share_a_label_and_unlabelled_ends_go_to_zero_zero():
    lab = np.zeros((3, 3, 3), np.int32)
    lab[1, 1, 1] = 4
    data, offsets = _pack([[(1, 1, 1)], [(0, 0, 0), (0, 0, 2)], [], [(1, 1, 1), (2.2, 2, 2)]])
    m, pairs = _both(data, offsets, lab, 0.0)
    assert pairs.tolist() == [[4, 4], [0, 0], [0, 0], [4, 0]]
    assert m[4, 4] == 1 and m[0, 0] == 1 and m[0, 4] == m[4, 0] == 1 and m.sum() == 4
    assert m.shape == (5, 5)


def _random_set(rng, n, dims, junk=True, lo=0, hi=40):
    sl = []
    for _ in range(n):
        L = int(rng.randint(lo, hi))
        s = np.cumsum(rng.randn(L, 3) * 0.8, axis=0) + rng.rand(3) * (np.asarray(dims) + 2) - 1
        if junk and L:
            hit = rng.rand(L) < 0.05
            s[hit, rng.randint(0, 3)] = rng.choice([np.nan, np.inf, -np.inf, -0.5, dims[0] - 0.5, -3.0])
        sl.append(s.astype(F32))
    return sl


def _parcellation(rng, dims, n_labels, density):
    lab = rng.randint(1, n_labels + 1, size=dims).astype(np.int32)
    lab[rng.rand(*dims) >= density] = 0
    return lab


@pytest.mark.parametrize('r', [0.0, 0.5, 1.0, 2.5, 8.0])
def test_loop_and_vectorised_restatements_agree_and_keep_the_triangle_invariant(r):
    rng = np.random.RandomState(int(r * 10))
    dims = (9, 7, 8)
    lab = _parcellation(rng, dims, 6, 0.15)
    sl = _random_set(rng, 250, dims)
    data, offsets = _pack(sl)
    m, pairs = _both(data, offsets, lab, r)
    n_nonempty = sum(len(s) > 0 for s in sl)
    assert int(np.triu(m).sum()) == n_nonempty
    np.testing.assert_array_equal(m, m.T)
    assert C.end_labels_fast(np.zeros((0, 3), F32), lab, r).shape == (0,)


def _dipy_connectivity(streamlines, labels):
    """dipy.tracking.utils.connectivity_matrix(streamlines, eye, labels, symmetric=True) for streamlines of 2+
    points whose ends lie in the grid: end voxels int(p + 0.5), the sorted end-label pairs counted with a
    bincount, then np.maximum(M, M.T)."""
    mx = int(labels.max()) + 1
    ends = np.asarray([[s[0], s[-1]] for s in streamlines], dtype=F32).astype(np.float64)
    i, j, k = (ends + 0.5).astype(int).transpose(2, 1, 0)
    endlabels = labels[i, j, k]
    endlabels.sort(0)
    m = np.bincount(endlabels[0] * mx + endlabels[1], minlength=mx * mx).reshape(mx, mx)
    return np.maximum(m, m.T)


def test_radius_zero_is_dipys_end_voxel_rule():
    rng = np.random.RandomState(7)
    dims = (10, 9, 11)
    lab = _parcellation(rng, dims, 9, 0.6)
    sl = _random_set(rng, 600, dims, junk=False, lo=2)
    inside = [s for s in sl if all(np.all((np.floor(p.astype(np.float64) + 0.5) >= 0)
                                          & (np.floor(p.astype(np.float64) + 0.5) < dims)) for p in (s[0], s[-1]))]
    assert len(inside) > 100
    m, _ = _both(*_pack(inside), lab, 0.0)
    np.testing.assert_array_equal(m, _dipy_connectivity(inside, lab))


def test_label_values_outside_the_matrix_read_as_zero():
    lab = np.zeros((3, 3, 3), np.int32)
    lab[0, 0, 0], lab[2, 2, 2], lab[1, 1, 1] = 3, 9, -4
    data, offsets = _pack([[(0, 0, 0), (2, 2, 2)], [(1, 1, 1), (0, 0, 0)]])
    m, pairs = _both(data, offsets, lab, 0.0, K=4)
    assert pairs.tolist() == [[3, 0], [0, 3]] and m[0, 3] == m[3, 0] == 2 and m.shape == (4, 4)


# ------------------------------------------------------------------------------------ C ABI

_ARGS_PROBE = r'''
import ctypes, json, math, sys
sys.path.insert(0, sys.argv[1])
from tracktolearn_b200 import _lib
lib = _lib.load()
fake = iter(range(1 << 20, 1 << 30, 1 << 16))          # distinct aligned addresses, never dereferenced
pts, off, lab, mat, pairs = (ctypes.c_void_p(next(fake)) for _ in range(5))


def call(n=10, labels=lab, dims=(4, 5, 6), K=7, r=2.0, matrix=mat, pairs=pairs, points=pts, offsets=off):
    return lib.ttl_connectome(points, offsets, n, labels, *dims, K, r, matrix, pairs, None)


codes = {
    'n < 0': call(n=-1),
    'zero x': call(dims=(0, 5, 6)), 'zero y': call(dims=(4, 0, 6)), 'zero z': call(dims=(4, 5, 0)),
    'negative dim': call(dims=(4, -5, 6)),
    'grid of 2^31 voxels': call(dims=(1 << 11, 1 << 10, 1 << 10)),
    'grid above 2^31 voxels': call(dims=(65535, 65535, 65535)),
    'K = 0': call(K=0), 'K < 0': call(K=-3), 'K = 16385': call(K=16385),
    'radius NaN': call(r=math.nan), 'radius inf': call(r=math.inf), 'radius -inf': call(r=-math.inf),
    'radius < 0': call(r=-1e-9), 'radius > 8': call(r=8.000001),
    'both outputs NULL': call(matrix=None, pairs=None),
    'no labels': call(labels=None), 'no labels, n = 0': call(n=0, labels=None),
    'no points': call(points=None), 'no offsets': call(offsets=None),
}
ok = {'n = 0': call(n=0), 'n = 0 without points': call(n=0, points=None, offsets=None)}
accepted = [call(), call(matrix=None), call(pairs=None), call(K=1), call(K=16384), call(r=0.0), call(r=8.0),
            call(dims=(1 << 11, 1 << 10, (1 << 10) - 1))]
print(json.dumps({'bad': codes, 'ok': ok, 'accepted': accepted}))
'''


def test_connectome_is_exported_bound_and_rejects_bad_arguments():
    """Every bad argument is refused with TTL_ERR_BAD_ARG before any CUDA call.  No device is visible to the
    probe: an accepted call gets past every check and fails at its launch instead of running on the fake
    pointers."""
    build.build()
    lib = _lib.load()
    assert hasattr(lib, 'ttl_connectome') and 'ttl_connectome' in _lib.SIGNATURES
    assert re.search(r'\bttl_connectome\(', open(os.path.join(ROOT, 'include', 'ttl_b200.h')).read())
    assert lib.ttl_abi_version() == _lib.ABI_VERSION == 5
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, '-c', _ARGS_PROBE, ROOT], env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT)
    assert out.returncode == 0, out.stdout.decode()
    res = json.loads(out.stdout.decode().strip().splitlines()[-1])
    assert len(res['bad']) == 20 and all(c == -1 for c in res['bad'].values()), res['bad']
    assert all(c == 0 for c in res['ok'].values()), res['ok']
    assert all(c > 0 for c in res['accepted']), res['accepted']


def test_connectome_kernel_has_no_stack_frame():
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    build.build()
    out = subprocess.run([tool, '-res-usage', _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()
    found = re.findall(r'Function \S*connectome_kernel\S*:\s*\n\s*REG:(\d+) STACK:(\d+).*LOCAL:(\d+)', out)
    assert len(found) == 1, found
    reg, stack, local = (int(x) for x in found[0])
    assert stack == 0 and local == 0, found


# ------------------------------------------------------------------------------------ label volumes

AFFINE = np.array([[1.25, 0, 0, -5.0], [0, 1.25, 0, 3.0], [0, 0, 1.25, 1.0], [0, 0, 0, 1]])
DIMS = (6, 7, 5)


def _labels_file(tmp_path, data, affine=AFFINE, name='labels.nii.gz'):
    path = str(tmp_path / name)
    nifti.save(path, data, affine)
    return path


@pytest.mark.parametrize('dtype', [np.uint8, np.int16, np.int32, np.float32, np.float64])
def test_load_labels_accepts_integer_and_integral_float_volumes(tmp_path, dtype):
    from tracktolearn_b200.runners.ttl_connectivity import load_labels
    rng = np.random.RandomState(1)
    top = 200 if dtype == np.uint8 else 16383
    data = rng.randint(0, top + 1, size=DIMS)
    data.flat[5] = top
    path = _labels_file(tmp_path, data.astype(dtype))
    vol, K = load_labels(path, DIMS, AFFINE + 3e-5, device='cpu')
    assert vol.dtype == torch.int32 and tuple(vol.shape) == DIMS and vol.is_contiguous() and K == top + 1
    np.testing.assert_array_equal(vol.numpy(), data)
    vol, K = load_labels(_labels_file(tmp_path, np.zeros(DIMS, dtype), name='z.nii'), DIMS, AFFINE, device='cpu')
    assert K == 1 and int(vol.sum()) == 0


def test_load_labels_refuses_what_is_not_a_label_volume_of_the_grid(tmp_path):
    from tracktolearn_b200.runners.ttl_connectivity import load_labels
    good = np.ones(DIMS, np.int32)
    frac = good.astype(np.float32)
    frac[1, 2, 3] = 2.5
    neg = good.copy()
    neg[0, 0, 0] = -1
    big = good.copy()
    big[0, 0, 0] = 16384
    nan = good.astype(np.float32)
    nan[2, 2, 2] = np.nan
    shifted = AFFINE.copy()
    shifted[0, 3] += 2e-4
    cases = [_labels_file(tmp_path, frac, name='frac.nii'), _labels_file(tmp_path, neg, name='neg.nii'),
             _labels_file(tmp_path, big, name='big.nii'), _labels_file(tmp_path, nan, name='nan.nii'),
             _labels_file(tmp_path, np.ones((6, 7, 4), np.int32), name='shape.nii'),
             _labels_file(tmp_path, np.ones(DIMS + (2,), np.int32), name='4d.nii'),
             _labels_file(tmp_path, good, shifted, name='affine.nii'),
             _labels_file(tmp_path, good, np.diag([1.25, 1.25, -1.25, 1]), name='flip.nii'),
             str(tmp_path / 'missing.nii.gz')]
    open(str(tmp_path / 'junk.nii'), 'wb').write(b'not a nifti')
    cases.append(str(tmp_path / 'junk.nii'))
    for path in cases:
        with pytest.raises(ValueError):
            load_labels(path, DIMS, AFFINE, device='cpu')


# ------------------------------------------------------------------------------------ command lines

def _touch(path):
    open(path, 'wb').close()
    return str(path)


def _track_argv(tmp_path, out, *extra):
    ins = [_touch(tmp_path / n) for n in ('fodf.nii.gz', 'seed.nii.gz', 'mask.nii.gz')]
    return ins + [str(tmp_path / out), '--agent', str(tmp_path), '--hyperparameters', _touch(tmp_path / 'hp.json')] \
        + list(extra)


def test_ttl_track_connectivity_options(tmp_path):
    from tracktolearn_b200.runners.ttl_track import parse_args
    args = parse_args(_track_argv(tmp_path, 'out.trk'))
    assert args.in_labels is None and args.out_connectivity is None and args.connectivity_radius == 0.0
    assert not args.save_connectivity_labels
    lab = _touch(tmp_path / 'aparc.nii.gz')
    c = str(tmp_path / 'c.npy')
    args = parse_args(_track_argv(tmp_path, 'out.tck', '--in_labels', lab, '--out_connectivity', c,
                                  '--connectivity_radius', '2.5'))
    assert args.in_labels == lab and args.out_connectivity == c and args.connectivity_radius == 2.5
    args = parse_args(_track_argv(tmp_path, 'out.trk', '--in_labels', lab, '--save_connectivity_labels'))
    assert args.save_connectivity_labels and args.out_connectivity is None
    _touch(tmp_path / 'c.npy')
    parse_args(_track_argv(tmp_path, 'out.trk', '--in_labels', lab, '--out_connectivity', c, '-f'))
    d = str(tmp_path / 'd.nii')
    bad = [('--in_labels', lab),                                                         # no output
           ('--out_connectivity', str(tmp_path / 'x.npy')),                              # no labels
           ('--save_connectivity_labels',),
           ('--in_labels', str(tmp_path / 'missing.nii.gz'), '--out_connectivity', str(tmp_path / 'x.npy')),
           ('--in_labels', lab, '--out_connectivity', str(tmp_path / 'x.csv')),          # not .npy
           ('--in_labels', lab, '--out_connectivity', c),                                # exists, no -f
           ('--in_labels', lab, '--out_connectivity', str(tmp_path / 'out.trk'), '-f'),  # the tractogram
           ('--in_labels', lab, '--out_connectivity', str(tmp_path / 'y.npy'), '--connectivity_radius', '-1'),
           ('--in_labels', lab, '--out_connectivity', str(tmp_path / 'y.npy'), '--connectivity_radius', 'nan'),
           ('--in_labels', lab, '--out_connectivity', str(tmp_path / 'y.npy'), '--connectivity_radius', 'inf')]
    for extra in bad:
        with pytest.raises(SystemExit):
            parse_args(_track_argv(tmp_path, 'out.trk', *extra))
    with pytest.raises(SystemExit):                                                      # .tck holds no labels
        parse_args(_track_argv(tmp_path, 'out.tck', '--in_labels', lab, '--save_connectivity_labels'))
    with pytest.raises(SystemExit):                                                      # a NIfTI name
        parse_args(_track_argv(tmp_path, 'out.trk', '--in_labels', lab, '--out_connectivity', d))


def _trk(tmp_path, name, dims, zooms):
    path = str(tmp_path / name)
    w = TrkWriter(path, dims, zooms, np.eye(4))
    w.write(np.zeros((2, 3), F32), np.array([0, 2], np.int64))
    w.close()
    return path


def test_ttl_connectivity_options(tmp_path):
    from tracktolearn_b200.runners.ttl_connectivity import parse_args
    lab = _labels_file(tmp_path, np.arange(np.prod(DIMS)).reshape(DIMS) % 5)
    trk = _trk(tmp_path, 'in.trk', DIMS, (1.25, 1.25, 1.25))
    tck = _touch(tmp_path / 'in.tck')
    out = str(tmp_path / 'c.npy')
    args = parse_args([trk, lab, out])
    assert args.out_connectivity == out and args.radius == 0.0 and args.labels_image.shape == DIMS
    assert parse_args([tck, lab, out, '--radius', '10']).radius == 10.0                   # 8 voxels of 1.25 mm
    _touch(tmp_path / 'c.npy')
    parse_args([trk, lab, out, '-f'])
    bad = [[trk, lab, out],                                                              # exists, no -f
           [trk, lab, str(tmp_path / 'c.txt')],                                          # not .npy
           [trk, lab, lab, '-f'], [trk, lab, trk, '-f'],
           [trk, lab, str(tmp_path / 'x.npy'), '--radius', '-0.5'],
           [trk, lab, str(tmp_path / 'x.npy'), '--radius', 'nan'],
           [trk, lab, str(tmp_path / 'x.npy'), '--radius', '10.01'],                     # above 8 voxels
           [str(tmp_path / 'in.vtk'), lab, str(tmp_path / 'x.npy')],
           [str(tmp_path / 'missing.trk'), lab, str(tmp_path / 'x.npy')],
           [trk, str(tmp_path / 'missing.nii'), str(tmp_path / 'x.npy')],
           [trk, _labels_file(tmp_path, np.full(DIMS, 0.5, np.float32), name='f.nii'), str(tmp_path / 'x.npy')],
           [_trk(tmp_path, 'dims.trk', (6, 7, 6), (1.25, 1.25, 1.25)), lab, str(tmp_path / 'x.npy')],
           [_trk(tmp_path, 'vox.trk', DIMS, (1.25, 1.5, 1.25)), lab, str(tmp_path / 'x.npy')],
           [_touch(tmp_path / 'empty.trk'), lab, str(tmp_path / 'x.npy')]]
    for argv in bad:
        with pytest.raises(SystemExit):
            parse_args(argv)


def test_help_lists_the_connectivity_options():
    for script, flags in (('ttl_track.py', ('Connectivity', '--in_labels', '--out_connectivity',
                                            '--connectivity_radius', '--save_connectivity_labels')),
                          ('ttl_connectivity.py', ('in_tractogram', 'in_labels', 'out_connectivity', '--radius'))):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', script), '--help'],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        for flag in flags:
            assert flag in out.stdout, (script, flag)


# ------------------------------------------------------------------------------------ ranks and files

GRID = (6, 7, 5)


def _rank_part(rank):
    rng = np.random.RandomState(30 + rank)
    lab = _parcellation(np.random.RandomState(99), GRID, 5, 0.5)
    sl = _random_set(rng, 40 + 13 * rank, GRID, lo=1)
    data, offsets = _pack(sl)
    m, pairs = C.connectome(data, offsets, lab, 1.5)
    return sl, data, offsets, m, pairs


def _worker(rank, world, port, via, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    _, data, offsets, m, pairs = _rank_part(rank)
    matrix = torch.from_numpy(m)
    total = parallel.reduce_maps([None, None, matrix], 3 + rank)
    n = len(offsets) - 1
    merged = parallel.gather_packed(torch.from_numpy(data), torch.from_numpy(np.diff(offsets)),
                                    torch.zeros((n, 3), dtype=torch.float64), torch.zeros((n,), dtype=torch.int64),
                                    via=via, labels=torch.from_numpy(pairs))
    if rank == 0:
        q.put((matrix.numpy().copy(), total, merged.offsets, dict(merged.data_per_streamline)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('via', ['nccl', 'host'])
def test_two_rank_reduce_sums_the_matrices_and_gather_carries_the_labels(via):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, via, q)) for r in range(2)]
    for p in procs:
        p.start()
    matrix, total, offsets, per = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    parts = [_rank_part(r) for r in range(2)]
    lab = _parcellation(np.random.RandomState(99), GRID, 5, 0.5)
    whole = C.connectome(*_pack(parts[0][0] + parts[1][0]), lab, 1.5)
    np.testing.assert_array_equal(matrix, whole[0])
    assert total == 7
    np.testing.assert_array_equal(np.stack((per['start_label'], per['end_label']), 1), whole[1])
    assert per['start_label'].dtype == np.int32 and 'oracle_score' not in per


@pytest.mark.parametrize('save_seeds,save_scores', [(False, False), (True, True), (False, True)])
def test_trk_start_and_end_label_round_trip(tmp_path, save_seeds, save_scores):
    rng = np.random.RandomState(5)
    path = str(tmp_path / 'a.trk')
    w = TrkWriter(path, (10, 11, 12), (1.25, 1.25, 1.25), np.eye(4), save_seeds=save_seeds, save_scores=save_scores,
                  save_labels=True)
    batches = []
    for n in (9, 0, 25):
        lens = rng.randint(1, 30, size=n)
        offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
        data = rng.randn(int(offsets[-1]), 3).astype(F32)
        seeds, scores = rng.randn(n, 3), rng.rand(n).astype(F32)
        labels = rng.randint(0, 16384, size=(n, 2)).astype(np.int32)
        labels[:1] = 16383
        w.write(data, offsets, seeds if save_seeds else None, scores if save_scores else None, labels)
        batches.append((data, offsets, seeds, scores, labels))
    w.close()
    data, offsets, hdr = read_trk(path)
    names = ['seeds_x', 'seeds_y', 'seeds_z'] * save_seeds + ['oracle_score'] * save_scores + \
        ['start_label', 'end_label']
    assert hdr['property_names'] == names and hdr['n_count'] == 34
    np.testing.assert_array_equal(data, np.concatenate([b[0] for b in batches]))
    np.testing.assert_array_equal(np.diff(offsets), np.concatenate([np.diff(b[1]) for b in batches]))
    props = hdr['properties']
    np.testing.assert_array_equal(props[:, -2:].astype(np.int32), np.concatenate([b[4] for b in batches]))
    assert props.dtype == np.float32
    if save_scores:
        np.testing.assert_array_equal(props[:, -3], np.concatenate([b[3] for b in batches]))
    if save_seeds:
        np.testing.assert_array_equal(props[:, :3], np.concatenate([b[2] for b in batches]).astype(F32))


def test_trk_bytes_unchanged_without_labels(tmp_path):
    rng = np.random.RandomState(6)
    lens = rng.randint(1, 30, size=12)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = rng.randn(int(offsets[-1]), 3).astype(F32)
    seeds, scores = rng.randn(12, 3), rng.rand(12)
    outs = []
    for kw in ({}, {'save_labels': False}):
        path = str(tmp_path / ('%d.trk' % len(outs)))
        w = TrkWriter(path, (10, 11, 12), (2.0, 2.0, 2.0), np.eye(4), True, save_scores=True, **kw)
        w.write(data, offsets, seeds, scores)
        w.close()
        outs.append(open(path, 'rb').read())
    assert outs[0] == outs[1]


def test_unlabelled_endpoint_count_from_row_zero():
    from tracktolearn_b200.tracking.postprocess import radius_voxels, unlabelled_endpoints
    lab = np.zeros((4, 4, 4), np.int32)
    lab[0, 0, 0], lab[3, 3, 3] = 1, 2
    sl = [[(0, 0, 0), (3, 3, 3)], [(0, 0, 0), (2, 0, 0)], [(1, 2, 1), (2, 1, 2)], [(1, 1, 1)], [(3, 3, 3), (1, 0, 3)]]
    m, pairs = C.connectome(*_pack(sl), lab, 0.0)
    assert unlabelled_endpoints(m) == int((pairs == 0).sum()) == 6
    assert radius_voxels(4.0, AFFINE) == 3.2 and radius_voxels(0, AFFINE) == 0.0
    for bad in (-1.0, float('nan'), float('inf'), 10.01):
        with pytest.raises(ValueError):
            radius_voxels(bad, AFFINE)
