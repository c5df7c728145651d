"""Streamline maps without a GPU: the restatement against dipy's density_map rule on hand-made cases, the
C ABI of ttl_tract_maps and its argument checks, the kernel's stack frame, the argument checks of
ttl_track.py --out_density / --out_endpoints and ttl_tract_maps.py, the world-2 gloo reduction of per-rank
maps and the int32 NIfTI round trip."""
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

from tests import maps_oracle as M
from tracktolearn_b200 import _lib, build, parallel
from tracktolearn_b200.io import nifti
from tracktolearn_b200.io.streamlines import TrkWriter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def _pack(streamlines):
    lens = [len(s) for s in streamlines]
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = np.concatenate([np.asarray(s, dtype=F32).reshape(-1, 3) for s in streamlines]) if streamlines else \
        np.zeros((0, 3), F32)
    return data.astype(F32), offsets


def _dipy_density(streamlines, dims):
    """dipy.tracking.utils.density_map(streamlines, affine=eye, vol_dims) for in-grid streamlines: the voxel
    index is int(p + 0.5) in float64, and counts[i, j, k] += 1 counts a voxel once per streamline."""
    counts = np.zeros(dims, dtype=np.int64)
    for s in streamlines:
        inds = (np.asarray(s, dtype=F32).astype(np.float64) + 0.5).astype(int)
        i, j, k = inds.T
        counts[i, j, k] += 1
    return counts


def test_voxel_rule_at_the_faces():
    dims = (4, 5, 6)
    below = np.nextafter(F32(0.5), F32(0))                     # 0.49999997: a float32 sum would round to 1
    assert M.voxel_of((below, 0, 0), dims) == (0, 0, 0)
    for k in range(4):                                          # exactly k - 0.5 belongs to voxel k
        assert M.voxel_of((F32(k - 0.5), 0, 0), dims) == (k, 0, 0)
    assert M.voxel_of((F32(-0.5), F32(-0.5), F32(-0.5)), dims) == (0, 0, 0)
    assert M.voxel_of((np.nextafter(F32(-0.5), F32(-1)), 0, 0), dims) is None
    assert M.voxel_of((F32(-3), 0, 0), dims) is None
    assert M.voxel_of((F32(3.5), 0, 0), dims) is None           # dim - 0.5: voxel dim, outside
    assert M.voxel_of((np.nextafter(F32(3.5), F32(0)), 0, 0), dims) == (3, 0, 0)
    assert M.voxel_of((0, F32(4.5), 0), dims) is None and M.voxel_of((0, 0, F32(5.5)), dims) is None
    for bad in (np.nan, np.inf, -np.inf):
        assert M.voxel_of((F32(bad), 1, 1), dims) is None
        assert M.voxel_of((1, 1, F32(bad)), dims) is None


def test_restatement_counts_a_revisit_once_and_both_endpoints():
    dims = (3, 3, 3)
    a, b = (0.1, 0.2, 0.3), (1.2, 0.1, 0.0)
    sl = [[a, a, b, b, a, (F32(np.nan), 0, 0), a],             # leaves voxel 0 and comes back
          [b],                                                  # one point: 2 at its voxel
          [],                                                   # no point: nothing
          [(-1.0, 0, 0), b, (2.4, 2.6, 0)]]                     # first point outside, last point outside
    data, offsets = _pack(sl)
    density, endpoints, skipped = M.tract_maps(data, offsets, dims)
    assert density[0, 0, 0] == 1 and density[1, 0, 0] == 3 and density.sum() == 4
    assert endpoints[0, 0, 0] == 2 and endpoints[1, 0, 0] == 2 and endpoints.sum() == 4
    assert skipped == 3
    for got, want in zip(M.tract_maps_fast(data, offsets, dims), (density, endpoints, skipped)):
        np.testing.assert_array_equal(got, want)


def _random_set(rng, n, dims, junk=True):
    sl = []
    for _ in range(n):
        L = int(rng.randint(0, 60))
        # a random walk of small steps: revisits after leaving a voxel are common
        s = np.cumsum(rng.randn(L, 3) * 0.6, axis=0) + rng.rand(3) * np.asarray(dims)
        if junk and L:
            hit = rng.rand(L) < 0.05
            s[hit, rng.randint(0, 3)] = rng.choice([np.nan, np.inf, -np.inf, -0.5, dims[0] - 0.5])
        sl.append(s.astype(F32))
    return sl


def test_restatement_matches_dipy_and_keeps_the_endpoint_invariant():
    rng = np.random.RandomState(0)
    dims = (9, 7, 8)
    sl = _random_set(rng, 300, dims, junk=False)
    # dipy raises for any point outside; compare on the streamlines entirely inside the grid
    inside = [s for s in sl if len(s) and all(M.voxel_of(p, dims) is not None for p in s)]
    assert len(inside) > 30
    density, _, skipped = M.tract_maps(*_pack(inside), dims)
    assert skipped == 0
    np.testing.assert_array_equal(density, _dipy_density(inside, dims))
    sl = _random_set(rng, 400, dims)
    data, offsets = _pack(sl)
    density, endpoints, skipped = M.tract_maps(data, offsets, dims)
    nonempty = [s for s in sl if len(s)]
    ends_out = sum(M.voxel_of(p, dims) is None for s in nonempty for p in (s[0], s[-1]))
    assert endpoints.sum() == 2 * len(nonempty) - ends_out
    assert skipped == sum(M.voxel_of(p, dims) is None for s in sl for p in s) > 0
    for got, want in zip(M.tract_maps_fast(data, offsets, dims), (density, endpoints, skipped)):
        np.testing.assert_array_equal(got, want)


# ------------------------------------------------------------------------------------ C ABI

_MAPS_ARGS_PROBE = r'''
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from tracktolearn_b200 import _lib
lib = _lib.load()
fake = iter(range(1 << 20, 1 << 30, 1 << 16))          # distinct aligned addresses, never dereferenced
pts, off, den, end, skip = (ctypes.c_void_p(next(fake)) for _ in range(5))


def call(n=10, dims=(4, 5, 6), density=den, endpoints=end, skipped=skip, points=pts, offsets=off):
    return lib.ttl_tract_maps(points, offsets, n, *dims, density, endpoints, skipped, None)


codes = {
    'n < 0': call(n=-1),
    'zero x': call(dims=(0, 5, 6)), 'zero y': call(dims=(4, 0, 6)), 'zero z': call(dims=(4, 5, 0)),
    'negative dim': call(dims=(4, -5, 6)),
    'grid of 2^31 voxels': call(dims=(1 << 11, 1 << 10, 1 << 10)),
    'grid above 2^31 voxels': call(dims=(65535, 65535, 65535)),
    'both maps NULL': call(density=None, endpoints=None),
    'no skipped counter': call(skipped=None),
    'no points': call(points=None), 'no offsets': call(offsets=None),
}
ok = {'n = 0': call(n=0), 'n = 0 without points': call(n=0, points=None, offsets=None)}
accepted = [call(), call(density=None), call(endpoints=None), call(dims=(1 << 11, 1 << 10, (1 << 10) - 1))]
print(json.dumps({'bad': codes, 'ok': ok, 'accepted': accepted}))
'''


def test_tract_maps_is_exported_bound_and_rejects_bad_arguments():
    """Every bad argument is refused with TTL_ERR_BAD_ARG before any CUDA call.  No device is visible to the
    probe: an accepted call fails at its launch instead of running on the fake pointers."""
    build.build()
    lib = _lib.load()
    assert hasattr(lib, 'ttl_tract_maps') and 'ttl_tract_maps' in _lib.SIGNATURES
    assert re.search(r'\bttl_tract_maps\(', open(os.path.join(ROOT, 'include', 'ttl_b200.h')).read())
    assert lib.ttl_abi_version() == _lib.ABI_VERSION == 5
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, '-c', _MAPS_ARGS_PROBE, ROOT], env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT)
    assert out.returncode == 0, out.stdout.decode()
    res = json.loads(out.stdout.decode().strip().splitlines()[-1])
    assert len(res['bad']) == 11 and all(c == -1 for c in res['bad'].values()), res['bad']
    assert all(c == 0 for c in res['ok'].values()), res['ok']
    assert all(c > 0 for c in res['accepted']), res['accepted']


def test_tract_maps_kernel_has_no_stack_frame():
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    build.build()
    out = subprocess.run([tool, '-res-usage', _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()
    found = re.findall(r'Function \S*tract_maps_kernel\S*:\s*\n\s*REG:(\d+) STACK:(\d+).*LOCAL:(\d+)', out)
    assert len(found) == 1, found
    reg, stack, local = (int(x) for x in found[0])
    assert stack == 0 and local == 0, found


# ------------------------------------------------------------------------------------ command lines

def _touch(path):
    open(path, 'wb').close()
    return str(path)


def _track_argv(tmp_path, out, *extra):
    ins = [_touch(tmp_path / n) for n in ('fodf.nii.gz', 'seed.nii.gz', 'mask.nii.gz')]
    return ins + [str(tmp_path / out), '--agent', str(tmp_path), '--hyperparameters', _touch(tmp_path / 'hp.json')] \
        + list(extra)


def test_ttl_track_map_options(tmp_path):
    from tracktolearn_b200.runners.ttl_track import parse_args
    args = parse_args(_track_argv(tmp_path, 'out.trk'))
    assert args.out_density is None and args.out_endpoints is None
    d, e = str(tmp_path / 'd.nii.gz'), str(tmp_path / 'e.nii')
    args = parse_args(_track_argv(tmp_path, 'out.tck', '--out_density', d, '--out_endpoints', e))
    assert args.out_density == d and args.out_endpoints == e
    _touch(tmp_path / 'd.nii.gz')
    parse_args(_track_argv(tmp_path, 'out.trk', '--out_density', d, '-f'))
    bad = [('--out_density', str(tmp_path / 'd.mgz')),
           ('--out_endpoints', str(tmp_path / 'e.trk')),
           ('--out_density', d),                                           # exists, no -f
           ('--out_density', e, '--out_endpoints', e),                     # the same file twice
           ('--out_density', str(tmp_path / 'x.nii'), '--out_endpoints', str(tmp_path / 'x.nii'), '-f')]
    for extra in bad:
        with pytest.raises(SystemExit):
            parse_args(_track_argv(tmp_path, 'out.trk', *extra))
    with pytest.raises(SystemExit):                                        # one file, spelled twice
        parse_args(_track_argv(tmp_path, 'out.trk', '--out_density', e,
                               '--out_endpoints', os.path.join(str(tmp_path), '.', 'e.nii')))


def _reference(tmp_path, shape=(10, 11, 12), zooms=(1.25, 1.25, 1.25), name='ref.nii.gz'):
    affine = np.diag(list(zooms) + [1.0])
    affine[:3, 3] = [-5.0, 3.0, 1.0]
    path = str(tmp_path / name)
    nifti.save(path, np.zeros(shape, dtype=np.uint8), affine)
    return path


def _trk(tmp_path, name, dims, zooms):
    path = str(tmp_path / name)
    w = TrkWriter(path, dims, zooms, np.eye(4))
    w.write(np.zeros((2, 3), F32), np.array([0, 2], np.int64))
    w.close()
    return path


def test_ttl_tract_maps_options(tmp_path):
    from tracktolearn_b200.runners.ttl_tract_maps import parse_args
    ref = _reference(tmp_path)
    trk = _trk(tmp_path, 'in.trk', (10, 11, 12), (1.25, 1.25, 1.25))
    tck = _touch(tmp_path / 'in.tck')
    d, e = str(tmp_path / 'd.nii.gz'), str(tmp_path / 'e.nii')
    args = parse_args([trk, '--reference', ref, '--out_density', d])
    assert args.out_density == d and args.out_endpoints is None and args.reference_image.shape == (10, 11, 12)
    parse_args([tck, '--reference', ref, '--out_endpoints', e])
    parse_args([trk, '--reference', ref, '--out_density', d, '--out_endpoints', e])
    _touch(tmp_path / 'e.nii')
    parse_args([trk, '--reference', ref, '--out_endpoints', e, '-f'])
    bad = [[trk, '--out_density', d],                                                  # no --reference
           [trk, '--reference', ref],                                                  # no output
           [trk, '--reference', ref, '--out_endpoints', e],                            # exists, no -f
           [trk, '--reference', ref, '--out_density', d, '--out_endpoints', d],        # the same file twice
           [trk, '--reference', ref, '--out_density', ref, '-f'],                      # the reference itself
           [trk, '--reference', ref, '--out_density', str(tmp_path / 'd.trk')],        # not NIfTI
           [str(tmp_path / 'in.vtk'), '--reference', ref, '--out_density', d],         # not .trk / .tck
           [str(tmp_path / 'missing.trk'), '--reference', ref, '--out_density', d],
           [trk, '--reference', str(tmp_path / 'missing.nii'), '--out_density', d],
           [_trk(tmp_path, 'dims.trk', (10, 11, 13), (1.25, 1.25, 1.25)), '--reference', ref, '--out_density', d],
           [_trk(tmp_path, 'vox.trk', (10, 11, 12), (1.25, 1.5, 1.25)), '--reference', ref, '--out_density', d],
           [_touch(tmp_path / 'empty.trk'), '--reference', ref, '--out_density', d]]
    for argv in bad:
        with pytest.raises(SystemExit):
            parse_args(argv)


def test_help_lists_the_map_options():
    for script, flags in (('ttl_track.py', ('Maps', '--out_density', '--out_endpoints')),
                          ('ttl_tract_maps.py', ('in_tractogram', '--reference', '--out_density',
                                                 '--out_endpoints'))):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', script), '--help'],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        for flag in flags:
            assert flag in out.stdout, (script, flag)


# ------------------------------------------------------------------------------------ reduction and files

DIMS = (6, 7, 5)


def _rank_maps(rank):
    sl = _random_set(np.random.RandomState(20 + rank), 50 + 17 * rank, DIMS)
    return sl, M.tract_maps(*_pack(sl), DIMS)


def _reduce_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    _, (density, endpoints, skipped) = _rank_maps(rank)
    d, e = torch.from_numpy(density), torch.from_numpy(endpoints)
    total = parallel.reduce_maps([d, None, e], skipped)
    if rank == 0:
        q.put((d.numpy().copy(), e.numpy().copy(), total))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_reduce_sums_the_maps():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_reduce_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    density, endpoints, skipped = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    whole = M.tract_maps(*_pack(_rank_maps(0)[0] + _rank_maps(1)[0]), DIMS)
    np.testing.assert_array_equal(density, whole[0])
    np.testing.assert_array_equal(endpoints, whole[1])
    assert skipped == whole[2] > 0
    assert parallel.reduce_maps([torch.zeros(DIMS, dtype=torch.int32)], 7) == 7        # one process


@pytest.mark.parametrize('ext', ['nii', 'nii.gz'])
def test_int32_map_nifti_round_trip(tmp_path, ext):
    rng = np.random.RandomState(2)
    m = rng.randint(0, 1 << 30, size=(5, 7, 3)).astype(np.int32)
    affine = np.array([[-1.25, 0, 0, 30.0], [0, 1.25, 0, -12.5], [0, 0, 1.5, 4.0], [0, 0, 0, 1]])
    path = str(tmp_path / ('m.' + ext))
    nifti.save(path, m, affine)
    img = nifti.load(path)
    assert img.data.dtype == np.int32 and img.shape == m.shape
    np.testing.assert_array_equal(img.data, m)
    np.testing.assert_array_equal(img.affine, affine.astype(np.float32))
