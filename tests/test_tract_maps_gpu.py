"""Streamline maps on the device: ttl_tract_maps against the restatement of tests/maps_oracle.py (integer
equality, exact skipped counts), accumulation across calls, Tracker.track_to_file with maps,
ttl_track.py --out_density / --out_endpoints, ttl_tract_maps.py, and an out-of-bounds check of the maps."""
import os

import numpy as np
import pytest
import torch

from tests import maps_oracle as M

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
F32 = np.float32


def _pack(streamlines):
    lens = [len(s) for s in streamlines]
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = np.concatenate([np.asarray(s, dtype=F32).reshape(-1, 3) for s in streamlines])
    return data.astype(F32), offsets


def _device_maps(data, offsets, dims, density=True, endpoints=True):
    from tracktolearn_b200.tracking.postprocess import tract_maps_packed
    maps = [torch.zeros(dims, dtype=torch.int32, device=DEV) if w else None for w in (density, endpoints)]
    skipped = tract_maps_packed(torch.from_numpy(data).to(DEV), torch.from_numpy(offsets).to(DEV), dims, *maps)
    return tuple(None if m is None else m.cpu().numpy() for m in maps) + (skipped,)


def _check(data, offsets, dims, want=None):
    want = want if want is not None else M.tract_maps(data, offsets, dims)
    for flags in ((True, True), (True, False), (False, True)):
        got = _device_maps(data, offsets, dims, *flags)
        assert got[2] == want[2]
        for g, w, on in zip(got[:2], want[:2], flags):
            if on:
                assert g.dtype == np.int32
                np.testing.assert_array_equal(g, w)
            else:
                assert g is None
    return want


def _walks(rng, n, dims, lo, hi, step=0.6, junk=0.03, wrap=False):
    out = []
    for _ in range(n):
        L = int(rng.randint(lo, hi))
        s = np.cumsum(rng.randn(L, 3) * step, axis=0) + rng.rand(3) * np.asarray(dims)
        if wrap:          # back into the grid: long walks keep meeting new voxels and old ones
            s = np.mod(s + 0.5, np.asarray(dims)) - 0.5
        if junk and L:
            hit = rng.rand(L) < junk
            s[hit, rng.randint(0, 3)] = rng.choice([np.nan, np.inf, -np.inf, -0.5, -0.51, dims[0] - 0.5])
        out.append(s.astype(F32))
    return out


def test_random_streamlines_with_revisits():
    rng = np.random.RandomState(0)
    dims = (13, 11, 9)
    data, offsets = _pack(_walks(rng, 3000, dims, 0, 300) + [np.zeros((0, 3), F32)] * 5)
    want = _check(data, offsets, dims)
    assert want[2] > 0 and want[0].max() > 50


def _faces(dims):
    """Points on and beside every face of the grid, in every axis."""
    vals = []
    for d in dims:
        edge = [F32(-0.5), np.nextafter(F32(-0.5), F32(-1)), np.nextafter(F32(-0.5), F32(0)),
                F32(d - 0.5), np.nextafter(F32(d - 0.5), F32(0)), np.nextafter(F32(d - 0.5), F32(d)),
                np.nextafter(F32(0.5), F32(0)), F32(0.5), F32(0.0), F32(d - 1), F32(np.nan), F32(np.inf),
                F32(-np.inf), F32(-1e30), F32(1e30)]
        vals.append(np.asarray(edge, dtype=F32))
    g = np.stack(np.meshgrid(*vals, indexing='ij'), -1).reshape(-1, 3)
    return g


@pytest.mark.parametrize('dims', [(1, 1, 1), (1, 7, 1), (5, 3, 7), (2, 9, 4)])
def test_adversarial_boundary_points(dims):
    rng = np.random.RandomState(1)
    pts = _faces(dims)
    rng.shuffle(pts)
    cuts = np.sort(rng.choice(np.arange(1, len(pts)), size=len(pts) // 7, replace=False))
    sl = np.split(pts, cuts)
    data, offsets = _pack(sl + [pts[:1], pts[-1:]])
    want = _check(data, offsets, dims)
    assert want[2] > 0 and want[0].sum() > 0


def test_streamlines_longer_than_the_shared_window():
    """More distinct voxels than the per-warp shared set holds (512): the rescan path stays exact."""
    rng = np.random.RandomState(2)
    dims = (40, 41, 39)
    long = _walks(rng, 6, dims, 10000, 20000, step=0.8, junk=0.01, wrap=True)
    distinct = [len({M.voxel_of(p, dims) for p in s} - {None}) for s in long]
    assert min(distinct) > 512, distinct
    short = _walks(rng, 200, dims, 1, 200)
    data, offsets = _pack(long[:3] + short + long[3:])
    _check(data, offsets, dims, M.tract_maps_fast(data, offsets, dims))


def test_a_million_short_streamlines():
    rng = np.random.RandomState(3)
    dims = (64, 70, 58)
    n = 1_000_000
    lens = rng.randint(0, 8, size=n)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    start = np.repeat(rng.rand(n, 3) * (np.asarray(dims) + 2) - 1, lens, axis=0)
    data = (start + rng.randn(int(offsets[-1]), 3) * 0.7).astype(F32)
    want = _check(data, offsets, dims, M.tract_maps_fast(data, offsets, dims))
    assert want[2] > 0 and want[1].sum() > n


def test_maps_accumulate_across_calls_in_any_order():
    from tracktolearn_b200.tracking.postprocess import tract_maps_packed
    rng = np.random.RandomState(4)
    dims = (17, 15, 16)
    sl = _walks(rng, 5000, dims, 0, 150)
    whole = _device_maps(*_pack(sl), dims)
    maps = [torch.zeros(dims, dtype=torch.int32, device=DEV) for _ in range(2)]
    skipped = 0
    for part in (sl[:2222], sl[2222:]):
        d, o = _pack(part)
        skipped += tract_maps_packed(torch.from_numpy(d).to(DEV), torch.from_numpy(o).to(DEV), dims, *maps)
    assert skipped == whole[2]
    for m, w in zip(maps, whole[:2]):
        assert m.cpu().numpy().tobytes() == w.tobytes()
    rev = _device_maps(*_pack(sl[::-1]), dims)
    assert rev[2] == whole[2]
    for r, w in zip(rev[:2], whole[:2]):
        assert r.tobytes() == w.tobytes()


def test_no_write_outside_the_maps():
    """The maps and the skipped counter are carved out of larger allocations with 4 KB of 0xA5 on each side;
    at awkward sizes, with points on every face, no guard byte may change."""
    from tracktolearn_b200 import _lib
    from tracktolearn_b200.environments.tracking_env import GUARD_BYTES, GUARD_FILL
    lib = _lib.load()
    rng = np.random.RandomState(5)
    for dims in ((1, 1, 1), (1, 9, 1), (3, 1, 5), (7, 5, 3), (11, 13, 1)):
        pts = _faces(dims)
        rng.shuffle(pts)
        cuts = np.sort(rng.choice(np.arange(1, len(pts)), size=len(pts) // 5, replace=False))
        data, offsets = _pack(np.split(pts, cuts))
        want = M.tract_maps(data, offsets, dims)
        raws, views = [], []
        for nbytes, dtype in ((4 * int(np.prod(dims)), torch.int32), (4 * int(np.prod(dims)), torch.int32),
                              (8, torch.int64)):
            raw = torch.full((nbytes + 2 * GUARD_BYTES,), GUARD_FILL, dtype=torch.uint8, device=DEV)
            v = raw[GUARD_BYTES:GUARD_BYTES + nbytes].view(dtype)
            v.zero_()
            raws.append((raw, nbytes))
            views.append(v)
        d, o = torch.from_numpy(data).to(DEV), torch.from_numpy(offsets).to(DEV)
        _lib.check(lib.ttl_tract_maps(_lib.ptr(d), _lib.ptr(o), len(offsets) - 1, *dims, _lib.ptr(views[0]),
                                      _lib.ptr(views[1]), _lib.ptr(views[2]), _lib.stream_ptr(DEV)), 'ttl_tract_maps')
        torch.cuda.synchronize()
        for raw, nbytes in raws:
            assert int((raw[:GUARD_BYTES] != GUARD_FILL).sum()) == 0, dims
            assert int((raw[GUARD_BYTES + nbytes:] != GUARD_FILL).sum()) == 0, dims
        np.testing.assert_array_equal(views[0].cpu().numpy().reshape(dims), want[0])
        np.testing.assert_array_equal(views[1].cpu().numpy().reshape(dims), want[1])
        assert int(views[2].item()) == want[2] > 0


# ------------------------------------------------------------------------------------ Tracker.track_to_file

def test_track_to_file_maps(tmp_path):
    from tests.test_tracker_gpu import _setup
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.tracking.postprocess import lengths_packed
    from tracktolearn_b200.tracking.tracker import Tracker
    env, alg, sub, seeds, _ = _setup(precision='fp16')
    seeds = np.array(env.seeds, copy=True)
    dims = tuple(sub['mask'].shape[:3])

    def tracker(compress=0.0):
        env.seeds = seeds.copy()
        np.random.seed(0)
        return Tracker(alg, 256, min_length=5, max_length=200, save_seeds=True, compress=compress)

    def run(name, compress=0.0, maps=True, **kw):
        t = tracker(compress)
        path = str(tmp_path / name)
        stem = path.rsplit('.', 1)[0]
        if maps:
            kw.update(density_path=stem + '_density.nii', endpoints_path=stem + '_endpoints.nii')
        n = t.track_to_file(env, path, dims, (1.0, 1.0, 1.0), **kw)
        out = (open(path, 'rb').read(), n, t.maps_skipped)
        if maps:
            out += tuple(nifti.load(kw[k]) for k in ('density_path', 'endpoints_path'))
        return out

    trk, n, skipped, den, end = run('a.trk')
    assert den.data.dtype == np.int32 and den.shape == dims and end.shape == dims
    np.testing.assert_array_equal(den.affine, np.asarray(env.affine_vox2rasmm, dtype=np.float32))

    # the restatement on the length-kept voxel-space streamlines of a separate track_packed run
    t = tracker()
    np.random.shuffle(env.seeds)
    kept = []
    for batch in t.track_packed(env):
        lens = lengths_packed(batch.data, batch.offsets).cpu().numpy()
        for i in np.nonzero((lens >= 5.0) & (lens <= 200.0))[0]:
            kept.append(batch.data[batch.offsets[i]:batch.offsets[i + 1]])
    assert len(kept) == n > 100
    want = M.tract_maps(*_pack(kept), dims)
    np.testing.assert_array_equal(den.data, want[0])
    np.testing.assert_array_equal(end.data, want[1])
    assert skipped == want[2]
    assert int(end.data.sum()) == 2 * n - sum(M.voxel_of(p, dims) is None for s in kept for p in (s[0], s[-1]))

    # the tractogram does not change with maps, and the maps do not change with --compress
    assert run('b.trk', maps=False)[0] == trk
    assert run('a.tck')[0] == run('b.tck', maps=False)[0]
    comp = run('c.trk', compress=0.2)
    assert comp[0] != trk and comp[1] == n
    assert comp[3].data.tobytes() == den.data.tobytes() and comp[4].data.tobytes() == end.data.tobytes()
    assert run('c2.trk', compress=0.2, maps=False)[0] == comp[0]


# ------------------------------------------------------------------------------------ command line

def test_ttl_track_maps_and_ttl_tract_maps(tmp_path, capsys):
    from tests.test_oracle_filter_gpu import _subject, _track
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.io.streamlines import read_trk
    from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
    from tracktolearn_b200.runners.ttl_tract_maps import main as maps_main
    agent, affine = _subject(tmp_path)
    outs = {}
    for n_actor in (500, 173):
        d, e = str(tmp_path / ('d%d.nii' % n_actor)), str(tmp_path / ('e%d.nii' % n_actor))
        trk = _track(tmp_path, agent, 't%d.trk' % n_actor, '--n_actor', str(n_actor), '--noise_rng', 'device',
                     '--noise', '0.1', '--out_density', d, '--out_endpoints', e)
        outs[n_actor] = (open(trk, 'rb').read(), open(d, 'rb').read(), open(e, 'rb').read(), d, e, trk)
    assert outs[500][:3] == outs[173][:3]
    d, e, trk = outs[500][3:]
    den, end = nifti.load(d), nifti.load(e)
    assert den.data.dtype == np.int32 and int(den.data.sum()) > 0
    np.testing.assert_array_equal(den.affine, affine.astype(np.float32))

    # the standalone command on the .trk: equal except at voxels touched by points within float32 round-trip
    # distance of a voxel face
    d2, e2 = str(tmp_path / 'd_post.nii.gz'), str(tmp_path / 'e_post.nii.gz')
    capsys.readouterr()
    maps_main([trk, '--reference', str(tmp_path / 'mask.nii.gz'), '--out_density', d2, '--out_endpoints', e2])
    assert 'Wrote' in capsys.readouterr().out
    post_d, post_e = nifti.load(d2), nifti.load(e2)
    data, offsets, hdr = read_trk(trk)
    vox = voxel_points(data, 'trk', hdr['voxel_sizes']).astype(np.float64)
    dims = den.shape
    frac = vox + 0.5 - np.round(vox + 0.5)
    near = np.any(np.abs(frac) <= 8 * np.spacing(np.abs(vox).astype(F32) + F32(1)), axis=1)
    excluded = np.zeros(dims, dtype=bool)
    for p in vox[near]:
        lo = np.floor(p + 0.5 - 1e-4).astype(int)
        hi = np.floor(p + 0.5 + 1e-4).astype(int)
        sl = tuple(slice(max(a, 0), min(b, dd - 1) + 1) for a, b, dd in zip(lo, hi, dims))
        excluded[sl] = True
    print('points within float32 round-trip distance of a voxel face: %d, voxels excluded: %d'
          % (int(near.sum()), int(excluded.sum())))
    np.testing.assert_array_equal(post_d.data[~excluded], den.data[~excluded])
    np.testing.assert_array_equal(post_e.data[~excluded], end.data[~excluded])
    if not excluded.any():
        assert post_d.data.tobytes() == den.data.tobytes() and post_e.data.tobytes() == end.data.tobytes()
