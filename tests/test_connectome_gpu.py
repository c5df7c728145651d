"""Connectivity matrix on the device: ttl_connectome against the restatement of tests/connectome_oracle.py (integer
equality of the matrix and of every streamline's end labels), accumulation across calls, the worst-case
contention case, an out-of-bounds check of the matrix and the pairs, Tracker.track_to_file with labels,
ttl_track.py --in_labels / --out_connectivity and ttl_connectivity.py."""

import numpy as np
import pytest
import torch

from tests import connectome_oracle as C

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
F32 = np.float32


def _pack(streamlines):
    lens = [len(s) for s in streamlines]
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = np.concatenate([np.asarray(s, dtype=F32).reshape(-1, 3) for s in streamlines])
    return data.astype(F32), offsets


def _device(data, offsets, labels, r, matrix=True, pairs=True, K=None):
    from tracktolearn_b200.tracking.postprocess import connectome_packed
    K = int(labels.max()) + 1 if K is None else K
    lab = torch.from_numpy(np.ascontiguousarray(labels, dtype=np.int32)).to(DEV)
    m = torch.zeros((K, K), dtype=torch.int32, device=DEV) if matrix else None
    p = connectome_packed(torch.from_numpy(data).to(DEV), torch.from_numpy(offsets).to(DEV), lab, m, r, pairs=pairs)
    return (None if m is None else m.cpu().numpy()), (None if p is None else p.cpu().numpy())


def _check(data, offsets, labels, r, want=None):
    want = want if want is not None else C.connectome_fast(data, offsets, labels, r)
    for flags in ((True, True), (True, False), (False, True)):
        m, p = _device(data, offsets, labels, r, *flags)
        if flags[0]:
            assert m.dtype == np.int32
            np.testing.assert_array_equal(m, want[0])
        else:
            assert m is None
        if flags[1]:
            assert p.dtype == np.int32
            np.testing.assert_array_equal(p, want[1])
        else:
            assert p is None
    return want


def _walks(rng, n, dims, lo, hi, step=0.7, junk=0.03):
    out = []
    for _ in range(n):
        L = int(rng.randint(lo, hi))
        s = np.cumsum(rng.randn(L, 3) * step, axis=0) + rng.rand(3) * (np.asarray(dims) + 4) - 2
        if junk and L:
            hit = rng.rand(L) < junk
            s[hit, rng.randint(0, 3)] = rng.choice([np.nan, np.inf, -np.inf, -0.5, -0.51, dims[0] - 0.5, -1e30])
        out.append(s.astype(F32))
    return out


def _parcellation(rng, dims, n_labels, density):
    lab = rng.randint(1, n_labels + 1, size=dims).astype(np.int32)
    lab[rng.rand(*dims) >= density] = 0
    return lab


@pytest.mark.parametrize('r', [0.0, 0.5, 1.0, 2.5, 8.0])
@pytest.mark.parametrize('kind', ['dense', 'sparse', 'single'])
def test_random_walks(kind, r):
    rng = np.random.RandomState(int(r * 10) + len(kind))
    dims = (13, 11, 9)
    if kind == 'single':
        lab = np.zeros(dims, np.int32)
        lab[6, 5, 4] = 1
    else:
        lab = _parcellation(rng, dims, 40, 0.8 if kind == 'dense' else 0.03)
    data, offsets = _pack(_walks(rng, 3000, dims, 1, 60) + [np.zeros((0, 3), F32)] * 5)
    want = _check(data, offsets, lab, r)
    assert want[0].sum() > 0


def _face_and_tie_points(dims):
    """Points on and beside every voxel face and grid face, at voxel centres (exact tie distances to the six
    neighbours) and at midpoints between centres (ties between two or four voxels), plus NaN / inf."""
    vals = []
    for d in dims:
        v = [F32(-0.5), np.nextafter(F32(-0.5), F32(-1)), np.nextafter(F32(-0.5), F32(0)), F32(d - 0.5),
             np.nextafter(F32(d - 0.5), F32(0)), np.nextafter(F32(d - 0.5), F32(d)), F32(0.5),
             np.nextafter(F32(0.5), F32(0)), F32(0.0), F32(d - 1), F32(d // 2), F32(d // 2 + 0.5), F32(-2.0),
             F32(d + 1.5), F32(np.nan), F32(np.inf), F32(-np.inf)]
        vals.append(np.asarray(v, dtype=F32))
    return np.stack(np.meshgrid(*vals, indexing='ij'), -1).reshape(-1, 3)


@pytest.mark.parametrize('dims', [(1, 1, 1), (1, 7, 1), (5, 3, 7)])
@pytest.mark.parametrize('r', [0.0, 0.5, 1.0, 2.5, 8.0])
def test_faces_and_ties_on_small_grids(dims, r):
    rng = np.random.RandomState(1)
    pts = _face_and_tie_points(dims)
    rng.shuffle(pts)
    cuts = np.sort(rng.choice(np.arange(1, len(pts)), size=len(pts) // 3, replace=False))
    sl = np.split(pts, cuts)
    for lab in (_parcellation(rng, dims, 5, 0.5), np.arange(1, int(np.prod(dims)) + 1).reshape(dims) % 4):
        data, offsets = _pack(sl + [pts[:1], pts[-1:]])
        want = C.connectome(data, offsets, lab, r)
        _check(data, offsets, lab, r, want)


def test_full_size_grid_with_face_points_and_long_streamlines():
    rng = np.random.RandomState(2)
    dims = (145, 174, 145)
    centres = rng.rand(200, 3) * np.asarray(dims)
    g = np.stack(np.meshgrid(*[np.arange(d) for d in dims], indexing='ij'), -1).reshape(-1, 3)
    from scipy.spatial import cKDTree
    lab = (cKDTree(centres).query(g)[1] + 1).reshape(dims).astype(np.int32)
    lab[rng.rand(*dims) < 0.4] = 0
    long = _walks(rng, 8, dims, 10000, 15000, step=0.5, junk=0.0)
    short = _walks(rng, 20000, dims, 1, 30)
    faces = _face_and_tie_points((145, 174, 145))[::7]
    data, offsets = _pack(long[:4] + short + [faces[i:i + 3] for i in range(0, len(faces), 3)] + long[4:])
    assert max(np.diff(offsets)) >= 10000
    for r in (0.0, 2.5, 8.0):
        _check(data, offsets, lab, r)


def test_a_million_short_streamlines():
    rng = np.random.RandomState(3)
    dims = (64, 70, 58)
    lab = _parcellation(rng, dims, 300, 0.3)
    n = 1_000_000
    lens = rng.randint(0, 6, size=n)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    start = np.repeat(rng.rand(n, 3) * (np.asarray(dims) + 2) - 1, lens, axis=0)
    data = (start + rng.randn(int(offsets[-1]), 3) * 0.7).astype(F32)
    want = _check(data, offsets, lab, 1.0)
    assert int(np.triu(want[0]).sum()) == int((lens > 0).sum())


def test_matrix_accumulates_across_calls_in_any_order():
    from tracktolearn_b200.tracking.postprocess import connectome_packed
    rng = np.random.RandomState(4)
    dims = (17, 15, 16)
    lab = _parcellation(rng, dims, 30, 0.2)
    sl = _walks(rng, 6000, dims, 0, 80)
    whole, _ = _device(*_pack(sl), lab, 2.0)
    labels = torch.from_numpy(lab).to(DEV)
    m = torch.zeros(whole.shape, dtype=torch.int32, device=DEV)
    for part in (sl[3001:], sl[:1234], sl[1234:3001]):
        d, o = _pack(part)
        connectome_packed(torch.from_numpy(d).to(DEV), torch.from_numpy(o).to(DEV), labels, m, 2.0)
    assert m.cpu().numpy().tobytes() == whole.tobytes()
    rev, _ = _device(*_pack(sl[::-1]), lab, 2.0)
    assert rev.tobytes() == whole.tobytes()


def test_every_end_unlabelled_counts_exactly_in_zero_zero():
    """The worst contention: every streamline adds to the same cell."""
    rng = np.random.RandomState(5)
    dims = (30, 31, 29)
    n = 1_000_000
    lens = rng.randint(0, 4, size=n)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = (rng.rand(int(offsets[-1]), 3) * 40 - 5).astype(F32)
    lab = np.zeros(dims, np.int32)
    for r in (0.0, 3.0):
        m, p = _device(data, offsets, lab, r, K=3)
        assert m[0, 0] == int((lens > 0).sum()) and int(m.sum()) == m[0, 0]
        assert not p.any()


def test_no_write_outside_the_matrix_or_the_pairs():
    """The matrix and the pairs are carved out of larger allocations with 4 KB of 0xA5 on each side; label
    values >= K and < 0 are passed straight to the ABI and must read as 0."""
    from tracktolearn_b200 import _lib
    from tracktolearn_b200.environments.tracking_env import GUARD_BYTES, GUARD_FILL
    lib = _lib.load()
    rng = np.random.RandomState(6)
    for dims, K in (((1, 1, 1), 1), ((1, 9, 1), 2), ((3, 1, 5), 3), ((7, 5, 3), 5), ((11, 13, 1), 7)):
        pts = _face_and_tie_points(dims)
        rng.shuffle(pts)
        cuts = np.sort(rng.choice(np.arange(1, len(pts)), size=len(pts) // 4, replace=False))
        data, offsets = _pack(np.split(pts, cuts))
        n = len(offsets) - 1
        lab = rng.randint(-3, 3 * K + 2, size=dims).astype(np.int32)
        lab[rng.rand(*dims) < 0.3] = 1 << 30
        for r in (0.0, 8.0):
            want = C.connectome(data, offsets, lab, r, K)
            raws, views = [], []
            for nbytes in (4 * K * K, 8 * n):
                raw = torch.full((nbytes + 2 * GUARD_BYTES,), GUARD_FILL, dtype=torch.uint8, device=DEV)
                v = raw[GUARD_BYTES:GUARD_BYTES + nbytes].view(torch.int32)
                v.zero_()
                raws.append((raw, nbytes))
                views.append(v)
            d, o = torch.from_numpy(data).to(DEV), torch.from_numpy(offsets).to(DEV)
            t = torch.from_numpy(lab).to(DEV)
            _lib.check(lib.ttl_connectome(_lib.ptr(d), _lib.ptr(o), n, _lib.ptr(t), *dims, K, r, _lib.ptr(views[0]),
                                          _lib.ptr(views[1]), _lib.stream_ptr(DEV)), 'ttl_connectome')
            torch.cuda.synchronize()
            for raw, nbytes in raws:
                assert int((raw[:GUARD_BYTES] != GUARD_FILL).sum()) == 0, dims
                assert int((raw[GUARD_BYTES + nbytes:] != GUARD_FILL).sum()) == 0, dims
            np.testing.assert_array_equal(views[0].cpu().numpy().reshape(K, K), want[0])
            np.testing.assert_array_equal(views[1].cpu().numpy().reshape(n, 2), want[1])


# ------------------------------------------------------------------------------------ Tracker.track_to_file

def _shell_labels(mask, n_labels=40, seed=0):
    """A synthetic parcellation: labels from the nearest of n_labels random centres, on the voxels within two
    voxels outside the tracking mask and on a thin layer inside its border."""
    from scipy import ndimage
    from scipy.spatial import cKDTree
    inside = np.asarray(mask) > 0.5
    shell = ndimage.binary_dilation(inside, iterations=2) & ~ndimage.binary_erosion(inside, iterations=1)
    rng = np.random.RandomState(seed)
    idx = np.argwhere(shell)
    centres = idx[rng.choice(len(idx), n_labels, replace=False)]
    lab = np.zeros(inside.shape, np.int32)
    lab[shell] = cKDTree(centres).query(idx)[1] + 1
    return lab


def test_track_to_file_connectivity(tmp_path):
    from tests.test_tracker_gpu import _setup
    from tracktolearn_b200.io.streamlines import read_trk
    from tracktolearn_b200.tracking.postprocess import lengths_packed
    from tracktolearn_b200.tracking.tracker import Tracker
    env, alg, sub, seeds, _ = _setup(precision='fp16')
    seeds = np.array(env.seeds, copy=True)
    dims = tuple(sub['mask'].shape[:3])
    lab = _shell_labels(sub['mask'])
    labels = torch.from_numpy(lab).to(DEV)
    radius_mm = 2.0                              # 2 voxels of 1 mm

    def tracker(compress=0.0):
        env.seeds = seeds.copy()
        np.random.seed(0)
        return Tracker(alg, 256, min_length=5, max_length=200, save_seeds=True, compress=compress)

    def run(name, compress=0.0, conn=True, save_labels=False, **kw):
        t = tracker(compress)
        path = str(tmp_path / name)
        if conn or save_labels:
            kw.update(labels=labels, connectivity_radius=radius_mm, save_labels=save_labels)
        if conn:
            kw['connectivity_path'] = path.rsplit('.', 1)[0] + '.npy'
        n = t.track_to_file(env, path, dims, (1.0, 1.0, 1.0), **kw)
        return open(path, 'rb').read(), n, (np.load(kw['connectivity_path']) if conn else None), \
            t.connectome_unlabelled, path

    trk, n, m, unl, _ = run('a.trk')
    assert m.dtype == np.int32 and m.shape == (int(lab.max()) + 1,) * 2

    # the restatement on the length-kept voxel-space streamlines of a separate track_packed run
    t = tracker()
    np.random.shuffle(env.seeds)
    kept = []
    for batch in t.track_packed(env):
        lens = lengths_packed(batch.data, batch.offsets).cpu().numpy()
        for i in np.nonzero((lens >= 5.0) & (lens <= 200.0))[0]:
            kept.append(batch.data[batch.offsets[i]:batch.offsets[i + 1]])
    assert len(kept) == n > 100
    want_m, want_p = C.connectome_fast(*_pack(kept), lab, radius_mm)
    np.testing.assert_array_equal(m, want_m)
    assert unl == int((want_p == 0).sum())
    assert int(np.triu(m).sum()) == n

    # the per-streamline labels in the .trk
    lab_trk, n2, m2, _, path = run('l.trk', save_labels=True)
    _, _, hdr = read_trk(path)
    assert hdr['property_names'][-2:] == ['start_label', 'end_label'] and n2 == n
    np.testing.assert_array_equal(hdr['properties'][:, -2:].astype(np.int32), want_p)
    np.testing.assert_array_equal(m2, m)
    only, n3, _, _, path = run('o.trk', conn=False, save_labels=True)
    assert only == lab_trk

    # the tractogram does not change with a matrix, and the matrix does not change with --compress
    assert run('b.trk', conn=False)[0] == trk
    assert run('a.tck')[0] == run('b.tck', conn=False)[0]
    comp = run('c.trk', compress=0.2)
    assert comp[0] != trk and comp[1] == n and comp[2].tobytes() == m.tobytes()
    assert run('c2.trk', compress=0.2, conn=False)[0] == comp[0]


# ------------------------------------------------------------------------------------ command line

def test_ttl_track_connectivity_and_ttl_connectivity(tmp_path, capsys):
    from tests.test_oracle_filter_gpu import _subject, _track
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.io.streamlines import read_trk
    from tracktolearn_b200.runners.ttl_connectivity import main as conn_main
    from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
    agent, affine = _subject(tmp_path)
    lab = _shell_labels(nifti.load(str(tmp_path / 'mask.nii.gz')).data, n_labels=25, seed=1)
    nifti.save(str(tmp_path / 'labels.nii.gz'), lab.astype(np.int16), affine)
    radius_mm = 2.5                              # 2 voxels of 1.25 mm
    outs = {}
    for n_actor in (500, 173):
        c = str(tmp_path / ('c%d.npy' % n_actor))
        capsys.readouterr()
        trk = _track(tmp_path, agent, 't%d.trk' % n_actor, '--n_actor', str(n_actor), '--noise_rng', 'device',
                     '--noise', '0.1', '--in_labels', str(tmp_path / 'labels.nii.gz'), '--out_connectivity', c,
                     '--connectivity_radius', str(radius_mm), '--save_connectivity_labels')
        assert 'have no label' in capsys.readouterr().out
        outs[n_actor] = (open(trk, 'rb').read(), open(c, 'rb').read(), trk, c)
    assert outs[500][:2] == outs[173][:2]
    trk, c = outs[500][2:]
    m = np.load(c)
    assert m.dtype == np.int32 and int(m.sum()) > 0

    # the standalone command on the .trk: equal, except for streamlines with an end within float32 round-trip
    # distance of a voxel face or of the radius sphere
    post = str(tmp_path / 'post.npy')
    capsys.readouterr()
    conn_main([trk, str(tmp_path / 'labels.nii.gz'), post, '--radius', str(radius_mm)])
    assert 'Wrote' in capsys.readouterr().out
    m_post = np.load(post)
    data, offsets, hdr = read_trk(trk)
    pairs_track = hdr['properties'][:, -2:].astype(np.int64)
    vox = voxel_points(data, 'trk', hdr['voxel_sizes'])
    r = radius_mm / 1.25
    pairs_post = C.connectome_fast(vox, offsets, lab, r)[1].astype(np.int64)
    ends = np.concatenate((vox[offsets[:-1]], vox[offsets[1:] - 1]))
    # an end is sensitive when moving it by a few float32 ulps on any axis can change its label
    base = C.end_labels_fast(ends, lab, r)
    sensitive = np.zeros(len(ends), bool)
    for axis in range(3):
        for sign in (-1, 1):
            moved = ends.copy()
            moved[:, axis] = moved[:, axis] + sign * 8 * np.spacing(np.abs(moved[:, axis]) + F32(1))
            sensitive |= C.end_labels_fast(moved.astype(F32), lab, r) != base
    n = len(offsets) - 1
    excluded = sensitive[:n] | sensitive[n:]
    print('streamlines with an end within float32 round-trip distance of a face or the sphere: %d'
          % int(excluded.sum()))
    K = m.shape[0]

    def cells(p):
        a, b = p[:, 0], p[:, 1]
        return np.bincount(np.concatenate((a * K + b, (b * K + a)[a != b])), minlength=K * K).reshape(K, K)
    np.testing.assert_array_equal(cells(pairs_track), m)
    np.testing.assert_array_equal(cells(pairs_post), m_post)
    np.testing.assert_array_equal(pairs_post[~excluded], pairs_track[~excluded])
    np.testing.assert_array_equal(m_post - cells(pairs_post[excluded]), m - cells(pairs_track[excluded]))
