"""Tractometry on the device: ttl_sample_metrics against the restatement of tests/tractometry_oracle.py, the bits of
a streamline's mean across batches, ttl_connectome_sums against int64 numpy sums, guard bands around every
output, Tracker.track_to_file with metrics, and ttl_track.py against ttl_tractometry.py and ttl_connectivity.py."""
import numpy as np
import pytest
import torch

from tests import connectome_oracle as CO
from tests import maps_oracle as M
from tests import tractometry_oracle as T

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
F32 = np.float32


def _pack(streamlines):
    lens = [len(s) for s in streamlines]
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    data = np.concatenate([np.asarray(s, dtype=F32).reshape(-1, 3) for s in streamlines])
    return data.astype(F32), offsets


def _device_means(data, offsets, vol):
    from tracktolearn_b200.tracking.postprocess import sample_metrics_packed
    v = torch.from_numpy(np.ascontiguousarray(vol, dtype=F32)).to(DEV)
    means, skipped = sample_metrics_packed(torch.from_numpy(data).to(DEV), torch.from_numpy(offsets).to(DEV), v)
    return means.cpu().numpy(), skipped


def _check(data, offsets, vol):
    """Equal to the restatement, or within 1 ulp where the fp64 sums differ by summation order only."""
    got, skipped = _device_means(data, offsets, vol)
    want, want_skipped = T.sample_means(data, offsets, vol)
    assert got.dtype == F32 and got.shape == want.shape
    assert skipped == want_skipped == M.tract_maps_fast(data, offsets, vol.shape[:3])[2]
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    diff = np.abs(got[ok].view(np.int32).astype(np.int64) - want[ok].view(np.int32).astype(np.int64))
    assert int(diff.max(initial=0)) <= 1, int(diff.max())
    return got, want


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


def _face_points(dims):
    vals = []
    for d in dims:
        v = [F32(-0.5), np.nextafter(F32(-0.5), F32(-1)), np.nextafter(F32(-0.5), F32(0)), F32(d - 0.5),
             np.nextafter(F32(d - 0.5), F32(0)), F32(0.5), F32(0.0), F32(d - 1), np.nextafter(F32(d - 1), F32(d)),
             F32(d // 2 + 0.5), F32(np.nan), F32(np.inf)]
        vals.append(np.asarray(v, dtype=F32))
    return np.stack(np.meshgrid(*vals, indexing='ij'), -1).reshape(-1, 3)


@pytest.mark.parametrize('C', [1, 2, 3, 4, 5, 6, 7, 8])
def test_random_walks_and_face_points(C):
    rng = np.random.RandomState(C)
    dims = (13, 11, 9)
    vol = (rng.randn(*dims, C) * 10 ** rng.uniform(-3, 3, size=C)).astype(F32)
    faces = _face_points(dims)
    rng.shuffle(faces)
    sl = _walks(rng, 3000, dims, 0, 90) + np.split(faces, np.arange(7, len(faces), 7)) + [np.zeros((0, 3), F32)]
    got, _ = _check(*_pack(sl), vol)
    assert np.isfinite(got).sum() > 1000


def test_long_streamlines_and_a_full_size_grid():
    rng = np.random.RandomState(10)
    dims = (145, 174, 145)
    vol = rng.rand(*dims, 2).astype(F32)
    sl = _walks(rng, 6, dims, 10000, 15000, step=0.5, junk=0.001) + _walks(rng, 20000, dims, 1, 30)
    data, offsets = _pack(sl)
    assert max(np.diff(offsets)) >= 10000
    _check(data, offsets, vol)


def test_a_million_short_streamlines():
    rng = np.random.RandomState(11)
    dims = (64, 70, 58)
    vol = (rng.rand(*dims, 3) * 4 - 2).astype(F32)
    n = 1_000_000
    lens = rng.randint(0, 6, size=n)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    start = np.repeat(rng.rand(n, 3) * (np.asarray(dims) + 2) - 1, lens, axis=0)
    data = (start + rng.randn(int(offsets[-1]), 3) * 0.7).astype(F32)
    _check(data, offsets, vol)


def test_a_streamlines_means_do_not_depend_on_its_batch():
    rng = np.random.RandomState(12)
    dims = (17, 15, 16)
    vol = rng.randn(*dims, 5).astype(F32)
    sl = _walks(rng, 5000, dims, 0, 200)
    whole, _ = _device_means(*_pack(sl), vol)
    perm = rng.permutation(len(sl))
    shuffled, _ = _device_means(*_pack([sl[i] for i in perm]), vol)
    assert shuffled.tobytes() == whole[perm].tobytes()
    parts = [_device_means(*_pack(sl[a:b]), vol)[0] for a, b in ((0, 1), (1, 1234), (1234, 4999), (4999, 5000))]
    assert np.concatenate(parts).tobytes() == whole.tobytes()


# ------------------------------------------------------------------------------------ edge sums

def _device_sums(pairs, values, shifts, K, sums=None, counts=None):
    from tracktolearn_b200.tracking.postprocess import connectome_sums_packed
    C = values.shape[1]
    s = torch.zeros((C, K, K), dtype=torch.int64, device=DEV) if sums is None else sums
    c = torch.zeros((C, K, K), dtype=torch.int32, device=DEV) if counts is None else counts
    connectome_sums_packed(torch.from_numpy(np.ascontiguousarray(pairs, dtype=np.int32)).to(DEV),
                           torch.from_numpy(np.ascontiguousarray(values, dtype=F32)).to(DEV), shifts, s, c)
    return s, c


def test_connectome_sums_match_int64_numpy_and_accumulate():
    rng = np.random.RandomState(13)
    n, K = 200000, 97
    pairs = rng.randint(-3, K + 5, size=(n, 2)).astype(np.int32)
    values = np.stack([rng.rand(n), rng.randn(n) * 1e4, rng.rand(n) * 1e-6, rng.rand(n) * 250], 1).astype(F32)
    values[rng.rand(n) < 0.1, 0] = np.nan
    values[:5, 3] = [np.nan, np.inf, -np.inf, 0.0, -0.0]
    shifts = [T.metric_shift(1.0), T.metric_shift(np.abs(values[:, 1]).max()), T.metric_shift(1e-6),
              T.metric_shift(250.0)]
    want = T.edge_sums(pairs, values, shifts, K)
    s, c = _device_sums(pairs, values, shifts, K)
    assert s.cpu().numpy().tobytes() == want[0].tobytes() and c.cpu().numpy().tobytes() == want[1].tobytes()
    s, c = (torch.zeros((4, K, K), dtype=dt, device=DEV) for dt in (torch.int64, torch.int32))
    perm = rng.permutation(n)
    for part in np.array_split(perm, 5):
        _device_sums(pairs[part], values[part], shifts, K, s, c)
    assert s.cpu().numpy().tobytes() == want[0].tobytes() and c.cpu().numpy().tobytes() == want[1].tobytes()


def test_every_value_in_zero_zero_sums_exactly():
    """The worst contention: every streamline adds to the same cell."""
    rng = np.random.RandomState(14)
    n = 2_000_000
    values = (rng.rand(n, 2) * [1.0, 300.0]).astype(F32)
    shifts = [T.metric_shift(1.0), T.metric_shift(300.0)]
    s, c = _device_sums(np.zeros((n, 2), np.int32), values, shifts, 3)
    q = np.rint(np.ldexp(values.astype(np.float64), np.asarray(shifts))).astype(np.int64)
    assert s.cpu().numpy()[:, 0, 0].tolist() == q.sum(0).tolist()
    assert c.cpu().numpy()[:, 0, 0].tolist() == [n, n] and int(c.sum()) == 2 * n


def test_no_write_outside_the_means_sums_or_counts():
    """Every output is carved out of a larger allocation with 4 KB of 0xA5 on each side."""
    from tracktolearn_b200 import _lib
    from tracktolearn_b200.environments.tracking_env import GUARD_BYTES, GUARD_FILL
    lib = _lib.load()
    rng = np.random.RandomState(15)

    def guarded(nbytes, dtype):
        raw = torch.full((nbytes + 2 * GUARD_BYTES,), GUARD_FILL, dtype=torch.uint8, device=DEV)
        v = raw[GUARD_BYTES:GUARD_BYTES + nbytes].view(dtype)
        v.zero_()
        return raw, nbytes, v

    def intact(raw, nbytes):
        return int((raw[:GUARD_BYTES] != GUARD_FILL).sum()) == 0 and \
            int((raw[GUARD_BYTES + nbytes:] != GUARD_FILL).sum()) == 0

    for dims, C, K in (((1, 1, 1), 1, 1), ((1, 9, 1), 3, 2), ((3, 1, 5), 8, 3), ((7, 5, 3), 5, 7)):
        pts = _face_points(dims)
        rng.shuffle(pts)
        data, offsets = _pack(np.split(pts, np.sort(rng.choice(np.arange(1, len(pts)), len(pts) // 4, False))))
        n = len(offsets) - 1
        vol = rng.randn(*dims, C).astype(F32)
        raw_m, nb_m, means = guarded(4 * n * C, torch.float32)
        raw_k, nb_k, skipped = guarded(8, torch.int64)
        d, o, v = (torch.from_numpy(x).to(DEV) for x in (data, offsets, vol))
        _lib.check(lib.ttl_sample_metrics(_lib.ptr(d), _lib.ptr(o), n, _lib.ptr(v), C, *dims, _lib.ptr(means),
                                          _lib.ptr(skipped), _lib.stream_ptr(DEV)), 'ttl_sample_metrics')
        raw_s, nb_s, sums = guarded(8 * C * K * K, torch.int64)
        raw_c, nb_c, counts = guarded(4 * C * K * K, torch.int32)
        pairs = rng.randint(-2, K + 3, size=(n, 2)).astype(np.int32)
        pairs[rng.rand(n) < 0.2] = 1 << 30
        p = torch.from_numpy(pairs).to(DEV)
        shifts = np.full(C, 20, np.int32)
        _lib.check(lib.ttl_connectome_sums(_lib.ptr(p), n, _lib.ptr(means), C, K, shifts.ctypes.data,
                                           _lib.ptr(sums), _lib.ptr(counts), _lib.stream_ptr(DEV)),
                   'ttl_connectome_sums')
        torch.cuda.synchronize()
        for raw, nb in ((raw_m, nb_m), (raw_k, nb_k), (raw_s, nb_s), (raw_c, nb_c)):
            assert intact(raw, nb), (dims, C, K)
        want_m, want_k = T.sample_means(data, offsets, vol)
        got_m = means.cpu().numpy().reshape(n, C)
        np.testing.assert_array_equal(np.isnan(got_m), np.isnan(want_m))
        np.testing.assert_allclose(got_m, want_m, rtol=2e-7, atol=0)
        assert int(skipped.item()) == want_k
        ws, wc = T.edge_sums(pairs, got_m, shifts, K)
        assert sums.cpu().numpy().reshape(C, K, K).tobytes() == ws.tobytes()
        assert counts.cpu().numpy().reshape(C, K, K).tobytes() == wc.tobytes()


# ------------------------------------------------------------------------------------ Tracker.track_to_file

def _shell_labels(mask, n_labels=40, seed=0):
    from tests.test_connectome_gpu import _shell_labels as shell
    return shell(mask, n_labels, seed)


def test_track_to_file_tractometry(tmp_path):
    from tests.test_tracker_gpu import _setup
    from tracktolearn_b200.io.streamlines import read_trk
    from tracktolearn_b200.tracking.postprocess import edge_means, lengths_packed
    from tracktolearn_b200.tracking.tracker import Tracker
    env, alg, sub, seeds, _ = _setup(precision='fp16')
    seeds = np.array(env.seeds, copy=True)
    dims = tuple(sub['mask'].shape[:3])
    rng = np.random.RandomState(16)
    vol = np.stack([rng.rand(*dims), rng.randn(*dims) * 50], -1).astype(F32)
    metrics = torch.from_numpy(vol).to(DEV)
    lab = _shell_labels(sub['mask'])
    labels = torch.from_numpy(lab).to(DEV)
    K = int(lab.max()) + 1

    def run(name, compress=0.0, tract=True, **kw):
        env.seeds = seeds.copy()
        np.random.seed(0)
        t = Tracker(alg, 256, min_length=5, max_length=200, save_seeds=True, compress=compress)
        path = str(tmp_path / name)
        stem = path.rsplit('.', 1)[0]
        if tract:
            kw.update(labels=labels, connectivity_path=stem + '.npy', metrics=metrics, metric_names=['FA', 'MD'],
                      save_metric_means=name.endswith('.trk'), metric_connectivity_prefix=stem + '_',
                      length_connectivity_path=stem + '_len.npy')
        n = t.track_to_file(env, path, dims, (1.0, 1.0, 1.0), **kw)
        mats = None
        if tract:
            mats = [open(f, 'rb').read() for f in (stem + '.npy', stem + '_FA.npy', stem + '_MD.npy', stem + '_len.npy')]
        return open(path, 'rb').read(), n, mats, path, t.metrics_unsampled

    trk, n, mats, path, unsampled = run('a.trk')
    _, _, hdr = read_trk(path)
    assert hdr['property_names'][-2:] == ['mean_FA', 'mean_MD']
    means_trk = hdr['properties'][:, -2:]

    # the restatement on the length-kept voxel-space streamlines of a separate track_packed run
    env.seeds = seeds.copy()
    np.random.seed(0)
    t = Tracker(alg, 256, min_length=5, max_length=200, save_seeds=True)
    np.random.shuffle(env.seeds)
    kept, kept_len = [], []
    for batch in t.track_packed(env):
        lens = lengths_packed(batch.data, batch.offsets).cpu().numpy()
        for i in np.nonzero((lens >= 5.0) & (lens <= 200.0))[0]:
            kept.append(batch.data[batch.offsets[i]:batch.offsets[i + 1]])
            kept_len.append(lens[i])
    assert len(kept) == n > 100
    data, offsets = _pack(kept)
    want, _ = T.sample_means(data, offsets, vol)
    d = np.abs(means_trk.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert int(d[~np.isnan(want)].max()) <= 1 and np.array_equal(np.isnan(means_trk), np.isnan(want))
    assert unsampled == int(np.isnan(want[:, 0]).sum())

    # the weighted matrices from the restatement's values and the end labels
    count = np.load(str(tmp_path / 'a.npy'))
    _, pairs = CO.connectome_fast(data, offsets, lab, 0.0)
    length_mm = (np.asarray(kept_len) * 1.0).astype(F32)
    shifts = [T.metric_shift(np.abs(vol[..., c]).max()) for c in range(2)] + [T.metric_shift(200 * 1.001)]
    sums, counts = T.edge_sums(pairs, np.concatenate([means_trk, length_mm[:, None]], 1), shifts, K)
    for c in range(3):
        np.testing.assert_array_equal(counts[c], count)
    mean = edge_means(sums, counts, shifts)
    for c, f in enumerate(('a_FA.npy', 'a_MD.npy', 'a_len.npy')):
        got = np.load(str(tmp_path / f))
        assert got.dtype == np.float64 and got.shape == (K, K)
        assert got.tobytes() == mean[c].tobytes()

    # the tractogram does not change with tractometry, and tractometry does not change with --compress
    assert run('b.trk', tract=False)[0] != trk        # the means are extra properties
    assert run('c.tck')[0] == run('d.tck', tract=False)[0]
    comp = run('e.trk', compress=0.2)
    assert comp[1] == n and comp[2][1:] == mats[1:] and comp[2][0] == mats[0]
    _, _, hdr_c = read_trk(comp[3])
    assert hdr_c['properties'][:, -2:].tobytes() == means_trk.tobytes()


# ------------------------------------------------------------------------------------ command line

def test_ttl_track_tractometry_and_the_standalone_commands(tmp_path, capsys):
    from tests.test_oracle_filter_gpu import _subject, _track
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.io.streamlines import read_trk
    from tracktolearn_b200.runners.ttl_connectivity import main as conn_main
    from tracktolearn_b200.runners.ttl_oracle_filter import voxel_points
    from tracktolearn_b200.runners.ttl_tractometry import main as tm_main
    from tracktolearn_b200.tracking.postprocess import edge_means
    agent, affine = _subject(tmp_path)
    mask = nifti.load(str(tmp_path / 'mask.nii.gz')).data
    lab = _shell_labels(mask, n_labels=25, seed=1)
    nifti.save(str(tmp_path / 'labels.nii.gz'), lab.astype(np.int16), affine)
    rng = np.random.RandomState(17)
    fa = rng.rand(*lab.shape).astype(F32)
    md = (rng.rand(*lab.shape) * 3e-3).astype(np.float64)
    nifti.save(str(tmp_path / 'fa.nii.gz'), fa, affine)
    nifti.save(str(tmp_path / 'md.nii.gz'), md, affine)
    outs = {}
    for n_actor in (500, 173):
        pre = str(tmp_path / ('w%d_' % n_actor))
        ln = str(tmp_path / ('len%d.npy' % n_actor))
        capsys.readouterr()
        trk = _track(tmp_path, agent, 't%d.trk' % n_actor, '--n_actor', str(n_actor), '--noise_rng', 'device',
                     '--noise', '0.1', '--in_labels', str(tmp_path / 'labels.nii.gz'),
                     '--out_connectivity', str(tmp_path / ('c%d.npy' % n_actor)), '--save_connectivity_labels',
                     '--in_metric', 'FA', str(tmp_path / 'fa.nii.gz'), '--in_metric', 'MD', str(tmp_path / 'md.nii.gz'),
                     '--save_metric_means', '--out_connectivity_metrics', pre, '--out_connectivity_length', ln)
        assert 'mean FA connectivity matrix' in capsys.readouterr().out
        outs[n_actor] = [open(f, 'rb').read() for f in (trk, pre + 'FA.npy', pre + 'MD.npy', ln)] + [trk, pre, ln]
    assert outs[500][:4] == outs[173][:4]
    trk, pre, ln = outs[500][4:]
    data, offsets, hdr = read_trk(trk)
    assert hdr['property_names'][-4:] == ['start_label', 'end_label', 'mean_FA', 'mean_MD']
    props = hdr['properties']

    # ttl_tractometry.py on the written .trk: the same means up to the float32 round trip of the points
    post = str(tmp_path / 'means.npy')
    tm_main([trk, post, '--in_metric', 'FA', str(tmp_path / 'fa.nii.gz'), '--in_metric', 'MD',
             str(tmp_path / 'md.nii.gz')])
    got = np.load(post)
    assert got.dtype == F32 and got.shape == (len(offsets) - 1, 2)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(props[:, -2:]))
    ok = ~np.isnan(got)
    scale = np.array([1.0, 3e-3])[None, :].repeat(len(got), 0)
    assert np.all(np.abs(got - props[:, -2:])[ok] <= 1e-4 * scale[ok])

    # ttl_connectivity.py --out_metrics / --out_length: equal on the streamlines whose end labels do not move
    # under an 8-ulp perturbation, recomputed from the same per-streamline values
    conn_main([trk, str(tmp_path / 'labels.nii.gz'), str(tmp_path / 'post.npy'), '--in_metric', 'FA',
               str(tmp_path / 'fa.nii.gz'), '--in_metric', 'MD', str(tmp_path / 'md.nii.gz'),
               '--out_metrics', str(tmp_path / 'p_'), '--out_length', str(tmp_path / 'plen.npy')])
    vox = voxel_points(data, 'trk', hdr['voxel_sizes'])
    pairs_post = CO.connectome_fast(vox, offsets, lab, 0.0)[1]
    pairs_track = props[:, -4:-2].astype(np.int64)
    ends = np.concatenate((vox[offsets[:-1]], vox[offsets[1:] - 1]))
    base = CO.end_labels_fast(ends, lab, 0.0)
    sensitive = np.zeros(len(ends), bool)
    for axis in range(3):
        for sign in (-1, 1):
            moved = ends.copy()
            moved[:, axis] = moved[:, axis] + sign * 8 * np.spacing(np.abs(moved[:, axis]) + F32(1))
            sensitive |= CO.end_labels_fast(moved.astype(F32), lab, 0.0) != base
    n = len(offsets) - 1
    keep = ~(sensitive[:n] | sensitive[n:])
    np.testing.assert_array_equal(pairs_post[keep], pairs_track[keep])
    K = lab.max() + 1
    for f_track, f_post, c in ((pre + 'FA.npy', 'p_FA.npy', 0), (pre + 'MD.npy', 'p_MD.npy', 1)):
        m_track, m_post = np.load(f_track), np.load(str(tmp_path / f_post))
        if keep.all():
            np.testing.assert_allclose(m_post, m_track, rtol=1e-4, atol=1e-4 * scale[0, c], equal_nan=True)
        # both from the same kept streamlines' values: the means over kept streamlines agree
        bound = [np.abs(fa).max(), np.abs(md).max()][c]
        shift = [T.metric_shift(bound)]
        a = edge_means(*T.edge_sums(pairs_track[keep], props[keep, -2 + c:][:, :1], shift, K), shift)[0]
        b = edge_means(*T.edge_sums(pairs_post[keep], got[keep, c:c + 1], shift, K), shift)[0]
        np.testing.assert_allclose(b, a, rtol=1e-4, atol=1e-4 * scale[0, c], equal_nan=True)
    m_len_track, m_len_post = np.load(ln), np.load(str(tmp_path / 'plen.npy'))
    np.testing.assert_array_equal(np.isnan(m_len_track), np.load(str(tmp_path / 'c500.npy')) == 0)
    if keep.all():
        np.testing.assert_allclose(m_len_post, m_len_track, rtol=1e-5, equal_nan=True)
