"""Oracle filtering on the device: the ordered select / gather kernels against a numpy restatement, batch
independence of the scores, Tracker.track_to_file with an oracle, ttl_track.py --oracle_checkpoint and
ttl_oracle_filter.py."""
import os

import numpy as np
import pytest
import torch

from tracktolearn_b200 import synthetic

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
FP16_TOL = 5e-3          # fp16 tensor-core tier against the fp32 arithmetic, on sigmoid outputs


def _oracle(ck, precision='fp16'):
    from tracktolearn_b200.oracles.oracle import OracleSingleton
    OracleSingleton.clear()
    return OracleSingleton(ck, DEV, batch_size=4096, precision=precision)


def _packed(lens, rng):
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    return rng.randn(int(offsets[-1]), 3).astype(np.float32), offsets


def _select_np(data, offsets, keep=None, scores=None, threshold=0.0):
    k = np.ones(len(offsets) - 1, dtype=bool)
    if keep is not None:
        k &= keep.astype(bool)
    if scores is not None:
        k &= scores >= np.float32(threshold)
    idx = np.nonzero(k)[0]
    new_off = np.concatenate(([0], np.cumsum(np.diff(offsets)[idx]))).astype(np.int64)
    return data[np.repeat(k, np.diff(offsets))], new_off, idx


def _check_select(data, offsets, keep=None, scores=None, threshold=0.0):
    from tracktolearn_b200.tracking.postprocess import select_packed
    t = (lambda a: None if a is None else torch.from_numpy(a).to(DEV))
    got = select_packed(t(data), t(offsets), keep=t(keep), scores=t(scores), threshold=threshold)
    want = _select_np(data, offsets, keep, scores, threshold)
    for g, w in zip(got, want):
        g = g.cpu().numpy()
        assert g.shape == w.shape, (g.shape, w.shape)
        np.testing.assert_array_equal(g, w)
        if g.dtype == np.float32:
            assert g.tobytes() == w.tobytes()
    return len(want[2])


def test_select_and_gather_match_numpy():
    rng = np.random.RandomState(0)
    # empty input
    assert _check_select(np.zeros((0, 3), np.float32), np.zeros((1,), np.int64)) == 0
    data, offsets = _packed(rng.randint(1, 50, size=300), rng)
    n = len(offsets) - 1
    assert _check_select(data, offsets, keep=np.zeros(n, np.uint8)) == 0                 # none kept
    assert _check_select(data, offsets) == n                                              # all kept
    assert _check_select(data, offsets, keep=np.ones(n, np.uint8)) == n
    ones, offs1 = _packed(np.ones(50, np.int64), rng)                                     # 1-point streamlines
    assert _check_select(ones, offs1, keep=(np.arange(50) % 3 == 0).astype(np.uint8)) == 17
    scores = rng.rand(n).astype(np.float32)
    scores[::7] = np.nan                                                                  # never kept
    scores[1::7] = np.float32(0.5)                                                        # == threshold: kept
    m = _check_select(data, offsets, scores=scores, threshold=0.5)
    assert m == int((scores >= 0.5).sum()) and m > 0
    _check_select(data, offsets, keep=(rng.rand(n) < 0.5).astype(np.uint8), scores=scores, threshold=0.5)
    _check_select(data, offsets, scores=np.full(n, np.nan, np.float32), threshold=0.0)
    # 100 000 random-length streamlines, both predicates
    data, offsets = _packed(rng.randint(1, 120, size=100000), rng)
    keep = (rng.rand(100000) < 0.7).astype(np.uint8)
    scores = rng.rand(100000).astype(np.float32)
    _check_select(data, offsets, keep=keep)
    _check_select(data, offsets, keep=keep, scores=scores, threshold=0.3)


@pytest.mark.parametrize('precision', ['fp16', 'fp32'])
def test_scores_do_not_depend_on_the_batch(precision):
    """A streamline's score is the same bits in the full set, in reversed order and in two halves: the
    filtered tractogram then does not depend on the GPU count or --n_actor."""
    rng = np.random.RandomState(1)
    sl = synthetic.random_streamlines(5000, rng, min_pts=2, max_pts=200)
    model = _oracle(synthetic.oracle_checkpoint(seed=78), precision)

    def score(items):
        lens = np.asarray([len(s) for s in items])
        off = torch.from_numpy(np.concatenate(([0], np.cumsum(lens))).astype(np.int64)).to(DEV)
        pts = torch.from_numpy(np.concatenate(items).astype(np.float32)).to(DEV)
        return model.predict_device(pts, off, distributed=False).cpu().numpy()
    full = score(sl)
    assert full.tobytes() == score(sl[::-1])[::-1].tobytes()
    assert full.tobytes() == np.concatenate([score(sl[:1777]), score(sl[1777:])]).tobytes()


# ------------------------------------------------------------------------------------ Tracker.track_to_file

def _calibrated_checkpoint(pts, off):
    """A synthetic checkpoint whose head is rescaled so that the scores of these streamlines are centred
    on 0.5 with a logit spread of 2 (the synthetic checkpoints alone score everything near 0.58)."""
    ck = synthetic.oracle_checkpoint(n_head=4, n_layers=4, seed=78)
    sd = ck['state_dict']
    sd['embedding.0.weight'] = sd['embedding.0.weight'] * 4.0
    p = _oracle(ck, 'fp32').predict_device(pts, off, distributed=False).double().cpu().numpy()
    logit = np.log(p / (1 - p))
    gain = 2.0 / max(float(logit.std()), 1e-6)
    sd['head.bias'] = sd['head.bias'] * gain - float(gain * np.median(logit))
    sd['head.weight'] = sd['head.weight'] * gain
    return ck


def _records(path):
    from tracktolearn_b200.io.streamlines import read_tck, read_trk
    raw = open(path, 'rb').read()
    out = (read_trk if path.endswith('.trk') else read_tck)(path, spans=True)
    return [raw[s:e] for s, e in zip(*out[3])], out[2]


def test_track_to_file_with_an_oracle(tmp_path):
    from tests.test_tracker_gpu import _setup
    from tracktolearn_b200.tracking.postprocess import lengths_packed
    from tracktolearn_b200.tracking.tracker import Tracker
    env, alg, sub, seeds, _ = _setup(precision='fp16')
    seeds = np.array(env.seeds, copy=True)

    def run(name, compress=0.0, **kw):
        env.seeds = seeds.copy()
        np.random.seed(0)
        tracker = Tracker(alg, 256, min_length=5, max_length=200, save_seeds=True, compress=compress)
        path = str(tmp_path / name)
        n = tracker.track_to_file(env, path, (32, 36, 30), (1.0, 1.0, 1.0), **kw)
        return path, n

    plain, n_plain = run('plain.trk')
    # the length-kept voxel-space streamlines of that run (one pass), restated with torch
    pts, off = env.get_streamlines_device()
    lens = lengths_packed(pts, off)
    keep = (lens >= 5.0) & (lens <= 200.0)
    npts = off[1:] - off[:-1]
    kpts = pts[torch.repeat_interleave(keep, npts)]
    koff = torch.zeros((int(keep.sum()) + 1,), dtype=torch.int64, device=DEV)
    torch.cumsum(npts[keep], 0, out=koff[1:])
    assert int(keep.sum()) == n_plain > 100
    ck = _calibrated_checkpoint(kpts, koff)
    oracle = _oracle(ck, 'fp16')
    s = oracle.predict_device(kpts, koff, distributed=False).cpu().numpy()
    assert not np.isnan(s).any()
    kept = s >= np.float32(0.5)
    assert 0 < kept.sum() < len(s), kept.sum()

    rec_plain, _ = _records(plain)
    filt, n_filt = run('filt.trk', oracle=oracle, save_scores=True)
    rec_filt, hdr = _records(filt)
    assert n_filt == int(kept.sum()) == hdr['n_count']
    assert hdr['property_names'] == ['seeds_x', 'seeds_y', 'seeds_z', 'oracle_score']
    # points and seeds: the unfiltered records selected by the scores; the score property: those scores
    assert [r[:-4] for r in rec_filt] == [r for r, k in zip(rec_plain, kept) if k]
    assert hdr['properties'][:, 3].tobytes() == s[kept].tobytes()
    # threshold 0 keeps everything: the unfiltered file byte for byte
    zero, _ = run('zero.trk', oracle=oracle, oracle_threshold=0.0)
    assert open(zero, 'rb').read() == open(plain, 'rb').read()
    # a threshold above every score: a valid empty file
    none, n_none = run('none.trk', oracle=oracle, oracle_threshold=float(s.max()) + 1e-3, save_scores=True)
    rec_none, hdr_none = _records(none)
    assert n_none == 0 and rec_none == [] and hdr_none['n_count'] == 0 and os.path.getsize(none) == 1000
    # scores are taken before --compress
    comp, _ = run('comp.trk', compress=0.2, oracle=oracle, save_scores=True)
    _, hdr_c = _records(comp)
    assert hdr_c['properties'][:, 3].tobytes() == s[kept].tobytes()
    with pytest.raises(ValueError):
        run('x.tck', oracle=oracle, save_scores=True)


# ------------------------------------------------------------------------------------ command line

def _subject(tmp_path):
    from tracktolearn_b200.io import nifti
    shape = (24, 26, 22)
    sub = synthetic.make_subject(shape, seed=5)
    affine = np.diag([1.25, 1.25, 1.25, 1.0])
    affine[:3, 3] = [-10.0, 4.0, 2.5]
    nifti.save(str(tmp_path / 'fodf.nii.gz'), sub['sh'].numpy(), affine)
    nifti.save(str(tmp_path / 'mask.nii.gz'), sub['mask'].numpy(), affine)
    nifti.save(str(tmp_path / 'seed.nii.gz'), synthetic.ellipsoid_mask(shape, frac=0.3).numpy().astype(np.uint8),
               affine)
    agent = synthetic.write_agent_dir(str(tmp_path / 'agent'), kind='tracking', hidden_dims='128-128-128')
    return agent, affine


def _track(tmp_path, agent, out, *extra):
    from tracktolearn_b200.runners.ttl_track import main
    path = str(tmp_path / out)
    main([str(tmp_path / 'fodf.nii.gz'), str(tmp_path / 'seed.nii.gz'), str(tmp_path / 'mask.nii.gz'), path,
          '--agent', agent, '--hyperparameters', os.path.join(agent, 'hyperparameters.json'), '--npv', '2',
          '--min_length', '5', '--max_length', '60', '-f'] + (['--save_seeds'] if out.endswith('.trk') else [])
         + list(extra))
    return path


def test_ttl_track_oracle_filter_end_to_end(tmp_path):
    from tracktolearn_b200.io.streamlines import read_trk
    from tracktolearn_b200.runners.ttl_oracle_filter import filter_tractogram, voxel_points
    agent, affine = _subject(tmp_path)
    plain = _track(tmp_path, agent, 'plain.trk', '--n_actor', '500')
    data, offsets, hdr = read_trk(plain)
    vox = torch.from_numpy(voxel_points(data, 'trk', hdr['voxel_sizes'])).to(DEV)
    ck = _calibrated_checkpoint(vox, torch.from_numpy(offsets).to(DEV))
    ckpt = str(tmp_path / 'oracle.ckpt')
    torch.save(ck, ckpt)
    rec_plain, _ = _records(plain)

    # every score, from the tracker (threshold 0): the same records as without the oracle, plus the score
    every = _track(tmp_path, agent, 'every.trk', '--n_actor', '500', '--oracle_checkpoint', ckpt,
                   '--oracle_threshold', '0', '--save_oracle_scores')
    rec_every, hdr_every = _records(every)
    assert [r[:-4] for r in rec_every] == rec_plain
    s_track = hdr_every['properties'][:, -1]
    kept = s_track >= 0.5
    assert 0 < kept.sum() < len(kept)

    # filtered in tracking, .trk and .tck, the same for two --n_actor values
    for ext in ('trk', 'tck'):
        outs = [_track(tmp_path, agent, 'f%d.%s' % (n, ext), '--n_actor', str(n), '--oracle_checkpoint', ckpt)
                for n in (500, 173)]
        assert open(outs[0], 'rb').read() == open(outs[1], 'rb').read()
        if ext == 'trk':
            assert _records(outs[0])[0] == [r for r, k in zip(rec_plain, kept) if k]
        else:
            plain_tck = _track(tmp_path, agent, 'plain.tck', '--n_actor', '500')
            assert _records(outs[0])[0] == [r for r, k in zip(_records(plain_tck)[0], kept) if k]

    # the standalone filter on the unfiltered outputs
    oracle = _oracle(ckpt, 'fp16')
    out = str(tmp_path / 'post.trk')
    keep_file, s_file = filter_tractogram(plain, out, oracle, threshold=0.5, save_scores=True)
    rec_out, hdr_out = _records(out)
    assert hdr_out['property_names'] == ['seeds_x', 'seeds_y', 'seeds_z', 'oracle_score']
    assert [r[:-4] for r in rec_out] == [r for r, k in zip(rec_plain, keep_file) if k]
    assert hdr_out['properties'][:, -1].tobytes() == s_file[keep_file].tobytes()
    clear = np.abs(s_track - 0.5) > FP16_TOL
    assert clear.mean() > 0.9
    np.testing.assert_array_equal(keep_file[clear], kept[clear])
    keep_tck, _ = filter_tractogram(str(tmp_path / 'plain.tck'), str(tmp_path / 'post.tck'), oracle, threshold=0.5,
                                    reference_affine=affine)
    np.testing.assert_array_equal(keep_tck[clear], kept[clear])
    rec_tck, hdr_tck = _records(str(tmp_path / 'post.tck'))
    assert hdr_tck['count'] == int(keep_tck.sum())
    assert rec_tck == [r for r, k in zip(_records(str(tmp_path / 'plain.tck'))[0], keep_tck) if k]
