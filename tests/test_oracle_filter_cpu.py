"""Oracle filtering without a GPU: argument checks of ttl_track.py and ttl_oracle_filter.py, the
``oracle_score`` property of TrkWriter through read_trk, and scores carried by the world-2 gather."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tracktolearn_b200 import parallel
from tracktolearn_b200.io.streamlines import TrkWriter, read_trk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _touch(path):
    open(path, 'wb').close()
    return str(path)


def _track_argv(tmp_path, out, *extra):
    ins = [_touch(tmp_path / n) for n in ('fodf.nii.gz', 'seed.nii.gz', 'mask.nii.gz')]
    return ins + [str(tmp_path / out), '--agent', str(tmp_path), '--hyperparameters', _touch(tmp_path / 'hp.json')] \
        + list(extra)


def _parse_track(argv):
    from tracktolearn_b200.runners.ttl_track import parse_args
    return parse_args(argv)


def _parse_filter(argv):
    from tracktolearn_b200.runners.ttl_oracle_filter import parse_args
    return parse_args(argv)


def test_ttl_track_oracle_options(tmp_path):
    ck = _touch(tmp_path / 'oracle.ckpt')
    args = _parse_track(_track_argv(tmp_path, 'out.trk'))
    assert args.oracle_checkpoint is None and args.oracle_threshold == 0.5 and args.oracle_precision == 'fp16'
    args = _parse_track(_track_argv(tmp_path, 'out.trk', '--oracle_checkpoint', ck, '--oracle_threshold', '0',
                                    '--save_oracle_scores', '--oracle_precision', 'fp32'))
    assert args.save_oracle_scores and args.oracle_threshold == 0.0 and args.oracle_precision == 'fp32'
    bad = [('out.trk', '--oracle_checkpoint', ck, '--oracle_threshold', '1.5'),
           ('out.trk', '--oracle_checkpoint', ck, '--oracle_threshold', '-0.1'),
           ('out.trk', '--oracle_checkpoint', ck, '--oracle_threshold', 'nan'),
           ('out.trk', '--save_oracle_scores'),
           ('out.tck', '--oracle_checkpoint', ck, '--save_oracle_scores'),
           ('out.trk', '--oracle_checkpoint', str(tmp_path / 'missing.ckpt'))]
    for out, *extra in bad:
        with pytest.raises(SystemExit):
            _parse_track(_track_argv(tmp_path, out, *extra))


def test_ttl_oracle_filter_options(tmp_path):
    ck = _touch(tmp_path / 'oracle.ckpt')
    trk, tck, ref = _touch(tmp_path / 'in.trk'), _touch(tmp_path / 'in.tck'), _touch(tmp_path / 'ref.nii.gz')
    args = _parse_filter([trk, str(tmp_path / 'o.trk'), '--oracle_checkpoint', ck])
    assert args.threshold == 0.5 and args.precision == 'fp16' and not args.save_scores
    _parse_filter([tck, str(tmp_path / 'o.tck'), '--oracle_checkpoint', ck, '--reference', ref, '--threshold', '1'])
    _touch(tmp_path / 'exists.trk')
    _parse_filter([trk, str(tmp_path / 'exists.trk'), '--oracle_checkpoint', ck, '-f', '--save_scores'])
    bad = [[trk, str(tmp_path / 'o.trk'), '--oracle_checkpoint', ck, '--threshold', '2'],
           [trk, str(tmp_path / 'o.trk'), '--oracle_checkpoint', ck, '--threshold', '-1'],
           [tck, str(tmp_path / 'o.tck'), '--oracle_checkpoint', ck, '--reference', ref, '--save_scores'],
           [tck, str(tmp_path / 'o.tck'), '--oracle_checkpoint', ck],
           [trk, str(tmp_path / 'o.tck'), '--oracle_checkpoint', ck, '--reference', ref],
           [trk, str(tmp_path / 'exists.trk'), '--oracle_checkpoint', ck],
           [trk, str(tmp_path / 'o.trk')],
           [str(tmp_path / 'missing.trk'), str(tmp_path / 'o.trk'), '--oracle_checkpoint', ck],
           [trk, str(tmp_path / 'o.nii'), '--oracle_checkpoint', ck]]
    for argv in bad:
        with pytest.raises(SystemExit):
            _parse_filter(argv)


def test_help_lists_the_oracle_groups():
    for script, flags in (('ttl_track.py', ('Oracle filtering', '--oracle_checkpoint', '--oracle_threshold',
                                            '--oracle_precision', '--save_oracle_scores')),
                          ('ttl_oracle_filter.py', ('Oracle filtering', 'in_tractogram', 'out_tractogram',
                                                    '--oracle_checkpoint', '--reference', '--threshold',
                                                    '--precision', '--save_scores'))):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', script), '--help'],
                             capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        for flag in flags:
            assert flag in out.stdout, (script, flag)


def _packed(rng, n):
    lens = rng.randint(1, 40, size=n)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    return rng.randn(int(offsets[-1]), 3).astype(np.float32), offsets


@pytest.mark.parametrize('save_seeds', [False, True])
def test_trk_writer_oracle_score_round_trip(tmp_path, save_seeds):
    rng = np.random.RandomState(3)
    path = str(tmp_path / 'a.trk')
    w = TrkWriter(path, (10, 11, 12), (1.25, 1.25, 1.25), np.eye(4), save_seeds=save_seeds, save_scores=True)
    batches = []
    for n in (7, 0, 30):
        data, offsets = _packed(rng, n)
        seeds, scores = rng.randn(n, 3), rng.rand(n).astype(np.float32)
        w.write(data, offsets, seeds if save_seeds else None, scores)
        batches.append((data, offsets, seeds, scores))
    w.close()
    data, offsets, hdr = read_trk(path)
    names = ['seeds_x', 'seeds_y', 'seeds_z'] * save_seeds + ['oracle_score']
    assert hdr['property_names'] == names and hdr['n_properties'] == len(names) and hdr['n_count'] == 37
    np.testing.assert_array_equal(data, np.concatenate([b[0] for b in batches]))
    np.testing.assert_array_equal(np.diff(offsets), np.concatenate([np.diff(b[1]) for b in batches]))
    props = hdr['properties']
    np.testing.assert_array_equal(props[:, -1], np.concatenate([b[3] for b in batches]))
    if save_seeds:
        np.testing.assert_array_equal(props[:, :3], np.concatenate([b[2] for b in batches]).astype(np.float32))


def test_trk_writer_bytes_unchanged_without_scores(tmp_path):
    rng = np.random.RandomState(4)
    data, offsets = _packed(rng, 20)
    seeds = rng.randn(20, 3)
    outs = []
    for kw in ({}, {'save_scores': False}):
        path = str(tmp_path / ('%d.trk' % len(outs)))
        w = TrkWriter(path, (10, 11, 12), (2.0, 2.0, 2.0), np.eye(4), True, **kw)
        w.write(data, offsets, seeds)
        w.close()
        outs.append(open(path, 'rb').read())
    assert outs[0] == outs[1]
    assert read_trk(os.path.join(str(tmp_path), '0.trk'))[2]['property_names'] == ['seeds_x', 'seeds_y', 'seeds_z']


def _rank_part(rank):
    rng = np.random.RandomState(10 + rank)
    n = 5 + 3 * rank
    data, offsets = _packed(rng, n)
    return data, offsets, rng.randn(n, 3), (np.arange(n) % 5).astype(np.int64), rng.rand(n).astype(np.float32)


def _gather_worker(rank, world, port, via, with_scores, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    data, offsets, seeds, flags, scores = _rank_part(rank)
    merged = parallel.gather_packed(torch.from_numpy(data), torch.from_numpy(np.diff(offsets)),
                                    torch.from_numpy(seeds), torch.from_numpy(flags), via=via,
                                    scores=torch.from_numpy(scores) if with_scores else None)
    if rank == 0:
        q.put((merged.data, merged.offsets, dict(merged.data_per_streamline)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('via', ['nccl', 'host'])
@pytest.mark.parametrize('with_scores', [False, True])
def test_two_rank_gather_carries_scores(via, with_scores):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, via, with_scores, q)) for r in range(2)]
    for p in procs:
        p.start()
    data, offsets, per = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    parts = [_rank_part(r) for r in range(2)]
    np.testing.assert_array_equal(data, np.concatenate([p[0] for p in parts]))
    np.testing.assert_array_equal(np.diff(offsets), np.concatenate([np.diff(p[1]) for p in parts]))
    np.testing.assert_array_equal(per['seeds'], np.concatenate([p[2] for p in parts]))
    np.testing.assert_array_equal(per['flags'], np.concatenate([p[3] for p in parts]))
    if with_scores:
        np.testing.assert_array_equal(per['oracle_score'], np.concatenate([p[4] for p in parts]))
    else:
        assert set(per) == {'seeds', 'flags'}
