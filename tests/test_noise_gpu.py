"""Tracking noise drawn inside the step kernels (NoisyTrackingEnvironment with noise_rng='device'):
the draws against the numpy Philox (tests/noise_oracle.py) and against N(0, 1), the env against
PhiloxNoiseOracleEnv,
and the tractogram's independence of how the run is scheduled."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.helpers import load_golden, meta, subject_for
from tests.noise_oracle import PhiloxNoiseOracleEnv, philox_normals
from tracktolearn_b200 import _lib, synthetic

pytestmark = pytest.mark.gpu
POS_TOL = 1e-5
STATE_TOL = 1e-5
SIGMA = 0.1


def _device_noise(env, sigma=SIGMA, seed=2024):
    """Switch a NoisyTrackingEnvironment built with the default host noise to device-drawn noise."""
    env.noise, env.noise_rng, env.noise_seed = sigma, 'device', seed
    return env


def _normals(seed, g, L):
    lib = _lib.load()
    dev = torch.device('cuda:0')
    g_d = torch.from_numpy(np.ascontiguousarray(g, dtype=np.int64)).to(dev)
    L_d = torch.from_numpy(np.ascontiguousarray(L, dtype=np.int32)).to(dev)
    out = torch.empty((len(g), 3), dtype=torch.float64, device=dev)
    nz = _lib.Noise(sigma=0.0, seed=seed, row_base=0)
    _lib.check(lib.ttl_noise_normals(ctypes.byref(nz), _lib.ptr(g_d), _lib.ptr(L_d), len(g), _lib.ptr(out),
                                     _lib.stream_ptr(dev)), 'ttl_noise_normals')
    return out.cpu().numpy()


def test_device_normals_equal_the_oracle_and_are_standard_normal():
    from scipy import stats
    rows, steps = 100000, 10
    g = np.repeat(np.arange(rows, dtype=np.int64), steps)
    L = np.tile(np.arange(1, steps + 1, dtype=np.int32), rows)
    z = _normals(12345, g, L)
    np.testing.assert_allclose(z, philox_normals(12345, g, L), rtol=0, atol=1e-13)
    # seeds and indices beyond 32 bits go into the counter / key
    gb = np.asarray([0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 3, 2 ** 62], dtype=np.int64)
    Lb = np.asarray([1, 2, 3, 799, 5, 1], dtype=np.int32)
    for seed in (0, 2 ** 32 + 5, 2 ** 64 - 1):
        np.testing.assert_allclose(_normals(seed, gb, Lb), philox_normals(seed, gb, Lb), rtol=0, atol=1e-13)
    flat = z.reshape(-1)
    n = flat.size
    assert stats.kstest(flat, 'norm').pvalue > 1e-3
    assert abs(flat.mean()) < 5 / np.sqrt(n)
    assert abs(flat.std() - 1) < 5 / np.sqrt(n)
    assert np.abs(z).max() <= 8.58

    def corr_ok(a, b):
        assert abs(np.corrcoef(a, b)[0, 1]) < 5 / np.sqrt(a.size), np.corrcoef(a, b)[0, 1]
    cube = z.reshape(rows, steps, 3)
    corr_ok(z[:, 0], z[:, 1])                                        # components
    corr_ok(z[:, 1], z[:, 2])
    corr_ok(z[:, 0], z[:, 2])
    corr_ok(cube[:-1].reshape(-1), cube[1:].reshape(-1))             # adjacent rows, same step
    corr_ok(cube[:, :-1].reshape(-1), cube[:, 1:].reshape(-1))       # adjacent steps, same row


def _parity_setups():
    """(name, golden-like meta, subject, seeds, geometry, reward): the env_noisy fixture volume, and the
    long-episode setup of test_env_gpu.py (1500 seeds, alignment reward on)."""
    g = load_golden('env_noisy')
    m = meta(g)
    yield 'fixture', g, subject_for(g), g['seeds'], dict(voxel=m['vox'], step=m['step_mm'], theta=m['theta'],
                                                          max_len=m['max_length']), False
    shape = (40, 44, 36)
    sub = {k: (v.numpy() if v is not None else None) for k, v in synthetic.make_subject(shape, seed=77).items()}
    rs = np.random.RandomState(5)
    seeds = synthetic.seeds_from_mask(synthetic.ellipsoid_mask(shape, frac=0.33).numpy(), 1, rs)
    rs.shuffle(seeds)
    gl = {'meta_shape': np.asarray(shape), 'meta': np.asarray([1.0, 0.75, 30.0, 24.0, 0.1, 32.0, 0.75])}
    yield 'long', gl, sub, seeds[:1500], dict(voxel=1.0, step=0.75, theta=30.0, max_len=24.0), True


@pytest.mark.parametrize('protocol', ['step', 'step_device'])
def test_env_with_device_noise_matches_oracle(protocol):
    """GPU env (noise_rng='device', sigma 0.1) against PhiloxNoiseOracleEnv with the same fixed
    actions: positions 1e-5 voxel, state 1e-5, flags, dones, lengths and alive order exactly; through the
    reference protocol (step / harvest) and the device one (step_device / harvest_device)."""
    from tests.gpu_helpers import make_gpu_env
    for name, g, sub, seeds, geo, reward in _parity_setups():
        n = len(seeds)
        env, _ = make_gpu_env(g, True, reward, sub=sub, seeds=seeds)
        _device_noise(env, seed=77)
        ref = PhiloxNoiseOracleEnv(sub['sh'], sub['mask'], seeds, geo['voxel'], geo['step'], theta=geo['theta'],
                                   max_length_mm=geo['max_len'], peaks=sub['peaks'] if reward else None,
                                   compute_reward=reward, noise=SIGMA, noise_seed=77)
        env.reset(0, n)
        ref.reset(0, n)
        rs = np.random.RandomState(9)
        a = rs.normal(size=(n, 3))
        t = 0
        while len(ref.continue_idx):
            ci = ref.continue_idx.copy()
            np.testing.assert_array_equal(env.continue_idx, ci)
            a = a + 0.17 * rs.normal(size=(n, 3))
            a /= np.linalg.norm(a, axis=1, keepdims=True)
            act = (a[ci] * rs.uniform(0.3, 1.0, size=(len(ci), 1))).astype(np.float32)
            st_r, r_r, d_r, _ = ref.step(act)
            if protocol == 'step':
                st_g, r_g, d_g, _ = env.step(act)
                np.testing.assert_array_equal(d_g, d_r)
                np.testing.assert_allclose(st_g.cpu().numpy(), st_r, rtol=0, atol=STATE_TOL)
                if reward:
                    np.testing.assert_allclose(r_g, r_r, rtol=0, atol=2e-6)
                h_g, _ = env.harvest()
            else:
                env.step_device(torch.from_numpy(act).cuda())
                env.harvest_device()
                env.n_alive()
                h_g = env.current_state()
            np.testing.assert_allclose(env.streamlines[ci, ref.length - 1], ref.streamlines[ci, ref.length - 1],
                                       rtol=0, atol=POS_TOL)
            np.testing.assert_array_equal(env.flags[ci], ref.flags[ci])
            h_r, _ = ref.harvest()
            np.testing.assert_allclose(h_g.cpu().numpy(), h_r, rtol=0, atol=STATE_TOL)
            t += 1
        assert t >= (25 if name == 'long' else 5), (name, t)
        assert env.n_alive() == 0
        np.testing.assert_array_equal(env.lengths, ref.lengths)
        np.testing.assert_array_equal(env.flags, ref.flags)
        tr = env.get_streamlines()
        sl, _, _ = ref.get_streamlines()
        np.testing.assert_array_equal(tr.lengths, [len(s) for s in sl])
        np.testing.assert_allclose(tr.data, np.concatenate(sl), rtol=0, atol=POS_TOL)


def _setup(n_seeds=900):
    """test_tracker_gpu.py's closed-loop setup with the fp16 actor tier."""
    from tests.gpu_helpers import make_gpu_env
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    shape = (32, 36, 30)
    sub = {k: (v.numpy() if v is not None else None) for k, v in synthetic.make_subject(shape, seed=11).items()}
    rs = np.random.RandomState(3)
    seeds = synthetic.seeds_from_mask(synthetic.ellipsoid_mask(shape, frac=0.36).numpy(), 1, rs)
    rs.shuffle(seeds)
    seeds = seeds[:n_seeds]
    g = {'meta_shape': np.asarray(shape), 'meta': np.asarray([1.0, 0.75, 30.0, 30.0, 0.1, 40.0, 0.75])}
    env, _ = make_gpu_env(g, True, False, sub=sub, seeds=seeds)
    alg = SACAuto(615, 3, '128-128-128', n_actors=1024, device=torch.device('cuda:0'), precision='fp16')
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(615, '128-128-128', seed=5, kind='tracking'))
    env.operand = 'fp16'
    return env, alg, seeds


def _episode(env, alg, start, end, slots=None, locality=True):
    """One pass as Tracker._run_pass runs it; returns (points, offsets, flags) as host arrays."""
    if slots is None:
        env.reset(start, end)
    else:
        env.reset_streaming(start, end, slots, fp32_state=False, operand='fp16', locality=locality)
    alg.validation_episode(None, env, 0.0)
    assert env.n_alive() == 0
    tr = env.get_streamlines()
    return tr.data, np.asarray(tr.offsets), np.asarray(tr.data_per_streamline['flags'])


def _concat(parts):
    offsets = [parts[0][1]]
    for _, o, _ in parts[1:]:
        offsets.append(o[1:] + offsets[-1][-1])
    return (np.concatenate([p for p, _, _ in parts]), np.concatenate(offsets), np.concatenate([f for _, _, f in parts]))


def _assert_same(a, b, what):
    for x, y, part in zip(a, b, ('points', 'offsets', 'flags')):
        assert x.shape == y.shape and np.array_equal(x, y), (what, part)


def test_device_noise_tractogram_does_not_depend_on_scheduling():
    env, alg, seeds = _setup()
    _device_noise(env)
    n = len(seeds)
    ref = _episode(env, alg, 0, n)                               # batch tracking, every seed in one batch
    legs = {'streaming 256': dict(slots=256), 'streaming 128': dict(slots=128),
            'no locality': dict(slots=256, locality=False)}
    for what, kw in legs.items():
        _assert_same(ref, _episode(env, alg, 0, n, **kw), what)
    # consecutive batches reset(start, end) of the same list
    parts = [_episode(env, alg, s, min(n, s + 300)) for s in range(0, n, 300)]
    _assert_same(ref, _concat(parts), 'batches of 300')
    try:
        alg.fuse_head = False
        _assert_same(ref, _episode(env, alg, 0, n, slots=256), 'unfused head')
        alg.fuse_head = True
        alg.use_cuda_graph = True
        _assert_same(ref, _episode(env, alg, 0, n, slots=256), 'graph replay')
        assert alg._runner.graphs is not None and alg._runner.replays > 10
    finally:
        alg.fuse_head, alg.use_cuda_graph = True, False
    # two shards of the same list, tracked one after the other, concatenated
    k = 377
    env.seeds, env.seed_offset = seeds[:k], 0
    p0, o0, f0 = _episode(env, alg, 0, k, slots=128)
    env.seeds, env.seed_offset = seeds[k:], k
    p1, o1, f1 = _episode(env, alg, 0, n - k, slots=128)
    _assert_same(ref, _concat([(p0, o0, f0), (p1, o1, f1)]), 'two shards')
    # the noise reached the streamlines: without it they differ
    env.seeds, env.seed_offset, env.noise_rng, env.noise = seeds, 0, 'host', 0.0
    plain = _episode(env, alg, 0, n)
    assert not (plain[1].shape == ref[1].shape and np.array_equal(plain[0], ref[0]))


def test_device_noise_keeps_the_fused_head_and_graph_replay():
    env, alg, seeds = _setup()
    n = len(seeds)
    per_step = {}
    try:
        alg.use_cuda_graph = True
        for mode in ('noise 0', 'device 0.1'):
            if mode == 'device 0.1':
                _device_noise(env)
            _episode(env, alg, 0, n, slots=256)
            assert alg._runner.fuse_head and alg._runner.use_graph and alg._runner.graphs is not None, mode
            per_step[mode] = alg._runner.kernels_per_step
    finally:
        alg.use_cuda_graph = False
    assert per_step['noise 0'] > 0 and per_step['device 0.1'] == per_step['noise 0'], per_step


def test_device_noise_at_sigma_zero_equals_no_noise():
    env, alg, seeds = _setup()
    n = len(seeds)
    plain = _episode(env, alg, 0, n, slots=256)
    _device_noise(env, sigma=0.0)
    _assert_same(plain, _episode(env, alg, 0, n, slots=256), 'sigma 0')


def test_device_noise_episode_stays_inside_its_buffers():
    from tracktolearn_b200.environments.tracking_env import _BatchBuffers
    old = _BatchBuffers.GUARD
    _BatchBuffers.GUARD = True
    try:
        env, alg, seeds = _setup()
        _device_noise(env)
        _episode(env, alg, 0, len(seeds), slots=128)
        assert len(env._batch._guarded) > 15
        assert env._batch.check_guards() == 0
    finally:
        _BatchBuffers.GUARD = old


def test_ttl_track_device_noise_output_does_not_depend_on_n_actor(tmp_path):
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.runners.ttl_track import main
    shape = (24, 26, 22)
    sub = synthetic.make_subject(shape, seed=5)
    affine = np.diag([1.25, 1.25, 1.25, 1.0])
    nifti.save(str(tmp_path / 'fodf.nii.gz'), sub['sh'].numpy(), affine)
    nifti.save(str(tmp_path / 'mask.nii.gz'), sub['mask'].numpy(), affine)
    nifti.save(str(tmp_path / 'seed.nii.gz'), synthetic.ellipsoid_mask(shape, frac=0.3).numpy().astype(np.uint8), affine)
    agent = synthetic.write_agent_dir(str(tmp_path / 'agent'), kind='tracking', hidden_dims='128-128-128')
    outs = []
    for n_actor in ('512', '4096', 'host'):
        out = str(tmp_path / ('out_%s.trk' % n_actor))
        extra = ['--noise_rng', 'device', '--n_actor', n_actor] if n_actor != 'host' else ['--n_actor', '512']
        main([str(tmp_path / 'fodf.nii.gz'), str(tmp_path / 'seed.nii.gz'), str(tmp_path / 'mask.nii.gz'), out,
              '--agent', agent, '--hyperparameters', os.path.join(agent, 'hyperparameters.json'),
              '--npv', '2', '--min_length', '5', '--max_length', '60', '--save_seeds', '--noise', '0.1',
              '--rng_seed', '3'] + extra)
        outs.append(open(out, 'rb').read())
    assert len(outs[0]) > 10000
    assert outs[0] == outs[1]
    assert outs[0] != outs[2]            # host-drawn noise: another stream
