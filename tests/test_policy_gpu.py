"""The stochastic policy sampled on the device (ttl_policy): the draws against the numpy restatement
(tests/policy_oracle.py) and N(0, 1), the sampling arithmetic against the actor's raw output, the fused route
against the actor-then-step route, and the tractogram's independence of how the run is scheduled."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.policy_oracle import policy_actions, policy_eps
from tests.test_noise_gpu import _assert_same, _concat
from tracktolearn_b200 import _lib, synthetic

pytestmark = pytest.mark.gpu
SEED = 2025


def _setup(precision='fp16', n_seeds=900):
    """test_noise_gpu.py's closed-loop setup (NoisyTrackingEnvironment at noise 0) with the given actor tier."""
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
    alg = SACAuto(615, 3, '128-128-128', n_actors=1024, device=torch.device('cuda:0'), precision=precision)
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(615, '128-128-128', seed=5, kind='tracking'))
    env.operand = 'fp16' if precision == 'fp16' else 'bf16'
    return env, alg, seeds


def _episode(env, alg, start, end, slots=None, locality=True, prob=1.0, seed=SEED):
    """One pass as Tracker._run_pass runs it; returns (points, offsets, flags) as host arrays."""
    if slots is None:
        env.reset(start, end)
    else:
        prec = alg.agent.actor.precision
        env.reset_streaming(start, end, slots, fp32_state=False, operand=prec, locality=locality)
    alg.validation_episode(None, env, prob, policy_seed=seed)
    assert env.n_alive() == 0
    tr = env.get_streamlines()
    return tr.data, np.asarray(tr.offsets), np.asarray(tr.data_per_streamline['flags'])


def _eps_for_records(seed, row_base, rows, L, n_alive=None, prob=1.0):
    """ttl_policy_eps over a hand-made alive list: rank r holds (rows[r], L[r])."""
    lib = _lib.load()
    dev = torch.device('cuda:0')
    n = len(rows)
    rec = np.zeros((n, 8), dtype=np.int32)
    rec[:, 0], rec[:, 1] = rows, L
    rec_d = torch.from_numpy(rec).to(dev)
    ctrl = torch.zeros((16,), dtype=torch.int32, device=dev)
    ctrl[0] = n if n_alive is None else n_alive
    b = _lib.Batch(n=n, n_slots=n, capacity=n, ctrl=ctrl.data_ptr())
    b.rank_rec[0] = rec_d.data_ptr()
    b.rank_rec[1] = rec_d.data_ptr()
    out = torch.full((n, 4), float('nan'), dtype=torch.float32, device=dev)
    pol = _lib.Policy(seed=seed, row_base=row_base, prob=prob)
    _lib.check(lib.ttl_policy_eps(ctypes.byref(pol), ctypes.byref(b), 0, n, _lib.ptr(out), 4, _lib.stream_ptr(dev)),
               'ttl_policy_eps')
    return out.cpu().numpy()


def _assert_eps_close(got, want):
    """Within 1 fp32 ulp everywhere, and equal except for rare rounding ties of the fp64 value."""
    gi, wi = got.view(np.int32).astype(np.int64), want.view(np.int32).astype(np.int64)
    assert np.abs(gi - wi).max() <= 1
    assert int((gi != wi).sum()) <= 3, int((gi != wi).sum())


def test_policy_eps_equals_numpy_and_is_standard_normal():
    n = 34000
    rs = np.random.RandomState(4)
    rows = rs.permutation(n).astype(np.int32)
    L = rs.randint(1, 800, size=n).astype(np.int32)
    for seed, row_base in ((SEED, 0), (2 ** 64 - 1, 2 ** 33 + 7)):
        out = _eps_for_records(seed, row_base, rows, L)
        want = policy_eps(seed, row_base + rows.astype(np.int64), L)
        _assert_eps_close(out[:, :3], want)
        assert np.isnan(out[:, 3]).all()                  # ld 4: the fourth column is not written
    flat = out[:, :3].astype(np.float64).reshape(-1)
    assert flat.size >= 100000
    assert abs(flat.mean()) < 5 / np.sqrt(flat.size)
    assert abs(flat.var() - 1) < 5 * np.sqrt(2.0 / flat.size)
    # ranks beyond the alive count are left alone
    part = _eps_for_records(SEED, 0, rows[:100], L[:100], n_alive=60)
    assert np.isfinite(part[:60, :3]).all() and np.isnan(part[60:]).all()


def test_sampled_actions_follow_the_formula_from_the_actors_own_output():
    env, alg, seeds = _setup()
    n = len(seeds)
    env.reset_streaming(0, n, 256, fp32_state=True)                           # refill: point counts differ
    alg.validation_episode(None, env, 1.0, max_steps=6, policy_seed=SEED)
    alive = env.n_alive()
    assert alive > 20
    bb = env._batch
    rec = bb.rank_rec[env._cur][:alive].cpu().numpy().view(np.int32)
    rows, L = rec[:, 0].astype(np.int64), rec[:, 1]
    np.testing.assert_array_equal(rows, bb.alive[env._cur][:alive].cpu().numpy())
    assert len(np.unique(L)) > 1
    eps_d = torch.empty((n, 3), dtype=torch.float32, device=env.device)
    env.policy_eps(env.policy(SEED, 1.0), eps_d)
    action, _, pre = alg.agent.actor.forward_device(env.current_state(), 1.0, n_rows=alive, eps=eps_d[:alive],
                                                    want_logp=False, want_pre=True)
    eps = policy_eps(SEED, env._row_base + rows, L)
    _assert_eps_close(eps_d[:alive].cpu().numpy(), eps)
    want = policy_actions(pre.cpu().numpy(), eps, 1.0)
    np.testing.assert_allclose(action.cpu().numpy(), want, rtol=0, atol=2e-6)
    assert np.abs(want - np.tanh(pre.cpu().numpy()[:, :3])).max() > 0.05     # the sampling moved the actions


@pytest.mark.parametrize('precision', ['fp16', 'bf16', 'tf32'])
def test_fused_and_eps_routes_give_the_same_tractogram(precision):
    env, alg, seeds = _setup(precision)
    n = len(seeds)
    fused = _episode(env, alg, 0, n, slots=256)
    assert alg._runner.fuse_head and alg._runner.policy_seed == SEED
    try:
        alg.fuse_head = False
        unfused = _episode(env, alg, 0, n, slots=256)
        assert not alg._runner.fuse_head and alg._runner.eps_buf is not None
    finally:
        alg.fuse_head = True
    _assert_same(fused, unfused, precision)


@pytest.mark.parametrize('sigma', [0.0, 0.1])
def test_seeded_policy_tractogram_does_not_depend_on_scheduling(sigma):
    env, alg, seeds = _setup()
    if sigma:
        env.noise, env.noise_rng, env.noise_seed = sigma, 'device', 77
    n = len(seeds)
    ref = _episode(env, alg, 0, n)                               # batch tracking, every seed in one batch
    legs = {'streaming 256': dict(slots=256), 'streaming 128': dict(slots=128),
            'no locality': dict(slots=256, locality=False)}
    for what, kw in legs.items():
        _assert_same(ref, _episode(env, alg, 0, n, **kw), what)
    parts = [_episode(env, alg, s, min(n, s + 300)) for s in range(0, n, 300)]
    _assert_same(ref, _concat(parts), 'batches of 300')
    try:
        alg.fuse_head = False
        _assert_same(ref, _episode(env, alg, 0, n, slots=256), 'unfused head')
        alg.fuse_head = True
        alg.use_cuda_graph = True
        _assert_same(ref, _episode(env, alg, 0, n, slots=256), 'graph replay')
        assert alg._runner.graphs is not None and alg._runner.replays > 3
    finally:
        alg.fuse_head, alg.use_cuda_graph = True, False
    k = 377
    env.seeds, env.seed_offset = seeds[:k], 0
    p0 = _episode(env, alg, 0, k, slots=128)
    env.seeds, env.seed_offset = seeds[k:], k
    p1 = _episode(env, alg, 0, n - k, slots=128)
    _assert_same(ref, _concat([p0, p1]), 'two shards')
    env.seeds, env.seed_offset = seeds, 0
    # the sampling reached the streamlines
    plain = _episode(env, alg, 0, n, prob=0.0, seed=None)
    assert not (plain[1].shape == ref[1].shape and np.array_equal(plain[0], ref[0]))


def _policy_step_loop(env, alg, seed, prob, slots=256):
    """ttl_env_step with the head partials and the policy, driven by hand until every streamline stopped."""
    n = len(env.seeds)
    env.reset_streaming(0, n, slots, fp32_state=False, operand='fp16')
    actor = alg.agent.actor
    pol = env.policy(seed, prob)
    while True:
        for _ in range(8):
            head = actor.forward_head_partial(env.current_state_bf16(), env._n_alive_host,
                                              n_rows_dev=env.alive_count_tensor(), layout=env.bf16_layout,
                                              state=env.current_state(), policy=True)
            assert head is not None
            env.step_device(head=head, policy=pol)
            env.harvest_device()
        if env.n_alive() == 0:
            break
    tr = env.get_streamlines()
    return tr.data, np.asarray(tr.offsets), np.asarray(tr.data_per_streamline['flags'])


def test_single_step_entry_with_policy_at_prob_zero_is_the_deterministic_step():
    env, alg, seeds = _setup()
    n = len(seeds)
    det = _episode(env, alg, 0, n, slots=256, prob=0.0, seed=None)
    _assert_same(det, _policy_step_loop(env, alg, SEED, 0.0), 'prob 0')
    a = _policy_step_loop(env, alg, 1, 1.0)
    b = _policy_step_loop(env, alg, 2, 1.0)
    assert not (a[1].shape == b[1].shape and np.array_equal(a[0], b[0]))
    _assert_same(a, _policy_step_loop(env, alg, 1, 1.0), 'same seed again')


def test_seeded_policy_keeps_the_fused_head_and_graph_replay():
    env, alg, seeds = _setup()
    n = len(seeds)
    per_step = {}
    try:
        alg.use_cuda_graph = True
        for mode, prob, seed in (('prob 0', 0.0, None), ('prob 1 seeded', 1.0, SEED)):
            _episode(env, alg, 0, n, slots=256, prob=prob, seed=seed)
            r = alg._runner
            assert r.fuse_head and r.use_graph and r.graphs is not None and r.replays > 3, mode
            per_step[mode] = r.kernels_per_step
    finally:
        alg.use_cuda_graph = False
    assert per_step['prob 1 seeded'] == per_step['prob 0'] == 3, per_step


def test_policy_episode_stays_inside_its_buffers():
    from tracktolearn_b200.algorithms.shared.offpolicy import MaxEntropyActor
    from tracktolearn_b200.environments.tracking_env import _BatchBuffers
    old = (_BatchBuffers.GUARD, MaxEntropyActor.GUARD)
    _BatchBuffers.GUARD = MaxEntropyActor.GUARD = True
    try:
        env, alg, seeds = _setup()
        env.noise, env.noise_rng, env.noise_seed = 0.1, 'device', 9
        _episode(env, alg, 0, len(seeds), slots=128)
        alg.fuse_head = False
        _episode(env, alg, 0, len(seeds), slots=128)
        assert len(env._batch._guarded) > 15
        assert env._batch.check_guards() == 0
        assert alg.agent.actor.check_guards() == 0
    finally:
        _BatchBuffers.GUARD, MaxEntropyActor.GUARD = old
        alg.fuse_head = True


def test_ttl_track_policy_prob_output_does_not_depend_on_n_actor(tmp_path):
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
    for n_actor, prob in (('512', '0.5'), ('4096', '0.5'), ('512', '0')):
        out = str(tmp_path / ('out_%s_%s.trk' % (n_actor, prob)))
        main([str(tmp_path / 'fodf.nii.gz'), str(tmp_path / 'seed.nii.gz'), str(tmp_path / 'mask.nii.gz'), out,
              '--agent', agent, '--hyperparameters', os.path.join(agent, 'hyperparameters.json'),
              '--npv', '2', '--min_length', '0', '--max_length', '60', '--save_seeds', '--rng_seed', '3',
              '--n_actor', n_actor, '--policy_prob', prob])
        outs.append(open(out, 'rb').read())
    assert len(outs[0]) > 5000
    assert outs[0] == outs[1]
    assert outs[0] != outs[2]            # the mean action: another tractogram
