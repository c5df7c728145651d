"""Device episode loop, streaming refill and the Tracker against the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import ttl_oracle as O
from tracktolearn_b200 import synthetic

pytestmark = pytest.mark.gpu

TC = ['bf16', 'fp16', 'tf32']        # tensor-core tiers of the actor = element types of the env's operand rows
OP_DTYPE = {'bf16': torch.bfloat16, 'fp16': torch.float16, 'tf32': torch.float32}


def _round_like_operand(x, prec):
    """numpy fp32 -> the values an operand row of type `prec` holds (as fp32)."""
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    if prec == 'tf32':          # cvt.rna.tf32.f32: nearest, ties away from zero, 13 low mantissa bits dropped
        return ((t.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32).numpy()
    return t.to(OP_DTYPE[prec]).float().numpy()


def _setup(shape=(32, 36, 30), n_seeds=900, precision='fp32', vox=1.0):
    from tests.gpu_helpers import make_gpu_env
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    sub = {k: (v.numpy() if v is not None else None) for k, v in synthetic.make_subject(shape, seed=11).items()}
    rs = np.random.RandomState(3)
    seeds = synthetic.seeds_from_mask(synthetic.ellipsoid_mask(shape, frac=0.36).numpy(), 1, rs)
    rs.shuffle(seeds)
    seeds = seeds[:n_seeds]
    g = {'meta_shape': np.asarray(shape), 'meta': np.asarray([vox, 0.75 * vox, 30.0, 30.0 * vox, 0.1, 40.0, 0.75])}
    env, _ = make_gpu_env(g, True, False, sub=sub, seeds=seeds)
    sd = synthetic.actor_state_dict(615, '128-128-128', seed=5, kind='tracking')
    alg = SACAuto(615, 3, '128-128-128', n_actors=256, device=torch.device('cuda:0'), precision=precision)
    alg.agent.actor.load_state_dict(sd)
    env.operand = precision if precision in TC else 'bf16'      # default element type of reset_streaming's rows
    return env, alg, sub, seeds, {k: v.numpy() for k, v in sd.items()}


def test_validation_episode_matches_oracle_closed_loop():
    """Closed loop (actor output feeds the env) with the fp32 actor tier: whole trajectories
    agree with the CPU oracle loop to 1e-4 voxels, flags and lengths exactly, for all but a
    handful of streamlines that sit on a float threshold."""
    env, alg, sub, seeds, sd = _setup()
    n = len(seeds)
    state = env.reset(0, n)
    alg.validation_episode(state, env, 0.0)
    tr = env.get_streamlines()
    ref = O.OracleEnv(sub['sh'], sub['mask'], seeds, 1.0, 0.75, theta=30.0, max_length_mm=30.0, noisy=True)
    O.validation_episode(ref, sd, 0, n)
    sl, _, fl = ref.get_streamlines()
    same_len = np.asarray([len(s) for s in sl]) == tr.lengths
    assert same_len.mean() > 0.99, same_len.mean()
    assert (np.asarray(fl) == tr.data_per_streamline['flags'])[same_len].all()
    worst = 0.0
    for i in np.nonzero(same_len)[0]:
        worst = max(worst, float(np.abs(sl[i] - tr.streamlines[i]).max()))
    assert worst < 1e-3, worst
    assert same_len.mean() < 1.0 or env.streamline_steps() == int(sum(ref.lengths - 1))


def test_config0_shape_closed_loop_matches_oracle():
    """BASELINE.json configs[0] at its exact shape: 64^3 1 mm order-8 volume, npv 1, n_actor 4096, step
    0.75 mm, the bundled agent's 615-1024-1024-1024-6 network, tracked to the end in closed loop -- the
    device path with the fp32 actor tier against the CPU oracle loop (the reference-path baseline)."""
    from tests.gpu_helpers import make_gpu_env
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    shape = (64, 64, 64)
    sub = {k: (v.numpy() if v is not None else None) for k, v in synthetic.make_subject(shape, seed=1234).items()}
    rs = np.random.RandomState(1337)
    seeds = synthetic.seeds_from_mask(sub['seed_mask'], 1, rs)          # npv = 1 on the mask shell
    rs.shuffle(seeds)
    seeds = seeds[:4096]
    assert len(seeds) == 4096
    g = {'meta_shape': np.asarray(shape), 'meta': np.asarray([1.0, 0.75, 30.0, 300.0, 0.1, 400.0, 0.75])}
    env, _ = make_gpu_env(g, True, False, sub=sub, seeds=seeds)
    assert env.max_nb_steps == 400
    sd = synthetic.actor_state_dict(615, '1024-1024-1024', seed=1111, kind='tracking')
    alg = SACAuto(615, 3, '1024-1024-1024', n_actors=4096, device=torch.device('cuda:0'), precision='fp32')
    alg.agent.actor.load_state_dict(sd)
    state = env.reset(0, 4096)
    alg.validation_episode(state, env, 0.0)
    tr = env.get_streamlines()
    ref = O.OracleEnv(sub['sh'], sub['mask'], seeds, 1.0, 0.75, theta=30.0, max_length_mm=300.0, noisy=True)
    O.validation_episode(ref, {k: v.numpy() for k, v in sd.items()}, 0, 4096)
    sl, _, fl = ref.get_streamlines()
    same_len = np.asarray([len(s) for s in sl]) == tr.lengths
    assert same_len.mean() > 0.99, same_len.mean()       # a handful sit on a float threshold and part ways
    assert (np.asarray(fl) == tr.data_per_streamline['flags'])[same_len].all()
    # closed loop over up to 400 steps: the 1e-6 differences between two fp32 matrix products feed back
    # through the policy, so whole trajectories agree to 1e-2 voxel (measured 3e-3); per-step parity at
    # 1e-5 is pinned by tests/test_env_gpu.py and tests/test_actor_gpu.py
    worst = max(float(np.abs(sl[i] - tr.streamlines[i]).max()) for i in np.nonzero(same_len)[0])
    assert worst < 1e-2, worst
    assert np.mean([len(s) for s in sl]) > 20


@pytest.mark.parametrize('prec', TC)
def test_streaming_refill_equals_batch_tracking(prec):
    """Streaming tracker (256 slots over 900 seeds) gives, seed for seed, bit-identical
    streamlines to tracking the seeds in consecutive batches (same kernels, same order of
    arithmetic per streamline)."""
    env, alg, sub, seeds, sd = _setup(precision=prec)
    n = len(seeds)
    batches = []
    for start in range(0, n, 256):
        st = env.reset(start, min(n, start + 256))
        alg.validation_episode(st, env, 0.0)
        batches.append(env.get_streamlines())
    st = env.reset_streaming(0, n, 256)
    alg.validation_episode(st, env, 0.0)
    tr = env.get_streamlines()
    total_steps = env.streamline_steps()
    lens = np.concatenate([b.lengths for b in batches])
    np.testing.assert_array_equal(tr.lengths, lens)
    np.testing.assert_array_equal(tr.data, np.concatenate([b.data for b in batches]))
    np.testing.assert_array_equal(tr.data_per_streamline['flags'],
                                  np.concatenate([b.data_per_streamline['flags'] for b in batches]))
    assert total_steps == int((env.lengths - 1).sum())
    assert env.n_alive() == 0


def test_tracker_track_filters_and_transforms():
    from tracktolearn_b200.tracking.tracker import Tracker, streamline_lengths
    env, alg, sub, seeds, sd = _setup(precision='bf16')
    tracker = Tracker(alg, 256, min_length=5, max_length=200, save_seeds=True)
    np.random.seed(0)
    items = list(tracker.track(env, 'trk'))
    assert len(items) > 100
    for it in items[:20]:
        L = O.streamline_length(it.streamline)
        assert 5 <= L <= 200
        assert it.data_for_streamline['seeds'].shape == (3,)
    # same seeds through track_packed: lengths agree with the oracle's dipy-length restatement
    batch = next(tracker.track_packed(env))
    lens = streamline_lengths(batch.data, batch.offsets)
    ref = np.asarray([O.streamline_length(s) for s in batch.streamlines])
    np.testing.assert_allclose(lens, ref, rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize('prec', TC)
def test_bf16_only_state_mode_tracks_the_same_streamlines(prec):
    """Streaming with the fp32 state tensor materialised vs the operand-only mode (channel-padded
    operand layout, permuted first-layer weights): same operand values, only the K order of the
    first GEMM differs, so trajectories agree to float rounding."""
    env, alg, sub, seeds, sd = _setup(precision=prec)
    n = len(seeds)
    st = env.reset_streaming(0, n, 256, fp32_state=True)
    alg.validation_episode(st, env, 0.0)
    a = env.get_streamlines()
    st = env.reset_streaming(0, n, 256, fp32_state=False)
    assert st is None and env.current_state() is None and env.bf16_layout[0] == 1
    alg.validation_episode(st, env, 0.0)
    b = env.get_streamlines()
    same = a.lengths == b.lengths
    assert same.mean() > 0.98, same.mean()
    worst = 0.0
    for i in np.nonzero(same)[0]:
        worst = max(worst, float(np.abs(a.streamlines[i] - b.streamlines[i]).max()))
    assert worst < 5e-2, worst
    assert (a.data_per_streamline['flags'] == b.data_per_streamline['flags'])[same].all()


@pytest.mark.parametrize('prec', TC)
def test_fused_head_step_is_bit_identical_to_action_round_trip(prec):
    """Device loop with the env step reading tanh(mu) from the actor's fused output layer
    (ttl_env_step with the head partials) vs actor -> action buffer -> ttl_env_step: same streamlines, bit for bit,
    in both state modes."""
    env, alg, sub, seeds, sd = _setup(precision=prec)
    n = len(seeds)
    for fp32_state in (True, False):
        out = []
        for fuse in (True, False):
            alg.fuse_head = fuse
            st = env.reset_streaming(0, n, 256, fp32_state=fp32_state)
            alg.validation_episode(st, env, 0.0)
            assert alg._runner.fuse_head == fuse
            out.append(env.get_streamlines())
        a, b = out
        np.testing.assert_array_equal(a.lengths, b.lengths)
        np.testing.assert_array_equal(a.data, b.data)
        np.testing.assert_array_equal(a.data_per_streamline['flags'], b.data_per_streamline['flags'])
    alg.fuse_head = True


@pytest.mark.parametrize('prec', TC)
def test_bf16_direction_block_is_the_rounded_point_differences(prec):
    """Device mode builds the previous-direction block of a state row by shifting the previous row's
    block (bf16) and putting the newest direction in front.  After a number of steps with refills it
    must equal, bit for bit, bf16(points[L-1-k] - points[L-2-k]) recomputed from the fp32 streamline
    buffer (env.py:549-563), zero padded."""
    from tracktolearn_b200.algorithms.rl import StepRunner
    env, alg, sub, seeds, sd = _setup(precision=prec)
    n = len(seeds)
    env.reset_streaming(0, n, 256, fp32_state=False)
    runner = StepRunner(env, alg.agent.actor, 0.0, use_graph=False)
    checked_long = False
    for step in range(1, 41):
        runner.step()
        if step not in (1, 2, 7, 40):
            continue
        n_alive = env.n_alive()
        assert n_alive > 0
        bb = env._batch
        rows = bb.alive[env._cur][:n_alive].cpu().numpy()
        npts = bb.npts.cpu().numpy()[rows]
        pts = bb.points.cpu().numpy()[rows]
        assert bb.state_bf16[env._cur].dtype == OP_DTYPE[prec]
        got = bb.state_bf16[env._cur][:n_alive].float().cpu().numpy()
        want = np.zeros((n_alive, 304), dtype=np.float32)
        for a in range(n_alive):
            L = int(npts[a])
            d = np.diff(pts[a, :L], axis=0)[::-1][:100]          # newest first
            want[a, :d.size] = d.reshape(-1)
        want = _round_like_operand(want, prec)
        np.testing.assert_array_equal(got[:, 336:640], want)
        checked_long = checked_long or int(npts.max()) > 10
    assert checked_long


@pytest.mark.parametrize('prec', TC)
def test_cuda_graph_replay_equals_plain_launches(prec):
    """validation_episode with the step replayed from two captured CUDA graphs (one per ping-pong
    parity; programmatic-dependent-launch edges inside) vs plain launches: same streamlines."""
    env, alg, sub, seeds, sd = _setup(precision=prec)
    n = len(seeds)
    out = []
    try:
        for graph in (False, True):
            alg.use_cuda_graph = graph
            st = env.reset_streaming(0, n, 256, fp32_state=False)
            alg.validation_episode(st, env, 0.0)
            if graph:
                assert alg._runner.graphs is not None and alg._runner.replays > 10
            out.append(env.get_streamlines())
    finally:
        alg.use_cuda_graph = False
    a, b = out
    np.testing.assert_array_equal(a.lengths, b.lengths)
    np.testing.assert_array_equal(a.data, b.data)
    np.testing.assert_array_equal(a.data_per_streamline['flags'], b.data_per_streamline['flags'])


@pytest.mark.parametrize('prec', TC)
def test_locality_order_does_not_change_any_streamline(prec):
    """Streaming tracker with the seeds entering the slots in voxel raster order (ttl_batch.order) vs
    in row order: every row holds the same streamline, bit for bit, and the output order is the
    rows' (shuffled) order in both."""
    env, alg, sub, seeds, sd = _setup(precision=prec)
    n = len(seeds)
    out = []
    for loc in (False, True):
        st = env.reset_streaming(0, n, 256, fp32_state=False, locality=loc)
        assert (env._order_dev is not None) == loc
        if loc:
            order = env._order_dev.cpu().numpy()
            assert sorted(order.tolist()) == list(range(n))
            first = env._batch.alive[0][:256].cpu().numpy()
            np.testing.assert_array_equal(first, order[:256])
        alg.validation_episode(st, env, 0.0)
        out.append(env.get_streamlines())
        assert env.streamline_steps() == int((env.lengths - 1).sum())
    a, b = out
    np.testing.assert_array_equal(a.lengths, b.lengths)
    np.testing.assert_array_equal(a.data, b.data)
    np.testing.assert_array_equal(a.data_per_streamline['flags'], b.data_per_streamline['flags'])
    np.testing.assert_array_equal(a.data_per_streamline['seeds'], b.data_per_streamline['seeds'])


def test_training_episode_rollout_replay_and_update():
    """A3 / config 4: DDPG._episode-style rollout with the tensor-core actor sampling at
    probabilistic=1, transitions pushed to the device replay buffer, one SAC update per env step,
    weights shared between learner and inference actor."""
    from tests.gpu_helpers import make_gpu_env
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    shape = (24, 26, 22)
    sub = {k: (v.numpy() if v is not None else None) for k, v in synthetic.make_subject(shape, seed=11).items()}
    rs = np.random.RandomState(3)
    seeds = synthetic.seeds_from_mask(synthetic.ellipsoid_mask(shape, frac=0.3).numpy(), 1, rs)
    g = {'meta_shape': np.asarray(shape), 'meta': np.asarray([1.0, 0.75, 30.0, 30.0, 0.1, 40.0, 0.75])}
    env, _ = make_gpu_env(g, False, True, sub=sub, seeds=seeds)
    alg = SACAuto(615, 3, '128-128-128', n_actors=200, device=torch.device('cuda:0'), precision='bf16')
    alg.agent.actor.load_state_dict(synthetic.actor_state_dict(615, '128-128-128', seed=5, kind='tracking'))
    learner = alg.enable_training(replay_size=20000, batch_size=256, start_timesteps=150)
    w_before = learner.actor.layers[0].weight.detach().clone()
    np.random.seed(0)
    torch.manual_seed(0)
    state = env.nreset(200)
    reward, losses, length, _ = alg._episode(state, env)
    assert length >= 3 and len(alg.replay_buffer) == alg.t - 1
    assert len(losses) >= 1 and all(np.isfinite(float(l['critic_loss'])) for l in losses)
    assert not torch.equal(w_before, learner.actor.layers[0].weight)
    # transitions are consistent: next_state of a surviving streamline at step t is a state at t+1
    rb = alg.replay_buffer
    n0 = 200
    first_next = rb.next_state[:n0]
    alive0 = rb.not_done[:n0, 0] > 0
    second_states = rb.state[n0:n0 + int(alive0.sum())]
    torch.testing.assert_close(first_next[alive0], second_states, rtol=0, atol=0)
    assert float(rb.reward[:len(rb)].abs().sum()) > 0
    # inference actor == learner's torch actor after the updates (bf16 tolerance)
    st = rb.state[:64]
    mu_ref = torch.tanh(learner.actor.layers(st)[:, :3])
    a_inf = alg.agent.select_action(st, 0.0)
    assert (a_inf - mu_ref).abs().max().item() < 2e-2
