"""Episode drivers (reference: algorithms/rl.py:58-106, the act -> step -> harvest loop).

The reference crosses the host/device boundary three times per step (action D2H with a
sync, coordinates H2D, previous directions H2D).  Here the loop only enqueues kernels: the
actor reads the alive count from device memory, the env step consumes the action tensor in
place, the launches of a step can be replayed from a CUDA graph, and the host learns the
alive count from asynchronous copies that lag a few steps behind (the queue never drains).
"""
import numpy as np
import torch


class StepRunner(object):
    """One act -> step -> harvest iteration of `env` with `actor`, enqueue-only.

    With ``use_graph`` the iteration is captured once per parity of the env's ping-pong
    buffers (two CUDA graphs) and replayed; that needs launch shapes that do not change, so the
    launches are sized for ``n_slots`` rows and rows beyond the device-side alive count exit
    early.  Capturing does not execute anything: the two captures flip the env's host-side
    parity twice, so host and device stay consistent."""

    def __init__(self, env, actor, prob=0.0, use_graph=True, fuse_head=True):
        self.env, self.actor, self.prob = env, actor, prob
        self.action_buf = torch.empty((env._b.n_slots, actor.action_dim), dtype=torch.float32,
                                      device=env.device)
        # host-drawn noise arrives as an array per step: no fused head, nothing to replay.  Noise the step
        # kernel draws itself (noise_rng = 'device') needs neither restriction.
        noisy = getattr(env, 'noise', 0.0) > 0.0 and env._device_noise() is None
        self.use_graph = bool(use_graph) and prob == 0.0 and not noisy and not env.compute_reward \
            and env._oracle is None
        self.graphs = None
        self.warm = 0
        self.replays = 0
        self.kernels_per_step = 0
        self._lib = __import__('tracktolearn_b200._lib', fromlist=['load']).load()
        # deterministic tracking: the env step reads tanh(mu) straight from the actor's fused output
        # layer (one launch and one HBM round trip less per step; same bits)
        self.fuse_head = prob == 0.0 and not noisy and env._oracle is None and fuse_head \
            and hasattr(actor, 'forward_head_partial')

    def _one(self, rows):
        env = self.env
        if self.fuse_head:
            head = self.actor.forward_head_partial(env.current_state_bf16(), rows,
                                                   n_rows_dev=env.alive_count_tensor(), layout=env.bf16_layout,
                                                   state=env.current_state())
            if head is not None:
                env.step_device_head(head)
                env.harvest_device()
                return
            self.fuse_head = False
        self.actor.forward_device(env.current_state(), self.prob, n_rows_dev=env.alive_count_tensor(),
                                  n_rows=rows, want_logp=False, out_action=self.action_buf,
                                  state_bf16=env.current_state_bf16(), layout=env.bf16_layout)
        env.step_device(self.action_buf)
        env.harvest_device()

    def _capture(self):
        env = self.env
        assert env._cur == 0 or env._cur == 1
        first = env._cur
        saved_upper, saved_len = env._n_alive_host, env.length
        env._n_alive_host = env._b.n_slots          # fixed launch shape
        graphs = {}
        n0 = self._lib.ttl_launch_count()
        for _ in range(2):
            g = torch.cuda.CUDAGraph()
            cur = env._cur
            with torch.cuda.graph(g):
                self._one(env._b.n_slots)
            graphs[cur] = g
        assert env._cur == first
        self.kernels_per_step = int(self._lib.ttl_launch_count() - n0) // 2
        env._n_alive_host, env.length = saved_upper, saved_len
        self.graphs = graphs

    def step(self):
        env = self.env
        if not self.use_graph:
            self._one(env._n_alive_host)
            return
        if self.graphs is None:
            if self.warm < 2:                       # warm path: lazy plans / attributes / TMA maps
                self._one(env._n_alive_host)
                self.warm += 1
                return
            self._capture()
        self.graphs[env._cur].replay()
        self.replays += 1
        env._cur ^= 1                               # what harvest_device() does
        env.length += 1
        env._continue_idx_cache = None


class RLAlgorithm(object):
    """Reference: algorithms/rl.py:8-56 (constructor arguments kept)."""

    def __init__(self, input_size, action_size=3, hidden_size=256, lr=3e-4, gamma=0.99,
                 batch_size=10000, rng=None, device=None):
        self.max_action = 1.
        self.t = 1
        self.action_size = action_size
        self.lr = lr
        self.gamma = gamma
        self.device = device
        self.batch_size = batch_size
        self.rng = rng
        self.sync_every = 8
        # CUDA-graph replay of the step is available but off: measured on B200 the loop is
        # GPU-bound even in the low-occupancy tail (800k-seed episode: 330 ms plain vs 323-331 ms
        # replayed), so the capture cost buys nothing
        self.use_cuda_graph = False
        # deterministic episodes read tanh(mu) straight from the actor's fused output layer
        self.fuse_head = True
        self._snap_ring = None
        self._runner = None
        self._runner_key = None

    def _runner_for(self, env, actor, prob, use_graph):
        """The captured graphs hold raw pointers into the env's batch buffers and the actor's plan:
        keep one runner per (buffers, plan) and reuse it across episodes."""
        nz = env._device_noise()      # a captured graph holds the noise parameters by value
        key = (id(env), id(env._batch), env._b.n_slots, env._batch.fp32_state, id(actor), id(actor._plan), prob,
               bool(use_graph), bool(getattr(self, 'fuse_head', True)),
               None if nz is None else (nz.sigma, nz.seed, nz.row_base))
        if getattr(self, '_runner_key', None) != key or self._runner is None:
            self._runner = StepRunner(env, actor, prob, use_graph=use_graph,
                                      fuse_head=getattr(self, 'fuse_head', True))
            self._runner_key = key
        elif self._runner.graphs is not None:
            env_cur = env._cur          # graphs were captured for both parities; nothing to redo
            assert env_cur in self._runner.graphs
        return self._runner

    def validation_episode(self, initial_state, env, prob=1., max_steps=None):
        """Run the agent until every streamline of the env's current batch is done.

        Reference: algorithms/rl.py:58-106.  ``initial_state`` is accepted for signature
        compatibility; the state rows are read from the env's device buffers.  Returns the
        cumulative reward (0 when the env does not compute rewards)."""
        actor = self.agent.actor
        running_reward = 0
        reward_acc = None
        if env._n_alive_host == 0:
            self.last_episode_steps = 0
            return running_reward
        # graphs pay off when the launch shapes are stable: the streaming tracker
        streaming = bool(env._params.refill)
        runner = self._runner_for(env, actor, prob, self.use_cuda_graph and streaming)
        bb = env._batch
        stream = torch.cuda.current_stream(env.device)
        pending = []          # (event, pinned ctrl snapshot, parity the snapshot describes)
        arange = None
        it = 0
        limit = max_steps if max_steps is not None else 1 << 30
        done = False
        while not done and it < limit:
            rows = env._n_alive_host
            runner.step()
            if env.compute_reward:
                # ctrl[3] = alive count the step just processed; rows beyond it hold stale rewards
                if arange is None or arange.shape[0] < rows:
                    arange = torch.arange(env._b.n_slots, device=env.device, dtype=torch.int32)
                live = arange[:rows] < bb.ctrl[3]
                r = torch.where(live, bb.reward[:rows], torch.zeros((), device=env.device)).sum(dtype=torch.float64)
                reward_acc = r if reward_acc is None else reward_acc + r
            it += 1
            if it % self.sync_every == 0:
                if self._snap_ring is None:
                    self._snap_ring = [torch.empty((16,), dtype=torch.int32).pin_memory() for _ in range(8)]
                snap = self._snap_ring[(it // self.sync_every) % 8]
                snap.copy_(bb.ctrl, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(stream)
                pending.append((ev, snap, env._cur))
            # consume the snapshots that have landed, oldest first, without blocking
            while pending and pending[0][0].query():
                _, snap, cur = pending.pop(0)
                alive = int(snap[cur])
                if env._params.refill and int(snap[6]) < env._n:
                    env._n_alive_host = env._b.n_slots      # seeds still waiting
                else:
                    env._n_alive_host = min(env._n_alive_host, alive)   # alive only decreases now
                if alive == 0:
                    done = True
            if len(pending) > 3:                             # bounded lag
                pending[0][0].synchronize()
        env.n_alive()
        if reward_acc is not None:
            running_reward = float(reward_acc.item())
        self.last_episode_steps = it
        return running_reward

