"""TrackingEnvironment on the device (reference: environments/tracking_env.py:13-294).

``reset / nreset / step / harvest / get_streamlines`` keep the reference's signatures and
return types (state: torch tensor on the env's device; reward / dones / continue_idx: numpy).
Underneath, everything -- streamline buffer, flags, alive list, state rows -- lives in HBM and
one ``step`` is three kernel launches through the C ABI (``ttl_env_step``).

Two ways to drive it:
  * the reference protocol: ``step(actions) -> (state, reward, dones, info)`` then
    ``harvest() -> (state, not_stopping)``; host arrays are produced on every call, which
    costs a few small D2H copies per step (what the parity tests use);
  * the device protocol used by ``Tracker``/``validation_episode`` in this package:
    ``step_device(actions)`` + ``harvest_device()`` enqueue kernels only and never touch the
    host; ``n_alive()`` reads the alive count back when the loop wants to know.
"""
import ctypes
import os

import numpy as np
import torch

from tracktolearn_b200 import _lib
from tracktolearn_b200.environments.env import BaseEnv
from tracktolearn_b200.tracking.tractogram import Tractogram


GUARD_BYTES = 4096
GUARD_FILL = 0xA5


class _BatchBuffers(object):
    """Device buffers of one batch of streamlines (``ttl_batch`` in include/ttl_b200.h).

    ``rows``: seeds held by the batch (one streamline buffer row each); ``slots``: streamlines
    tracked at once (== rows unless the streaming tracker refills freed slots).

    ``GUARD`` (class attribute, or TTL_GUARD=1): every buffer is carved out of a larger allocation with
    4 KB of 0xA5 on either side and ``check_guards()`` verifies that no kernel wrote there -- the
    out-of-bounds check this package can run itself (compute-sanitizer is not available on every pool)."""

    GUARD = os.environ.get('TTL_GUARD', '0') == '1'

    def _zeros(self, shape, dtype, device):
        if not self.GUARD:
            return torch.zeros(shape, dtype=dtype, device=device)
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        body = (n + 255) // 256 * 256
        raw = torch.full((body + 2 * GUARD_BYTES,), GUARD_FILL, dtype=torch.uint8, device=device)
        self._guarded.append((raw, n))
        view = raw[GUARD_BYTES:GUARD_BYTES + n].view(dtype).view(shape)
        view.zero_()
        return view

    def check_guards(self):
        """Names nothing: returns the number of guard bytes that were overwritten (0 = clean)."""
        bad = 0
        for raw, n in self._guarded:
            bad += int((raw[:GUARD_BYTES] != GUARD_FILL).sum().item())
            bad += int((raw[GUARD_BYTES + n:] != GUARD_FILL).sum().item())
        return bad

    def __init__(self, rows, slots, max_pts, state_size, device, fp32_state=True, operand='bf16'):
        self._guarded = []
        self.fp32_state = fp32_state
        self.operand = operand          # element type of the actor operand rows: 'bf16' / 'fp16' / 'tf32'
        if operand not in _lib.OPERAND_OF_PRECISION:
            raise ValueError('operand rows come in bf16, fp16 or tf32, not %r' % (operand,))
        if fp32_state and operand == 'tf32':
            raise ValueError('tf32 operand rows exist in the operand-only mode; with fp32 state rows a tf32 '
                             'actor packs its operand from them')
        self.rows = rows
        self.slots = slots
        self.max_pts = max_pts
        self.state_size = state_size
        self.ld_state = (state_size + 3) // 4 * 4
        i32 = (torch.int32, device)
        pad = (slots + 127) // 128 * 128 + 16   # stop[] is read in whole 128-rank groups
        self.points = self._zeros((rows, max_pts, 3), torch.float32, device)
        self.flags = self._zeros((rows,), *i32)
        self.lengths = self._zeros((rows,), *i32)
        self.npts = self._zeros((rows,), *i32)
        self.dones = self._zeros((rows,), torch.uint8, device)
        self.alive = [self._zeros((pad,), *i32), self._zeros((pad,), *i32)]
        self.ctrl = self._zeros((16,), *i32)
        self.stop = self._zeros((pad,), torch.uint8, device)
        self.dest = self._zeros((pad,), *i32)
        self.step_flags = self._zeros((pad,), *i32)
        self.reward = self._zeros((pad,), torch.float32, device)
        # fp32 state rows (the API's state tensor).  Without them the step kernel produces only the
        # bf16 rows, in the channel-padded column layout (ttl_batch.bf16_layout = 1).
        self.state = ([self._zeros((slots, self.ld_state), torch.float32, device),
                       self._zeros((slots, self.ld_state), torch.float32, device)]
                      if fp32_state else [None, None])
        self.ctrl_host = torch.zeros((16,), dtype=torch.int32).pin_memory()
        # copy of the state rows in the actor's operand type, zero padded to a multiple of 64 columns:
        # the actor's TMA operand
        self.ld_bf16 = (state_size + 63) // 64 * 64
        op_dtype = {'bf16': torch.bfloat16, 'fp16': torch.float16, 'tf32': torch.float32}[operand]
        self.state_bf16 = [self._zeros((slots, self.ld_bf16), op_dtype, device),
                           self._zeros((slots, self.ld_bf16), op_dtype, device)]
        self.max_groups = (slots + 31) // 32 + 1
        self.grp_stops = self._zeros((self.max_groups,), *i32)
        self.sg_stops = self._zeros((2 * ((self.max_groups + 63) // 64),), *i32)
        # per-rank records {row, npts, tip, previous point} of the two alive lists and the points added
        # by the step in flight (ttl_batch.rank_rec / step_tip)
        self.rank_rec = [self._zeros((pad, 8), torch.float32, device),
                         self._zeros((pad, 8), torch.float32, device)]
        self.step_tip = self._zeros((pad, 4), torch.float32, device)

    def as_struct(self, n, n_slots):
        b = _lib.Batch(n=n, n_slots=n_slots, capacity=self.rows, max_pts=self.max_pts,
                       ld_state=self.ld_state, state_size=self.state_size,
                       points=self.points.data_ptr(), flags=self.flags.data_ptr(),
                       lengths=self.lengths.data_ptr(), npts=self.npts.data_ptr(),
                       dones=self.dones.data_ptr(), ctrl=self.ctrl.data_ptr(),
                       stop=self.stop.data_ptr(), dest=self.dest.data_ptr(),
                       step_flags=self.step_flags.data_ptr(), reward=self.reward.data_ptr(),
                       ld_bf16=self.ld_bf16, max_groups=self.max_groups,
                       grp_stops=self.grp_stops.data_ptr(), sg_stops=self.sg_stops.data_ptr(),
                       operand_fmt=_lib.OPERAND_OF_PRECISION[self.operand])
        b.state_bf16[0] = self.state_bf16[0].data_ptr()
        b.state_bf16[1] = self.state_bf16[1].data_ptr()
        b.rank_rec[0] = self.rank_rec[0].data_ptr()
        b.rank_rec[1] = self.rank_rec[1].data_ptr()
        b.step_tip = self.step_tip.data_ptr()
        b.alive[0] = self.alive[0].data_ptr()
        b.alive[1] = self.alive[1].data_ptr()
        if self.fp32_state:
            b.state[0] = self.state[0].data_ptr()
            b.state[1] = self.state[1].data_ptr()
        b.bf16_layout = 0 if self.fp32_state else 1
        return b


class TrackingEnvironment(BaseEnv):
    """Reference: environments/tracking_env.py:13."""

    # Counter-based draws made on the device (the stochastic policy, ttl_policy; device tracking noise,
    # ttl_noise) are keyed by g = row_base + batch row.  ``seed_offset``: global index of seeds[0] in the seed
    # list the whole run shares (Tracker.track_to_file sets it when it shards the seeds over processes).
    # reset / reset_streaming(start, end) use row_base = seed_offset + start, so a seed keeps its index
    # whichever pass or shard tracks it; nreset uses 0.
    seed_offset = 0
    _row_base = 0

    # ------------------------------------------------------------------------------ reset
    def _ensure_buffers(self, rows, slots, fp32_state=True, operand='bf16'):
        need_pts = self.max_nb_steps + 1
        S = self.get_state_size()
        bb = self._batch
        if (bb is None or bb.rows < rows or bb.slots < slots or bb.max_pts != need_pts
                or bb.state_size != S or bb.fp32_state != fp32_state or bb.operand != operand):
            rows = max(rows, bb.rows if bb is not None else 0)
            slots = max(slots, bb.slots if bb is not None else 0)
            self._batch = None
            bb = _BatchBuffers(rows, slots, need_pts, S, self.device, fp32_state, operand)
            self._batch = bb
        return bb

    def _start(self, initial_points, n_slots=None, fp32_state=True, locality=False, operand=None):
        """``n_slots`` < N turns on the streaming tracker: only n_slots streamlines are alive
        at once and slots freed by stopped ones take the next seeds in the same step.
        ``fp32_state=False``: only the actor's operand rows are produced (no fp32 state tensor), in the
        element type ``operand`` ('bf16', 'fp16' or 'tf32'; default: the env's ``operand`` attribute).
        ``locality``: seeds take slots in voxel raster order instead of row order (ttl_batch.order);
        rows, results and the output order are unchanged."""
        if not fp32_state and (self._n_coefs != 45 or 7 * 48 + 3 * self.n_dirs > (self.get_state_size() + 63) // 64 * 64):
            fp32_state = True      # the operand-only layout is specialised for the order-8 volume
        operand = operand or getattr(self, 'operand', 'bf16')
        if fp32_state and operand == 'tf32':
            operand = 'bf16'       # unused copy: a tf32 actor packs from the fp32 rows
        if operand == 'fp16' and not fp32_state and not (getattr(self, '_sh_absmax', 0.0) <= 65504.0):
            raise _lib.TTLError('the SH volume holds values outside the fp16 range (max |c| = %g): fp16 operand '
                                'rows would saturate; use precision="tf32"' % self._sh_absmax)
        self.initial_points = initial_points
        N = initial_points.shape[0]
        streaming = n_slots is not None and n_slots < N
        slots = n_slots if streaming else max(N, 1)
        bb = self._ensure_buffers(max(N, 1), slots, fp32_state, operand)
        self._n = N
        self._b = bb.as_struct(N, slots)
        self._params.refill = int(streaming)
        self._params.state_stopped = int(bool(self.state_of_stopped) and not streaming)
        self._cur = 0
        self.length = 1
        self._n_alive_host = min(N, slots)   # host mirror of the alive count (upper bound between syncs)
        self._n_prev = self._n_alive_host
        self._continue_idx_cache = np.arange(self._n_alive_host)
        self._pending_harvest = False
        seeds_host = np.ascontiguousarray(initial_points, dtype=np.float64)
        seeds_dev = (torch.from_numpy(seeds_host).pin_memory().to(self.device, non_blocking=True)
                     if not isinstance(initial_points, torch.Tensor)
                     else initial_points.to(self.device, dtype=torch.float64, non_blocking=True))
        self._order_dev = None
        if locality and N > 1:
            # voxel of every seed (centre origin: voxel i spans [i-.5, i+.5]), raster key, stable sort
            vox = torch.floor(seeds_dev + 0.5).to(torch.int64)
            key = (vox[:, 0] * int(self._volume.Y) + vox[:, 1]) * int(self._volume.Z) + vox[:, 2]
            self._order_dev = torch.argsort(key, stable=True).to(torch.int32)
            self._b.order = self._order_dev.data_ptr()
            self._continue_idx_cache = None
        _lib.check(self._lib.ttl_env_reset(ctypes.byref(self._volume), ctypes.byref(self._params),
                                           ctypes.byref(self._b), _lib.ptr(seeds_dev),
                                           _lib.stream_ptr(self.device)), 'ttl_env_reset')
        self._seeds_dev = seeds_dev   # keep alive until the kernel ran
        return self._state_view(0, self._n_alive_host) if bb.fp32_state else None

    def _state_view(self, which, n):
        return self._batch.state[which][:n, :self._batch.state_size]

    def reset(self, start, end):
        """Reference: tracking_env.py:91-133."""
        self._row_base = int(self.seed_offset) + int(start)
        return self._start(self.seeds[start:end])

    def reset_streaming(self, start, end, n_slots, fp32_state=True, locality=True, operand=None):
        """Like ``reset`` but at most ``n_slots`` streamlines are tracked at once; the others
        wait in the batch and take over slots as streamlines stop (device-side refill).
        With ``fp32_state=False`` the fp32 state tensor is not materialised: the step kernel
        writes the actor's bf16 operand only (``current_state_bf16()``).
        ``locality`` (default): seeds enter the slots in voxel raster order, so streamlines that are
        neighbours in the alive list start in the same or adjacent voxels and their trilinear
        gathers share cache lines (the reference shuffles the seeds, tracker.py:94; the rows -- and
        with them every per-seed result and the output order -- stay in the shuffled order)."""
        self._row_base = int(self.seed_offset) + int(start)
        return self._start(self.seeds[start:end], n_slots=n_slots, fp32_state=fp32_state,
                           locality=locality and os.environ.get('TTL_LOCALITY', '1') != '0', operand=operand)

    def nreset(self, n_seeds):
        """Reference: tracking_env.py:47-89.  Random seeds with replacement: the rows are not seed-list
        indices, so device draws use row_base = 0 (row i of the batch is g = i)."""
        self._row_base = 0
        replace = n_seeds > len(self.seeds)
        seeds = np.random.choice(np.arange(len(self.seeds)), size=n_seeds, replace=replace)
        return self._start(self.seeds[seeds])

    # ------------------------------------------------------------------- device protocol
    def _device_noise(self):
        """``_lib.Noise`` when the step kernels draw the noise themselves (ttl_noise), else None."""
        return None

    def policy(self, seed, prob):
        """``_lib.Policy`` for the current batch: the stochastic policy with std scaled by ``prob``, its eps
        drawn from ``seed`` at (row_base + batch row, point count) -- ttl_policy in include/ttl_b200.h."""
        return _lib.Policy(seed=int(seed), row_base=int(self._row_base), prob=float(prob))

    def step_device(self, actions=None, noise=None, head=None, policy=None):
        """Enqueue one step for the alive rows (ttl_env_step).  No host synchronisation.  The actions come from
        ``actions``: CUDA float32 tensor [>= n_alive, >= 3] (row stride taken from the tensor), with an
        optional host-drawn ``noise`` array; or from ``head``, what ``actor.forward_head_partial`` returned:
        tanh(mu) read straight from the actor's fused output layer, one launch less per step and the same
        bits as forward_device + step_device.  ``policy`` (``self.policy(seed, prob)``, with ``head`` only):
        the stochastic policy sampled inside the step kernel; ``head`` must then hold all six outputs
        (``forward_head_partial(..., policy=True)``), and gives the same bits as ``policy_eps`` + the actor's
        head + step.  Device-drawn tracking noise, if any, is added on top."""
        if self._pending_harvest:
            raise RuntimeError('step() called twice without harvest()')
        if (actions is None) == (head is None):
            raise ValueError('step_device takes either actions or head')
        nz = self._device_noise()
        if nz is not None and noise is not None:
            raise ValueError('the step kernels draw the noise of this environment; no noise array is taken')
        if head is not None:
            if self._oracle is not None:
                raise RuntimeError('the fused-head step does not consult the oracle; pass actions')
            if getattr(self, 'noise', 0.0) > 0.0 and nz is None:
                raise RuntimeError('host-drawn noise arrives as an array: use policy_eps and actions')
            partial, n_tiles, tiles_per_256, bias = head
            act = _lib.StepAction(head_partial=partial, head_bias=bias, n_tiles=int(n_tiles),
                                  tiles_per_256=int(tiles_per_256))
        else:
            if actions.dtype != torch.float32 or actions.device != self.device or actions.stride(-1) != 1:
                actions = actions.to(self.device, dtype=torch.float32).contiguous()
            lda = actions.stride(0) if actions.dim() == 2 and actions.shape[0] > 1 else actions.shape[-1]
            act = _lib.StepAction(actions=actions.data_ptr(), lda=int(lda))
        sp = _lib.stream_ptr(self.device)
        n_up = int(self._n_alive_host)
        # with the oracle: propagate + geometric criteria, then score every alive streamline, then ORACLE flag /
        # bonus / compaction / state rows
        defer = int(self._oracle is not None)
        _lib.check(self._lib.ttl_env_step(
            ctypes.byref(self._volume), ctypes.byref(self._params), ctypes.byref(self._b), self._cur,
            ctypes.byref(act), _lib.ptr(noise), None if nz is None else ctypes.byref(nz),
            None if policy is None else ctypes.byref(policy), defer, n_up, sp), 'ttl_env_step')
        if defer and n_up > 0:
            slots = self._b.n_slots
            if getattr(self, '_oracle_dirs', None) is None or self._oracle_dirs.shape[0] < slots:
                self._oracle_dirs = torch.empty((slots, 127, 3), dtype=torch.float32, device=self.device)
                self._oracle_scores = torch.zeros((slots,), dtype=torch.float32, device=self.device)
            _lib.check(self._lib.ttl_oracle_features_rows(ctypes.byref(self._b), self._cur, n_up,
                                                          _lib.ptr(self._oracle_dirs), sp),
                       'ttl_oracle_features_rows')
            self._oracle.forward_dirs(self._oracle_dirs, _lib.ptr(self._oracle_scores), n_up)
            bonus = float(self.oracle_bonus) if self.compute_reward else 0.0
            _lib.check(self._lib.ttl_env_step_finish(
                ctypes.byref(self._volume), ctypes.byref(self._params), ctypes.byref(self._b), self._cur,
                _lib.ptr(self._oracle_scores), int(bool(self.oracle_stopping_criterion)),
                int(self.min_nb_steps * 5), int(self.min_nb_steps), bonus, n_up, sp), 'ttl_env_step_finish')
        self._keep = (actions, noise)
        self.length += 1
        self._pending_harvest = True

    def policy_eps(self, policy, out):
        """Enqueue ttl_policy_eps: ``out`` (CUDA float32 [>= n_alive, >= 3], row stride from the tensor)
        gets, rank by rank of the current alive list, the eps the fused route would draw -- for
        ``actor.forward_device(..., eps=out)``."""
        if out.dtype != torch.float32 or out.device != self.device or out.stride(-1) != 1 or out.dim() != 2:
            raise ValueError('policy_eps writes a CUDA float32 [rows, >= 3] tensor on the env device')
        _lib.check(self._lib.ttl_policy_eps(ctypes.byref(policy), ctypes.byref(self._b), self._cur,
                                            int(self._n_alive_host), _lib.ptr(out), int(out.stride(0)),
                                            _lib.stream_ptr(self.device)), 'ttl_policy_eps')
        return out

    def harvest_device(self):
        """The flip that makes the compacted alive list / state rows current (harvest)."""
        if self._pending_harvest:
            self._cur ^= 1
            self._pending_harvest = False
            self._continue_idx_cache = None
        return self._batch.state[self._cur]

    def n_alive(self):
        """Alive count after the last harvest (one 32-byte D2H copy + stream sync)."""
        bb = self._batch
        bb.ctrl_host.copy_(bb.ctrl, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        n = int(bb.ctrl_host[self._cur])
        if self._params.refill and int(bb.ctrl_host[6]) < self._n:
            # seeds are still waiting: later steps can have up to n_slots rows again
            self._n_alive_host = self._b.n_slots
        else:
            self._n_alive_host = n
        return n

    def streamline_steps(self):
        """Total streamline-steps taken since reset (device counter, valid after n_alive())."""
        h = self._batch.ctrl_host
        return (int(h[4]) & 0xffffffff) | (int(h[5]) << 32)

    def current_state(self):
        """State rows of the alive set, [n_alive_upper_bound, state_size] view (no sync).
        None when the batch was started without fp32 state rows."""
        if not self._batch.fp32_state:
            return None
        return self._state_view(self._cur, self._n_alive_host)

    @property
    def bf16_layout(self):
        """(layout id, C, CP, n_points) of ``current_state_bf16()`` rows."""
        return (0 if self._batch.fp32_state else 1, self._n_coefs, self._volume.CP, 7)

    def current_state_bf16(self):
        """Zero-padded copy of ``current_state()`` in the actor's operand type
        ([slots, round_up(state_size, 64)], dtype bf16 / fp16 / fp32-holding-tf32, see ``operand_format``)
        that the step kernel writes alongside (or instead of) the fp32 rows; the actor's first layer
        reads it by TMA."""
        return self._batch.state_bf16[self._cur]

    @property
    def operand_format(self):
        return self._batch.operand

    def operand_saturated(self):
        """True when fp16 operand rows cannot hold this volume's states: a state value is a convex
        combination of SH coefficients (trilinear weights) or a step vector, so the volume's largest
        coefficient magnitude, taken once at load time, bounds every value a row can hold."""
        return self._batch is not None and self._batch.operand == 'fp16' and \
            not (getattr(self, '_sh_absmax', 0.0) <= 65504.0)

    def alive_count_tensor(self):
        """Device int32 tensor holding the alive count of the current list."""
        return self._batch.ctrl[self._cur:self._cur + 1]

    # ---------------------------------------------------------------- reference protocol
    @property
    def continue_idx(self):
        if self._continue_idx_cache is None:
            n = self._n_alive_host
            self._continue_idx_cache = self._batch.alive[self._cur][:n].cpu().numpy().astype(np.int64)
        return self._continue_idx_cache

    def _host_actions(self, actions):
        if isinstance(actions, np.ndarray):
            return torch.from_numpy(np.ascontiguousarray(actions, dtype=np.float32)).to(self.device)
        return actions

    def step(self, actions):
        """Reference: tracking_env.py:135-221."""
        return self._step(self._host_actions(actions), None)

    def _step(self, actions, noise):
        A = self._n_alive_host
        ci = self.continue_idx
        self.step_device(actions, noise)
        bb = self._batch
        S = bb.state_size
        state = torch.empty((A, S), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ttl_env_gather_step_state(ctypes.byref(self._b), self._cur, A,
                                                       _lib.ptr(state), S, _lib.stream_ptr(self.device)),
                   'ttl_env_gather_step_state')
        stop = bb.stop[:A].cpu().numpy().astype(bool)
        self.not_stopping = np.logical_not(stop)
        self.new_continue_idx, self.stopping_idx = ci[~stop], ci[stop]
        reward_info = {}
        if self.compute_reward:
            reward = bb.reward[:A].cpu().numpy().astype(np.float64)
            reward_info = {'peaks_reward': float(np.mean(reward)) if A else 0.0, 'oracle_reward': 0.0}
        else:
            reward = np.zeros(self._n)          # the reference's shape quirk (tracking_env.py:204)
        self._n_prev = A
        return state, reward, stop, {'continue_idx': ci, 'reward_info': reward_info}

    def harvest(self):
        """Reference: tracking_env.py:223-245."""
        self.harvest_device()
        n = self.n_alive()
        self._continue_idx_cache = getattr(self, 'new_continue_idx', None)
        return self._state_view(self._cur, n), self.not_stopping

    # --------------------------------------------------------------------- results
    @property
    def flags(self):
        return self._batch.flags[:self._n].cpu().numpy().astype(int)

    @property
    def lengths(self):
        return self._batch.lengths[:self._n].cpu().numpy()

    @property
    def dones(self):
        return self._batch.dones[:self._n].cpu().numpy().astype(bool)

    @property
    def streamlines(self):
        """[N, max_nb_steps+1, 3] float32 host copy of the streamline buffer."""
        return self._batch.points[:self._n].cpu().numpy()

    def get_streamlines_device(self):
        """Packed streamlines on the device: (points [sum(L),3] fp32, offsets [N+1] int64)."""
        N = self._n
        offsets = torch.empty((N + 1,), dtype=torch.int64, device=self.device)
        sp = _lib.stream_ptr(self.device)
        _lib.check(self._lib.ttl_streamline_offsets(ctypes.byref(self._b), _lib.ptr(offsets), sp),
                   'ttl_streamline_offsets')
        total = int(offsets[N].item())
        pts = torch.empty((max(total, 1), 3), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ttl_pack_streamlines(ctypes.byref(self._b), _lib.ptr(offsets), _lib.ptr(pts), sp),
                   'ttl_pack_streamlines')
        return pts[:total], offsets

    def _pinned(self, name, numel, dtype):
        """Cached page-locked staging buffer (grown geometrically) for device->host copies."""
        cache = self.__dict__.setdefault('_pinned_cache', {})
        buf = cache.get(name)
        if buf is None or buf.numel() < numel or buf.dtype != dtype:
            buf = torch.empty((max(int(numel * 1.25), 1024),), dtype=dtype).pin_memory()
            cache[name] = buf
        return buf[:numel]

    def get_streamlines(self, copy=True):
        """Reference: tracking_env.py:247-294.  The last point is dropped when the CURVATURE or
        MASK flag stopped the streamline.  One packed D2H copy through pinned memory; with
        ``copy=False`` the returned arrays are views of that staging memory and are only valid
        until the next call."""
        pts, offsets = self.get_streamlines_device()
        N = self._n
        h_pts = self._pinned('pts', pts.numel(), torch.float32)
        h_off = self._pinned('off', N + 1, torch.int64)
        h_flags = self._pinned('flags', N, torch.int32)
        h_pts.copy_(pts.reshape(-1), non_blocking=True)
        h_off.copy_(offsets, non_blocking=True)
        h_flags.copy_(self._batch.flags[:N], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        data, off = h_pts.numpy().reshape(-1, 3), h_off.numpy()
        if copy:
            data, off = data.copy(), off.copy()
        return Tractogram(data=data, offsets=off,
                          data_per_streamline={'seeds': np.asarray(self.initial_points),
                                               'flags': h_flags.numpy().astype(int)})
