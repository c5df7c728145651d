"""SAC actor/critic holder with the reference's checkpoint format and calling convention
(reference: algorithms/shared/offpolicy.py:234-482).

The actor forward -- the only dense contraction on the tracking path -- runs through
``ttl_actor_forward`` (csrc/ttl_actor.cu, csrc/ttl_mlp.cuh) on tcgen05 tensor cores with fp32 TMEM
accumulators.  ``precision`` picks the operand type:

  'fp16'  (default) 11 significant bits at the full 16-bit tensor rate; outputs within 1e-3 of the
          reference's fp32 arithmetic (measured ~5e-4 of the output scale).  Range +-65504: values
          outside saturate and raise a flag (``MaxEntropyActor.overflowed()``); re-run in 'tf32' then.
  'tf32'  the same 11 bits with fp32's range at half the tensor rate.
  'bf16'  8 significant bits: ~4e-3 of the output scale, outside the 1e-3 tolerance; kept for
          throughput comparisons.
  'fp32'  the reference's arithmetic on the CUDA cores (1e-5), used by the parity tests.

The critic is carried for checkpoint compatibility (``load`` reads both files like the reference does,
offpolicy.py:342-357) and handed to the learner when training is enabled.
"""
import ctypes
import os
from os.path import join as pjoin

import numpy as np
import torch

from tracktolearn_b200 import _lib


def format_widths(widths_str):
    """Reference: algorithms/shared/utils.py:37-38."""
    return np.asarray([int(i) for i in str(widths_str).split('-')])


class MaxEntropyActor(object):
    """Weights of the reference's ``MaxEntropyActor`` (offpolicy.py:61-140) + device forward.

    ``state_dict`` keys: ``layers.{0,2,4,..}.{weight,bias}`` (shared/utils.py:41-51)."""

    def __init__(self, state_dim, action_dim, hidden_dims, device, precision='fp16'):
        if precision not in _lib.PRECISIONS:
            raise ValueError("precision must be one of %s, not %r" % (sorted(_lib.PRECISIONS), precision))
        self.state_dim = int(state_dim)
        self.action_dim = int(action_dim)
        self.hidden_layers = format_widths(hidden_dims)
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.TTLError('the actor forward runs on a CUDA device only (got %s)' % (self.device,))
        if self.device.index is None:       # 'cuda' -> 'cuda:N': tensors report the indexed device
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.precision = precision
        self._lib = _lib.load()
        dims = [self.state_dim] + [int(w) for w in self.hidden_layers] + [2 * self.action_dim]
        self._dims = dims
        g = torch.Generator().manual_seed(torch.initial_seed() % (2 ** 31))
        self._sd = {}
        for li in range(len(dims) - 1):   # nn.Linear default init (kaiming_uniform(a=sqrt(5)))
            bound = 1.0 / np.sqrt(dims[li])
            self._sd['layers.%d.weight' % (2 * li)] = \
                ((torch.rand((dims[li + 1], dims[li]), generator=g) * 2 - 1) * bound).to(self.device)
            self._sd['layers.%d.bias' % (2 * li)] = \
                ((torch.rand((dims[li + 1],), generator=g) * 2 - 1) * bound).to(self.device)
        self._plan = None
        self._plan_rows = 0
        self._workspace = None
        self._plan_layout = None

    # -- checkpoint format ---------------------------------------------------------------
    def state_dict(self):
        return {k: v.detach().clone() for k, v in self._sd.items()}

    def load_state_dict(self, sd):
        missing = [k for k in self._sd if k not in sd]
        unexpected = [k for k in sd if k not in self._sd]
        if missing or unexpected:
            raise RuntimeError('Error(s) in loading state_dict for MaxEntropyActor: missing %s, '
                               'unexpected %s' % (missing, unexpected))
        for k in self._sd:
            if tuple(sd[k].shape) != tuple(self._sd[k].shape):
                raise RuntimeError('size mismatch for %s: %s vs %s' % (k, tuple(sd[k].shape),
                                                                       tuple(self._sd[k].shape)))
            self._sd[k] = sd[k].detach().to(self.device, dtype=torch.float32).contiguous()
        self._drop_plan()

    def parameters(self):
        return list(self._sd.values())

    def share_parameters(self, module_state_dict):
        """Alias the weights of a torch module (its ``state_dict()`` tensors share storage with the
        parameters): optimiser steps then change the tensors this actor packs from, and
        ``refresh_weights`` makes the tensor-core copies current."""
        for k in self._sd:
            t = module_state_dict[k]
            if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError('shared parameter %s must be a contiguous fp32 tensor on %s' % (k, self.device))
            self._sd[k] = t
        self._drop_plan()

    def refresh_weights(self):
        if self._plan is not None:
            _lib.check(self._lib.ttl_actor_plan_refresh(self._plan, _lib.stream_ptr(self.device)),
                       'ttl_actor_plan_refresh')
            self._plan_layout = None

    # -- forward -------------------------------------------------------------------------
    def _drop_plan(self):
        if self._plan is not None:
            self._lib.ttl_actor_plan_destroy(self._plan)
        self._plan = None
        self._plan_rows = 0
        self._workspace = None
        self._plan_layout = None

    def __del__(self):
        try:
            self._drop_plan()
        except Exception:
            pass

    def _weights_struct(self):
        w = _lib.ActorWeights()
        nl = len(self._dims) - 1
        w.n_layers = nl
        for i in range(nl):
            w.in_dim[i] = self._dims[i]
            w.out_dim[i] = self._dims[i + 1]
            w.w[i] = self._sd['layers.%d.weight' % (2 * i)].data_ptr()
            w.b[i] = self._sd['layers.%d.bias' % (2 * i)].data_ptr()
        return w

    def _ensure_plan(self, rows):
        if self._plan is not None and rows <= self._plan_rows:
            return
        self._drop_plan()
        rows = max(int(rows), 128)
        w = self._weights_struct()
        prec = _lib.PRECISIONS[self.precision]
        nbytes = self._lib.ttl_actor_workspace_bytes(ctypes.byref(w), rows, prec)
        if nbytes < 0:
            raise _lib.TTLError('unsupported actor architecture %s' % (self._dims,))
        # GUARD (class attribute / TTL_GUARD=1): 4 KB of 0xA5 on either side of the plan's workspace,
        # verified by check_guards() -- see environments/tracking_env.py
        g = 4096 if self.GUARD else 0
        self._workspace = torch.full((nbytes + 1024 + 2 * g,), 0xA5 if g else 0, dtype=torch.uint8, device=self.device)
        base = (self._workspace.data_ptr() + g + 1023) // 1024 * 1024
        self._ws_span = (base - self._workspace.data_ptr(), int(nbytes))
        if g:
            self._workspace[self._ws_span[0]:self._ws_span[0] + nbytes].zero_()
        plan = ctypes.c_void_p()
        _lib.check(self._lib.ttl_actor_plan_create(ctypes.byref(plan), ctypes.byref(w), rows, prec,
                                                   ctypes.c_void_p(base), nbytes,
                                                   _lib.stream_ptr(self.device)), 'ttl_actor_plan_create')
        self._plan = plan
        self._plan_rows = rows
        self._w_struct = w

    GUARD = os.environ.get('TTL_GUARD', '0') == '1'

    def check_guards(self):
        """Guard bytes around the plan's workspace that a kernel overwrote (0 = clean; needs GUARD)."""
        if self._workspace is None or not self.GUARD:
            return 0
        off, n = self._ws_span
        ws = self._workspace
        return int((ws[:off] != 0xA5).sum().item()) + int((ws[off + n:] != 0xA5).sum().item())

    def forward_device(self, state, probabilistic, n_rows_dev=None, n_rows=None, eps=None,
                       want_logp=True, want_pre=False, out_action=None, state_bf16=None, layout=None):
        """state: CUDA fp32 [rows, >= state_dim] (row stride free).  ``n_rows_dev``: optional
        device int32 tensor with the live row count (no host sync).  ``state_bf16``: the env's
        zero-padded copy of the same rows in this actor's operand type ([rows_alloc,
        round_up(state_dim, 64)], ``env.current_state_bf16()``); with it the packing pass is skipped.  Returns
        (action [rows,3], logp [rows] or None, pre [rows,6] or None)."""
        if state is not None:
            if state.dim() < 2:
                state = state[None, :]
            if state.device != self.device or state.dtype != torch.float32 or state.stride(1) != 1:
                state = state.to(self.device, dtype=torch.float32).contiguous()
        elif state_bf16 is None or n_rows is None:
            raise ValueError('forward_device needs `state`, or `state_bf16` together with `n_rows`')
        rows = int(n_rows if n_rows is not None else state.shape[0])
        A = self.action_dim
        action = out_action if out_action is not None else torch.empty((rows, A), dtype=torch.float32,
                                                                       device=self.device)
        logp = torch.empty((rows,), dtype=torch.float32, device=self.device) if want_logp else None
        pre = torch.empty((rows, 2 * A), dtype=torch.float32, device=self.device) if want_pre else None
        if rows == 0:
            return action, logp, pre
        if probabilistic != 0.0 and eps is None:
            eps = torch.randn((rows, A), dtype=torch.float32, device=self.device)
        self._ensure_plan(rows)
        if self._operand_matches(state_bf16):
            _lib.check(self._lib.ttl_actor_forward_packed(
                self._plan, _lib.ptr(state_bf16), int(state_bf16.stride(0)), int(state_bf16.shape[0]),
                _lib.ptr(n_rows_dev), rows, float(probabilistic), _lib.ptr(eps), _lib.ptr(action),
                _lib.ptr(logp), _lib.ptr(pre), self._set_layout(layout), _lib.stream_ptr(self.device)),
                'ttl_actor_forward_packed')
            self._keep = (state_bf16, eps)
            return action, logp, pre
        if state is None:
            raise _lib.TTLError('the env produced %s operand rows only; a %s actor needs matching operand rows or the '
                                'fp32 state tensor' % (state_bf16.dtype, self.precision))
        ld = state.stride(0) if state.shape[0] > 1 else state.shape[1]
        _lib.check(self._lib.ttl_actor_forward(
            self._plan, _lib.ptr(state), int(ld), _lib.ptr(n_rows_dev), rows, float(probabilistic),
            _lib.ptr(eps), _lib.ptr(action), _lib.ptr(logp), _lib.ptr(pre),
            _lib.stream_ptr(self.device)), 'ttl_actor_forward')
        self._keep = (state, eps)
        return action, logp, pre

    def _set_layout(self, layout):
        """The plan's first-layer column layout for the env's operand rows (``env.bf16_layout``): 1 for the
        channel-padded rows (their weight copy packed once per layout), else 0."""
        if layout is None or layout[0] != 1:
            return 0
        if self._plan_layout != tuple(layout):
            _lib.check(self._lib.ttl_actor_plan_set_layout(
                self._plan, int(layout[1]), int(layout[2]), int(layout[3]),
                _lib.stream_ptr(self.device)), 'ttl_actor_plan_set_layout')
            self._plan_layout = tuple(layout)
        return 1

    def forward_head_partial(self, state_bf16, n_rows, n_rows_dev=None, layout=None, state=None, policy=False):
        """Deterministic policy (prob = 0) for the device loop: runs the tensor-core layers over the
        env's operand rows (or, when their element type is not this actor's, over ``state``: the fp32 rows,
        packed first) and leaves the 6-wide output layer as per-tile partial sums in the plan's scratch.
        Returns (partial_ptr, n_tiles, tiles_per_256, bias_ptr) for ``env.step_device(head=...)``, or None when
        this actor cannot do it (fp32 tier, output layer not fused, no usable rows).
        ``policy=True``: the partials of all six outputs (mu and log_std) for the stochastic policy that
        ``env.step_device(head=..., policy=...)`` samples; the mu partials are the same bits."""
        packed = self._operand_matches(state_bf16)
        if self.precision not in self._OPERAND_DTYPES or (not packed and state is None):
            return None
        rows = int(n_rows)
        self._ensure_plan(rows)
        partial, n_tiles, per256, bias = ctypes.c_void_p(), ctypes.c_int32(), ctypes.c_int32(), ctypes.c_void_p()

        def query():
            return self._lib.ttl_actor_head_partial(self._plan, ctypes.byref(partial), ctypes.byref(n_tiles),
                                                    ctypes.byref(per256), ctypes.byref(bias))
        if query() != 0:          # the output layer is not fused into the last hidden layer
            return None
        probabilistic = 1.0 if policy else 0.0      # with no action buffer: keep the log_std partials too
        if rows > 0 and packed:
            _lib.check(self._lib.ttl_actor_forward_packed(
                self._plan, _lib.ptr(state_bf16), int(state_bf16.stride(0)), int(state_bf16.shape[0]),
                _lib.ptr(n_rows_dev), rows, probabilistic, None, None, None, None, self._set_layout(layout),
                _lib.stream_ptr(self.device)), 'ttl_actor_forward_packed')
            self._keep = (state_bf16, None)
        elif rows > 0:
            ld = state.stride(0) if state.shape[0] > 1 else state.shape[1]
            _lib.check(self._lib.ttl_actor_forward(
                self._plan, _lib.ptr(state), int(ld), _lib.ptr(n_rows_dev), rows, probabilistic, None, None, None,
                None, _lib.stream_ptr(self.device)), 'ttl_actor_forward')
            self._keep = (state, None)
        query()                   # the geometry of the partials depends on the launch just made
        return partial.value, int(n_tiles.value), int(per256.value), bias.value

    _OPERAND_DTYPES = {'bf16': torch.bfloat16, 'fp16': torch.float16, 'tf32': torch.float32}

    def _operand_matches(self, rows):
        """Can ``rows`` (the env's operand rows) feed the first layer as they are?"""
        return (rows is not None and self.precision in self._OPERAND_DTYPES
                and rows.dtype == self._OPERAND_DTYPES[self.precision])

    def overflowed(self, clear=True):
        """fp16 tier: True when a state or activation value had to be saturated to +-65504 since the
        last clearing call (one 4-byte D2H copy + stream sync).  Always False for the other tiers."""
        if self.precision != 'fp16' or self._plan is None:
            return False
        out = ctypes.c_int32(0)
        _lib.check(self._lib.ttl_actor_overflow(self._plan, ctypes.byref(out), int(bool(clear)),
                                                _lib.stream_ptr(self.device)), 'ttl_actor_overflow')
        return bool(out.value)

    def __call__(self, state, probabilistic):
        """Reference: MaxEntropyActor.forward (offpolicy.py:94-140) -> (pi_action, logp_pi)."""
        action, logp, _ = self.forward_device(state, probabilistic)
        return action, logp

    def eval(self):
        return self

    def train(self):
        return self

    def to(self, device):
        return self


class SACActorCritic(object):
    """Reference: algorithms/shared/offpolicy.py:407-482 (+ ActorCritic base :234-372).

    The actor is the device forward above.  The critic (offpolicy.py:183-232, two Q networks over
    concat(state, action)) is not evaluated on the tracking path: it lives either in the learner that
    ``SACAuto.enable_training`` attaches (torch autograd modules, algorithms/sac_train.py) or, before
    that, as the state dict a checkpoint brought.  ``save`` always writes both files and ``load`` always
    reads both, like the reference."""

    def __init__(self, state_dim, action_dim, hidden_dims, device, precision='fp16'):
        self.device = torch.device(device)
        self.actor = MaxEntropyActor(state_dim, action_dim, hidden_dims, self.device, precision)
        self.hidden_dims = hidden_dims
        self.critic_state_dict = None   # q1.* / q2.* tensors of a loaded checkpoint (no learner yet)
        self.learner = None             # set by SACAuto.enable_training

    def attach_learner(self, learner):
        """Training starts: the learner's critic takes over a critic loaded earlier and from now on is
        what ``state_dict`` / ``save`` see."""
        if self.critic_state_dict is not None:
            learner.critic.load_state_dict({k: v.to(self.device) for k, v in self.critic_state_dict.items()})
            learner.target_critic.load_state_dict(learner.critic.state_dict())
        self.learner = learner
        self.critic_state_dict = None

    def _critic_state(self):
        if self.learner is not None:
            return {k: v.detach().clone() for k, v in self.learner.critic.state_dict().items()}
        if self.critic_state_dict is None:
            # never trained, never loaded: the freshly initialised critic the reference's constructor builds
            from tracktolearn_b200.algorithms.sac_train import TorchDoubleCritic
            widths = [int(w) for w in format_widths(self.hidden_dims)]
            self.critic_state_dict = TorchDoubleCritic(self.actor.state_dim, self.actor.action_dim, widths).state_dict()
        return self.critic_state_dict

    def act(self, state, probabilistic=1.0):
        return self.actor(state, probabilistic)

    def select_action(self, state, probabilistic=1.0):
        if len(state.shape) < 2:
            state = state[None, :]
        action, _ = self.act(state, probabilistic)
        return action

    def parameters(self):
        return self.actor.parameters()

    def load_state_dict(self, state_dict):
        """Reference: offpolicy.py:300-310."""
        actor_state_dict, critic_state_dict = state_dict
        if self.learner is not None:
            # the inference actor aliases the learner's parameters: load through the module
            self.learner.actor.load_state_dict(actor_state_dict)
            self.learner.target_actor.load_state_dict(actor_state_dict)
            self.actor.refresh_weights()
            if critic_state_dict is not None:
                self.learner.critic.load_state_dict(critic_state_dict)
                self.learner.target_critic.load_state_dict(critic_state_dict)
            return
        self.actor.load_state_dict(actor_state_dict)
        self.critic_state_dict = critic_state_dict

    def state_dict(self):
        """Reference: offpolicy.py:312-315 -> (actor state dict, critic state dict)."""
        return self.actor.state_dict(), self._critic_state()

    def save(self, path, filename):
        """Reference: offpolicy.py:327-340: <filename>_critic.pth and <filename>_actor.pth, CPU tensors
        under the reference's keys (q1.* / q2.*, layers.*)."""
        torch.save({k: v.detach().cpu() for k, v in self._critic_state().items()},
                   pjoin(path, filename + "_critic.pth"))
        torch.save({k: v.detach().cpu() for k, v in self.actor.state_dict().items()},
                   pjoin(path, filename + "_actor.pth"))

    def load(self, path, filename):
        """Reference: offpolicy.py:342-357 (both files are read, a missing one raises)."""
        critic = torch.load(pjoin(path, filename + '_critic.pth'), map_location='cpu')
        actor = torch.load(pjoin(path, filename + '_actor.pth'), map_location=self.device)
        self.load_state_dict((actor, critic))

    def eval(self):
        self.actor.eval()

    def train(self):
        self.actor.train()
