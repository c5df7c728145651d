"""ctypes binding of libttl_b200.so (C ABI declared in include/ttl_b200.h).

There is no fallback: if the library is missing or a call fails, we raise.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'lib', 'libttl_b200.so')

c_i32, c_i64, c_f32, c_f64, c_vp = (ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_double,
                                    ctypes.c_void_p)
MAX_LAYERS = 8
PRECISION_BF16, PRECISION_FP32, PRECISION_FP16, PRECISION_TF32 = 0, 1, 2, 3
PRECISIONS = {'bf16': PRECISION_BF16, 'fp32': PRECISION_FP32, 'fp16': PRECISION_FP16, 'tf32': PRECISION_TF32}
OPERAND_BF16, OPERAND_FP16, OPERAND_TF32 = 0, 1, 2
OPERAND_OF_PRECISION = {'bf16': OPERAND_BF16, 'fp16': OPERAND_FP16, 'tf32': OPERAND_TF32}
ABI_VERSION = 5


class Volume(ctypes.Structure):
    _fields_ = [('sh', c_vp), ('X', c_i32), ('Y', c_i32), ('Z', c_i32), ('C', c_i32), ('CP', c_i32),
                ('mask_coef', c_vp), ('MX', c_i32), ('MY', c_i32), ('MZ', c_i32),
                ('peaks', c_vp), ('PX', c_i32), ('PY', c_i32), ('PZ', c_i32)]


class Params(ctypes.Structure):
    _fields_ = [('step_vox', c_f64), ('mask_threshold', c_f64), ('alignment_weighting', c_f64),
                ('theta_rad', c_f32), ('max_nb_steps', c_i32), ('n_dirs', c_i32), ('dir_f64', c_i32),
                ('compute_reward', c_i32), ('state_stopped', c_i32), ('refill', c_i32)]


class Batch(ctypes.Structure):
    _fields_ = [('n', c_i32), ('n_slots', c_i32), ('capacity', c_i32), ('max_pts', c_i32), ('ld_state', c_i32),
                ('state_size', c_i32), ('points', c_vp), ('flags', c_vp), ('lengths', c_vp),
                ('npts', c_vp), ('dones', c_vp), ('alive', c_vp * 2), ('ctrl', c_vp), ('stop', c_vp), ('dest', c_vp),
                ('step_flags', c_vp), ('reward', c_vp), ('state', c_vp * 2),
                ('state_bf16', c_vp * 2), ('ld_bf16', c_i32), ('max_groups', c_i32), ('grp_stops', c_vp),
                ('sg_stops', c_vp), ('bf16_layout', c_i32), ('rank_rec', c_vp * 2), ('step_tip', c_vp),
                ('operand_fmt', c_i32), ('order', c_vp)]


class Noise(ctypes.Structure):
    """ttl_noise: N(0, sigma) tracking noise drawn inside the step kernel (include/ttl_b200.h)."""
    _fields_ = [('sigma', c_f64), ('seed', ctypes.c_uint64), ('row_base', c_i64)]


class Policy(ctypes.Structure):
    """ttl_policy: the stochastic policy sampled with counter-based draws (include/ttl_b200.h)."""
    _fields_ = [('seed', ctypes.c_uint64), ('row_base', c_i64), ('prob', c_f32), ('pad', c_i32)]


class StepAction(ctypes.Structure):
    """ttl_step_action: where the actions of an env step come from -- an action buffer or the actor's fused
    head partials (include/ttl_b200.h)."""
    _fields_ = [('actions', c_vp), ('head_partial', c_vp), ('head_bias', c_vp), ('lda', c_i32), ('n_tiles', c_i32),
                ('tiles_per_256', c_i32), ('pad', c_i32)]


class ActorWeights(ctypes.Structure):
    _fields_ = [('n_layers', c_i32), ('in_dim', c_i32 * MAX_LAYERS), ('out_dim', c_i32 * MAX_LAYERS),
                ('w', c_vp * MAX_LAYERS), ('b', c_vp * MAX_LAYERS)]


class OracleWeights(ctypes.Structure):
    _fields_ = ([('n_layers', c_i32), ('n_head', c_i32), ('d_model', c_i32), ('d_ff', c_i32),
                 ('n_tokens', c_i32), ('cls_token', c_vp), ('emb_w', c_vp), ('emb_b', c_vp), ('pe', c_vp)]
                + [(name, c_vp * 8) for name in ('in_proj_w', 'in_proj_b', 'out_proj_w', 'out_proj_b',
                                                 'lin1_w', 'lin1_b', 'lin2_w', 'lin2_b')]
                + [('norm1_w', c_vp * 8), ('norm1_b', c_vp * 8), ('norm2_w', c_vp * 8), ('norm2_b', c_vp * 8),
                   ('head_w', c_vp), ('head_b', c_vp)])


P = ctypes.POINTER
SIGNATURES = {
    'ttl_abi_version': (c_i32, []),
    'ttl_launch_count': (c_i64, []),
    'ttl_prof_enable': (None, [c_i32]),
    'ttl_pdl_enable': (None, [c_i32]),
    'ttl_prof_report': (c_i32, [ctypes.c_char_p, c_i32]),
    'ttl_pad_channels': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i32, c_vp]),
    'ttl_peaks_from_sh': (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_i32, c_f64, c_f64, c_f64,
                                  c_i32, c_vp, c_vp]),
    'ttl_env_reset': (c_i32, [P(Volume), P(Params), P(Batch), c_vp, c_vp]),
    'ttl_env_step': (c_i32, [P(Volume), P(Params), P(Batch), c_i32, P(StepAction), c_vp, P(Noise), P(Policy), c_i32,
                             c_i32, c_vp]),
    'ttl_env_step_finish': (c_i32, [P(Volume), P(Params), P(Batch), c_i32, c_vp, c_i32, c_i32, c_i32, c_f32, c_i32, c_vp]),
    'ttl_noise_normals': (c_i32, [P(Noise), c_vp, c_vp, c_i32, c_vp, c_vp]),
    'ttl_policy_eps': (c_i32, [P(Policy), P(Batch), c_i32, c_i32, c_vp, c_i32, c_vp]),
    'ttl_oracle_features_rows': (c_i32, [P(Batch), c_i32, c_i32, c_vp, c_vp]),
    'ttl_env_gather_step_state': (c_i32, [P(Batch), c_i32, c_i32, c_vp, c_i32, c_vp]),
    'ttl_format_state': (c_i32, [P(Volume), P(Params), c_vp, c_i32, c_i32, c_vp, c_i32, c_vp]),
    'ttl_stopping_flags': (c_i32, [P(Volume), P(Params), c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'ttl_streamline_offsets': (c_i32, [P(Batch), c_vp, c_vp]),
    'ttl_streamline_lengths': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp]),
    'ttl_compress_mask': (c_i32, [c_vp, c_vp, c_i32, c_f64, c_f64, c_vp, c_vp, c_vp]),
    'ttl_select_workspace_bytes': (c_i64, [c_i32]),
    'ttl_select_streamlines': (c_i32, [c_vp, c_i32, c_vp, c_vp, c_f32, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    'ttl_gather_streamlines': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'ttl_pack_streamlines': (c_i32, [P(Batch), c_vp, c_vp, c_vp]),
    'ttl_actor_workspace_bytes': (c_i64, [P(ActorWeights), c_i32, c_i32]),
    'ttl_actor_plan_create': (c_i32, [P(c_vp), P(ActorWeights), c_i32, c_i32, c_vp, c_i64, c_vp]),
    'ttl_actor_plan_destroy': (None, [c_vp]),
    'ttl_actor_precision': (c_i32, [c_vp]),
    'ttl_actor_options': (None, [c_i32]),
    'ttl_actor_plan_refresh': (c_i32, [c_vp, c_vp]),
    'ttl_actor_forward': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'ttl_actor_forward_packed': (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_i32, c_f32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp]),
    'ttl_actor_head_partial': (c_i32, [c_vp, P(c_vp), P(c_i32), P(c_i32), P(c_vp)]),
    'ttl_actor_overflow': (c_i32, [c_vp, P(c_i32), c_i32, c_vp]),
    'ttl_actor_plan_set_layout': (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp]),
    'ttl_gemm_tc': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp]),
    'ttl_gemm_bf16': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    'ttl_oracle_features': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp]),
    'ttl_oracle_forward': (c_i32, [P(OracleWeights), c_vp, c_i32, c_vp, c_vp]),
    'ttl_oracle_workspace_bytes': (c_i64, [P(OracleWeights)]),
    'ttl_oracle_plan_create': (c_i32, [P(c_vp), P(OracleWeights), c_vp, c_i64, c_vp]),
    'ttl_oracle_plan_destroy': (None, [c_vp]),
    'ttl_oracle_forward_tc': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp]),
}

_lib = None


class TTLError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TTLError('%s not found: build it with `python -m tracktolearn_b200.build` '
                       '(there is no CPU fallback)' % LIB_PATH)
    # a library built from other sources than the ones next to it must not be used silently
    from tracktolearn_b200 import build as _build
    stamp = os.path.join(os.path.dirname(LIB_PATH), 'libttl_b200.sha256')
    if os.path.isdir(_build.CSRC) and os.environ.get('TTL_SKIP_DIGEST', '0') != '1':
        have = open(stamp).read().strip() if os.path.exists(stamp) else None
        if have != _build._digest():
            raise TTLError('%s is stale (its stamp does not match csrc/ + include/ttl_b200.h): rebuild it with '
                           '`python -m tracktolearn_b200.build`' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ttl_abi_version() != ABI_VERSION:
        raise TTLError('%s has ABI version %d, this package binds version %d: rebuild it'
                       % (LIB_PATH, lib.ttl_abi_version(), ABI_VERSION))
    if os.environ.get('TTL_PDL', '1') == '0':      # A/B measurements: plain stream-ordered launches
        lib.ttl_pdl_enable(0)
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        raise TTLError('%s failed with code %d' % (what, rc))


def prof_report():
    """Per-kernel {name: (launches, total_ms)} since the last report (see ttl_prof_enable)."""
    import json
    lib = load()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.ttl_prof_report(buf, len(buf))
    return {k: (int(v[0]), float(v[1])) for k, v in json.loads(buf.value.decode()).items()}


def ptr(t):
    """Device (or host) pointer of a torch tensor / None."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
