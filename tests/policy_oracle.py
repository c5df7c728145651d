"""numpy restatement of the stochastic policy sampled on the device (ttl_policy in include/ttl_b200.h) -- test
infrastructure, the reference for tests/test_policy_*.py.

eps_c is the ttl_noise normal at counter words 3..5 (the tracking noise uses 0..2), rounded to float32; the action is
the actor head's arithmetic (MaxEntropyActor.forward) with that eps in place of torch.randn."""
import numpy as np

from tests.noise_oracle import philox4x32_10, philox_uniforms


def policy_normals(seed, g, L):
    """fp64 z[k, c] at counter (lo32(g[k]), hi32(g[k]), L[k], 3 + c), key = seed: before the fp32 rounding."""
    g = np.asarray(g, dtype=np.int64).astype(np.uint64)
    L = np.broadcast_to(np.asarray(L, dtype=np.int64), g.shape).astype(np.uint64)
    n = g.shape[0]
    ctr = np.empty((n, 3, 4), dtype=np.uint64)
    ctr[..., 0] = (g & np.uint64(0xFFFFFFFF))[:, None]
    ctr[..., 1] = (g >> np.uint64(32))[:, None]
    ctr[..., 2] = L[:, None]
    ctr[..., 3] = 3 + np.arange(3, dtype=np.uint64)[None, :]
    seed = int(seed)
    key = np.asarray([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint64)
    u1, u2 = philox_uniforms(philox4x32_10(ctr, key))
    return np.sqrt(-2 * np.log(u1)) * np.cos(2 * np.pi * u2)


def policy_eps(seed, g, L):
    """eps [n, 3] float32 of streamlines with global seed index g [n] and point count L [n] (before the step)."""
    return policy_normals(seed, g, L).astype(np.float32)


def policy_actions(pre, eps, prob):
    """a = tanh(mu + exp(clamp(log_std, -20, 2)) * prob * eps) in float32 from the head's raw output pre [n, 6]
    (bias included) and eps [n, 3]."""
    pre = np.asarray(pre, dtype=np.float32)
    mu, ls = pre[:, :3], pre[:, 3:6]
    std = np.exp(np.clip(ls, np.float32(-20), np.float32(2))) * np.float32(prob)
    return np.tanh(std * np.asarray(eps, dtype=np.float32) + mu)
