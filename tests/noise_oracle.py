"""numpy restatement of the device-drawn tracking noise (ttl_noise in include/ttl_b200.h, csrc/ttl_rng.cuh) and
an OracleEnv that draws its noise the same way -- test infrastructure, the reference for tests/test_noise_*.py.

The noise has no counterpart in the reference (which draws ``rng.normal`` on the host), so it lives beside the
tests rather than in the reference restatement (oracle/ttl_oracle.py)."""
import numpy as np

from oracle import ttl_oracle as O

PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11; Random123 constants), vectorised: ctr [..., 4] and key [..., 2]
    uint32 (broadcast) -> [..., 4] uint32."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    m = np.uint64(0xFFFFFFFF)
    x0, x1, x2, x3 = (ctr[..., i] & m for i in range(4))
    k0, k1 = key[..., 0] & m, key[..., 1] & m
    for _ in range(10):
        p0 = np.uint64(PHILOX_M0) * x0          # < 2^64: exact in uint64
        p1 = np.uint64(PHILOX_M1) * x2
        x0, x1, x2, x3 = ((p1 >> np.uint64(32)) ^ x1 ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ x3 ^ k1, p0 & m)
        k0 = (k0 + np.uint64(PHILOX_W0)) & m
        k1 = (k1 + np.uint64(PHILOX_W1)) & m
    return np.stack([x0, x1, x2, x3], -1).astype(np.uint32)


def philox_uniforms(w):
    """The two open-interval uniforms of one Philox output [..., 4]: u = ((hi:lo >> 12) + 0.5) * 2^-52,
    exact in float64 and strictly inside (0, 1)."""
    w = np.asarray(w, dtype=np.uint64)
    u1 = ((((w[..., 1] << np.uint64(32)) | w[..., 0]) >> np.uint64(12)).astype(np.float64) + 0.5) * 2.0 ** -52
    u2 = ((((w[..., 3] << np.uint64(32)) | w[..., 2]) >> np.uint64(12)).astype(np.float64) + 0.5) * 2.0 ** -52
    return u1, u2


def philox_normals(seed, g, L):
    """z[k, c] = standard normal of (seed, global seed index g[k], point count L[k], component c): the draw
    the step kernels add, times sigma, to the action of that streamline at that step."""
    g = np.asarray(g, dtype=np.int64).astype(np.uint64)
    L = np.broadcast_to(np.asarray(L, dtype=np.int64), g.shape).astype(np.uint64)
    n = g.shape[0]
    ctr = np.empty((n, 3, 4), dtype=np.uint64)
    ctr[..., 0] = (g & np.uint64(0xFFFFFFFF))[:, None]
    ctr[..., 1] = (g >> np.uint64(32))[:, None]
    ctr[..., 2] = L[:, None]
    ctr[..., 3] = np.arange(3, dtype=np.uint64)[None, :]
    seed = int(seed)
    key = np.asarray([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint64)
    u1, u2 = philox_uniforms(philox4x32_10(ctr, key))
    return np.sqrt(-2 * np.log(u1)) * np.cos(2 * np.pi * u2)


class PhiloxNoiseOracleEnv(O.OracleEnv):
    """``OracleEnv(noisy=True)`` whose noise is drawn as NoisyTrackingEnvironment draws it with
    ``noise_rng='device'``: ``noise * philox_normals(noise_seed, row_base + row, length)`` added in float64 to
    the float32 actions, with row_base = ``seed_offset + start`` after ``reset(start, end)`` and 0 after
    ``nreset``."""

    def __init__(self, *args, noise_seed, **kw):
        kw['noisy'] = True
        super().__init__(*args, **kw)
        self.noise_seed = noise_seed
        self.seed_offset = 0
        self.row_base = 0

    def reset(self, start, end):
        self.row_base = self.seed_offset + start
        return super().reset(start, end)

    def nreset(self, n_seeds):
        self.row_base = 0
        return super().nreset(n_seeds)

    def step(self, actions):
        z = philox_normals(self.noise_seed, self.row_base + self.continue_idx, self.length)
        noisy = np.asarray(actions, dtype=np.float32).astype(np.float64) + self.noise * z
        # the parent then adds rng.normal(0, 0): exact zeros, the float64 directions are unchanged
        sigma, self.noise = self.noise, 0.0
        try:
            return super().step(noisy)
        finally:
            self.noise = sigma
