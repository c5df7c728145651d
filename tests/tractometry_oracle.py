"""Plain restatement of tractometry (DESIGN.md section 2, "Tractometry") that the kernel tests compare with: the
sampled points, the fp64 trilinear value of a point, the per-streamline mean in the kernel's summation order, and
the int64 fixed-point edge sums."""
import math

import numpy as np


def sampled(data, dims):
    """The points the maps count (maps_oracle.voxel_of is not None): floor(p + 0.5) in the grid, in float64."""
    c = np.floor(np.asarray(data, dtype=np.float32).reshape(-1, 3).astype(np.float64) + 0.5)
    with np.errstate(invalid='ignore'):
        return np.all((c >= 0) & (c < np.asarray(dims, dtype=np.float64)), axis=1)


def trilinear(pts, vol):
    """fp64 trilinear values [m, C] of sampled points pts [m, 3] (float32) in vol [X, Y, Z, C]: per axis
    c = (double)p, i = floor(c), d = c - i, corners clamp(i, 0, n-1) and clamp(i+1, 0, n-1), weights 1-d and d;
    the sum over the corners, x then y then z lower before upper, of ((wx*wy)*wz)*v (numpy rounds every
    operation, as the kernel does without contraction)."""
    vol = np.asarray(vol, dtype=np.float32)
    if vol.ndim == 3:
        vol = vol[..., None]
    p = np.asarray(pts, dtype=np.float32).reshape(-1, 3).astype(np.float64)
    idx, w = [], []
    for k in range(3):
        n = vol.shape[k]
        f = np.floor(p[:, k])
        d = p[:, k] - f
        i = f.astype(np.int64)
        idx.append((np.clip(i, 0, n - 1), np.clip(i + 1, 0, n - 1)))
        w.append((1.0 - d, d))
    out = np.zeros((len(p), vol.shape[3]), dtype=np.float64)
    for a in range(2):
        for b in range(2):
            wxy = w[0][a] * w[1][b]
            for e in range(2):
                wt = wxy * w[2][e]
                out = out + wt[:, None] * vol[idx[0][a], idx[1][b], idx[2][e]].astype(np.float64)
    return out


def _tree(acc):
    """The kernel's xor-shuffle tree over the last-but-one axis (32 lanes): acc += acc[lane ^ off]."""
    lanes = np.arange(32)
    for off in (16, 8, 4, 2, 1):
        acc = acc + acc[:, lanes ^ off]
    return acc[:, 0]


def sample_means(data, offsets, vol, chunk=100000):
    """-> (means float32 [n, C], skipped): every streamline's fp64 sum of the trilinear values of its sampled
    points -- lane l (of 32) summing points l, l+32, ... in order, then the xor tree -- divided by their number
    and rounded to float32; NaN with no sampled point.  skipped = the points not sampled."""
    vol = np.asarray(vol, dtype=np.float32)
    if vol.ndim == 3:
        vol = vol[..., None]
    C = vol.shape[3]
    data = np.asarray(data, dtype=np.float32).reshape(-1, 3)
    offsets = np.asarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    ok = sampled(data, vol.shape[:3])
    means = np.empty((n, C), dtype=np.float32)
    for s0 in range(0, n, chunk):
        s1 = min(s0 + chunk, n)
        lo, hi = offsets[s0], offsets[s1]
        row = np.repeat(np.arange(s1 - s0), np.diff(offsets[s0:s1 + 1]))
        j = np.arange(lo, hi) - offsets[s0:s1][row]
        m = ok[lo:hi]
        row, j = row[m], j[m]
        vals = trilinear(data[lo:hi][m], vol)
        count = np.bincount(row, minlength=s1 - s0)
        acc = np.zeros((s1 - s0, 32, C), dtype=np.float64)
        rnd = j // 32
        order = np.argsort(rnd, kind='stable')
        bounds = np.searchsorted(rnd[order], np.arange(int(rnd.max()) + 2 if len(rnd) else 1))
        for r in range(len(bounds) - 1):          # one round of every lane at a time: sequential per lane
            sel = order[bounds[r]:bounds[r + 1]]
            acc[row[sel], j[sel] % 32] += vals[sel]
        total = _tree(acc)
        with np.errstate(invalid='ignore', divide='ignore'):
            mean = (total / count[:, None]).astype(np.float32)
        mean[count == 0] = np.nan
        means[s0:s1] = mean
    return means, int((~ok).sum())


def metric_shift(bound):
    """S = clamp(31 - e, 0, 62) with bound < 2^e."""
    return min(max(31 - math.frexp(float(bound))[1], 0), 62)


def edge_sums(pairs, values, shifts, K):
    """int64 sums [C, K, K] and int32 counts [C, K, K]: round(v * 2^S) (round half to even, as __double2ll_rn)
    at [a, b] and, when a != b, at [b, a], for every finite v; labels outside [0, K) read as 0."""
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    values = np.asarray(values, dtype=np.float32).reshape(len(pairs), -1)
    C = values.shape[1]
    a, b = (np.where((pairs[:, k] > 0) & (pairs[:, k] < K), pairs[:, k], 0) for k in range(2))
    sums = np.zeros((C, K, K), dtype=np.int64)
    counts = np.zeros((C, K, K), dtype=np.int32)
    for c in range(C):
        v = values[:, c].astype(np.float64)
        f = np.isfinite(v)
        q = np.rint(np.ldexp(v[f], int(shifts[c]))).astype(np.int64)
        af, bf = a[f], b[f]
        for x, y, qq in ((af, bf, q), (bf[af != bf], af[af != bf], q[af != bf])):
            np.add.at(sums[c], (x, y), qq)
            np.add.at(counts[c], (x, y), 1)
    return sums, counts
