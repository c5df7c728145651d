"""Plain restatement of the connectivity matrix (DESIGN.md section 2, "Connectivity matrix") that the kernel tests
compare with: ``end_label`` labels one endpoint with Python floats (IEEE fp64, rounded to nearest, no
contraction), in the operation order of the contract; ``connectome_fast`` is the same with numpy array
operations for millions of points."""
import math

import numpy as np


def _label(labels, K, v):
    lab = int(labels[v])
    return lab if 0 < lab < K else 0


def end_label(p, labels, r, K=None):
    """Label of the endpoint p (a float32 triple) in the int volume ``labels`` [X, Y, Z] at radius r voxels."""
    dims = labels.shape
    K = int(labels.max()) + 1 if K is None else K
    p = [float(np.float32(x)) for x in p]
    if all(math.isfinite(x) for x in p):
        own = [math.floor(x + 0.5) for x in p]
        if all(0 <= c < d for c, d in zip(own, dims)):
            lab = _label(labels, K, tuple(own))
            if lab > 0:
                return lab
    else:
        return 0
    r = float(r)
    r2 = r * r
    lo = [max(math.ceil(x - r), 0) for x in p]
    hi = [min(math.floor(x + r), d - 1) for x, d in zip(p, dims)]
    best = None
    for cx in range(lo[0], hi[0] + 1):
        for cy in range(lo[1], hi[1] + 1):
            for cz in range(lo[2], hi[2] + 1):
                dx, dy, dz = float(cx) - p[0], float(cy) - p[1], float(cz) - p[2]
                d2 = ((dx * dx) + (dy * dy)) + (dz * dz)
                if d2 > r2:
                    continue
                lab = _label(labels, K, (cx, cy, cz))
                key = (d2, (cx * dims[1] + cy) * dims[2] + cz)
                if lab > 0 and (best is None or key < best[0]):
                    best = (key, lab)
    return 0 if best is None else best[1]


def connectome(data, offsets, labels, r=0.0, K=None):
    """-> (matrix int32 [K, K], pairs int32 [n, 2]) by the per-endpoint loop."""
    K = int(labels.max()) + 1 if K is None else K
    n = len(offsets) - 1
    matrix = np.zeros((K, K), dtype=np.int32)
    pairs = np.zeros((n, 2), dtype=np.int32)
    data = np.asarray(data, dtype=np.float32)
    for i in range(n):
        s = data[offsets[i]:offsets[i + 1]]
        if not len(s):
            continue
        a, b = end_label(s[0], labels, r, K), end_label(s[-1], labels, r, K)
        pairs[i] = a, b
        matrix[a, b] += 1
        if a != b:
            matrix[b, a] += 1
    return matrix, pairs


def end_labels_fast(pts, labels, r, K=None):
    """``end_label`` of every row of pts [m, 3] float32, vectorised over the points: own voxel first, then
    one pass per integer offset of the search box around floor(p)."""
    dims = np.asarray(labels.shape, dtype=np.int64)
    K = int(labels.max()) + 1 if K is None else K
    flat = np.asarray(labels).reshape(-1).astype(np.int64)
    flat = np.where((flat > 0) & (flat < K), flat, 0)
    p = np.asarray(pts, dtype=np.float32).astype(np.float64)
    out = np.zeros(len(p), dtype=np.int32)
    finite = np.all(np.isfinite(p), axis=1)
    with np.errstate(invalid='ignore'):
        own = np.floor(p + 0.5)
        ing = finite & np.all((own >= 0) & (own < dims), axis=1)
    oi = own[ing].astype(np.int64)
    out[ing] = flat[(oi[:, 0] * dims[1] + oi[:, 1]) * dims[2] + oi[:, 2]]
    todo = np.nonzero(finite & (out == 0))[0]
    r = float(r)
    r2 = r * r
    q = p[todo]
    # box bounds, clamped to the grid; clipped first so that far points convert to int64 safely
    lo = np.maximum(np.clip(np.ceil(q - r), -1, dims), 0).astype(np.int64)
    hi = np.minimum(np.clip(np.floor(q + r), -1, dims), dims - 1).astype(np.int64)
    base = np.clip(np.floor(q), -2, dims + 1).astype(np.int64)
    best_d2 = np.full(len(todo), np.inf)
    best_v = np.full(len(todo), np.iinfo(np.int64).max)
    best_l = np.zeros(len(todo), dtype=np.int64)
    R = int(math.ceil(r)) + 1
    rng = range(-R, R + 1)
    for ox in rng:
        for oy in rng:
            for oz in rng:
                c = base + np.array([ox, oy, oz], dtype=np.int64)
                ok = np.all((c >= lo) & (c <= hi), axis=1)
                if not ok.any():
                    continue
                idx = np.nonzero(ok)[0]
                cc = c[idx]
                d = cc.astype(np.float64) - q[idx]
                d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
                v = (cc[:, 0] * dims[1] + cc[:, 1]) * dims[2] + cc[:, 2]
                lab = flat[v]
                upd = (d2 <= r2) & (lab > 0) & ((d2 < best_d2[idx]) | ((d2 == best_d2[idx]) & (v < best_v[idx])))
                j = idx[upd]
                best_d2[j], best_v[j], best_l[j] = d2[upd], v[upd], lab[upd]
    out[todo] = best_l
    return out


def connectome_fast(data, offsets, labels, r=0.0, K=None):
    """``connectome`` with numpy array operations (checked against the loop in test_connectome_cpu.py)."""
    K = int(labels.max()) + 1 if K is None else K
    offsets = np.asarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    nonempty = np.diff(offsets) > 0
    data = np.asarray(data, dtype=np.float32).reshape(-1, 3)
    ends = np.concatenate((data[offsets[:-1][nonempty]], data[offsets[1:][nonempty] - 1]))
    lab = end_labels_fast(ends, labels, r, K)
    m = int(nonempty.sum())
    a, b = lab[:m].astype(np.int64), lab[m:].astype(np.int64)
    pairs = np.zeros((n, 2), dtype=np.int32)
    pairs[nonempty, 0], pairs[nonempty, 1] = a, b
    cells = np.concatenate((a * K + b, (b * K + a)[a != b]))
    matrix = np.bincount(cells, minlength=K * K).astype(np.int32).reshape(K, K)
    return matrix, pairs
