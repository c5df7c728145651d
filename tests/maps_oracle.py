"""Plain restatement of the streamline maps (DESIGN.md section 2, "Streamline maps") that the kernel tests
compare with: per streamline, a Python set of voxel tuples."""
import math

import numpy as np


def voxel_of(p, dims):
    """floor(p_k + 0.5) per axis in float64 (exact for a float32 p_k); None outside 0 <= c_k < dim_k, NaN and
    +-inf included."""
    c = []
    for x, d in zip(p, dims):
        x = float(x)
        if not math.isfinite(x):
            return None
        k = math.floor(x + 0.5)
        if not 0 <= k < d:
            return None
        c.append(k)
    return tuple(c)


def tract_maps(data, offsets, dims):
    """-> (density, endpoints, skipped): int32 maps [X, Y, Z] and the number of points outside the grid."""
    dims = tuple(int(d) for d in dims)
    density = np.zeros(dims, dtype=np.int32)
    endpoints = np.zeros(dims, dtype=np.int32)
    skipped = 0
    data = np.asarray(data, dtype=np.float32)
    for i in range(len(offsets) - 1):
        s = data[offsets[i]:offsets[i + 1]]
        voxels = set()
        for p in s:
            v = voxel_of(p, dims)
            if v is None:
                skipped += 1
            else:
                voxels.add(v)
        for v in voxels:
            density[v] += 1
        if len(s):
            for p in (s[0], s[-1]):
                v = voxel_of(p, dims)
                if v is not None:
                    endpoints[v] += 1
    return density, endpoints, skipped


def tract_maps_fast(data, offsets, dims):
    """``tract_maps`` with numpy array operations, for inputs of millions of points (checked against the loop
    in test_tract_maps_cpu.py)."""
    dims = tuple(int(d) for d in dims)
    offsets = np.asarray(offsets, dtype=np.int64)
    c = np.floor(np.asarray(data, dtype=np.float32).astype(np.float64) + 0.5)
    with np.errstate(invalid='ignore'):
        ok = np.all((c >= 0) & (c < np.asarray(dims, dtype=np.float64)), axis=1)
    lin = np.full(len(c), -1, dtype=np.int64)
    ci = c[ok].astype(np.int64)
    lin[ok] = (ci[:, 0] * dims[1] + ci[:, 1]) * dims[2] + ci[:, 2]
    n_vox = int(np.prod(dims))
    row = np.repeat(np.arange(len(offsets) - 1, dtype=np.int64), np.diff(offsets))
    pairs = np.unique(row[ok] * n_vox + lin[ok])
    density = np.bincount(pairs % n_vox, minlength=n_vox).astype(np.int32).reshape(dims)
    nonempty = np.diff(offsets) > 0
    ends = np.concatenate((lin[offsets[:-1][nonempty]], lin[offsets[1:][nonempty] - 1]))
    endpoints = np.bincount(ends[ends >= 0], minlength=n_vox).astype(np.int32).reshape(dims)
    return density, endpoints, int((~ok).sum())
