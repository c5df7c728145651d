"""Per-streamline post-processing of a packed tractogram on the device (reference:
tracking/tracker.py:118-125): dipy ``length`` for the min/max length filter and dipy
``compress_streamlines`` for ``--compress``.  Packed layout: ``data`` [total, 3] float32 and
``offsets`` [n + 1] int64 (streamline i = data[offsets[i]:offsets[i+1]])."""
import math

import numpy as np
import torch

from tracktolearn_b200 import _lib


def _dev(device):
    device = torch.device(device if device is not None else 'cuda:0')
    if device.type != 'cuda':
        raise _lib.TTLError('tractogram post-processing runs on a CUDA device only (no CPU fallback)')
    return device


def _to_device(data, offsets, device):
    d = data if isinstance(data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(data, dtype=np.float32))
    o = offsets if isinstance(offsets, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64))
    return (d.to(device, dtype=torch.float32, non_blocking=True).contiguous(),
            o.to(device, dtype=torch.int64, non_blocking=True).contiguous())


def lengths_packed(data, offsets, device=None):
    """dipy ``length`` of every streamline -> float64 CUDA tensor [n]."""
    device = _dev(device if device is not None else (data.device if isinstance(data, torch.Tensor) else None))
    lib = _lib.load()
    d, o = _to_device(data, offsets, device)
    n = int(o.shape[0]) - 1
    out = torch.zeros((max(n, 0),), dtype=torch.float64, device=device)
    if n > 0:
        with torch.cuda.device(device):
            _lib.check(lib.ttl_streamline_lengths(_lib.ptr(d), _lib.ptr(o), n, _lib.ptr(out),
                                                  _lib.stream_ptr(device)), 'ttl_streamline_lengths')
    return out


def compress_packed(data, offsets, tol_error=0.01, max_segment_length=10.0, device=None):
    """dipy ``compress_streamlines(streamlines, tol_error, max_segment_length)`` on a packed
    tractogram.  Returns (data', offsets') as CUDA tensors: the kept points, in order."""
    device = _dev(device if device is not None else (data.device if isinstance(data, torch.Tensor) else None))
    lib = _lib.load()
    d, o = _to_device(data, offsets, device)
    n = int(o.shape[0]) - 1
    if n <= 0:
        return d[:0], torch.zeros((1,), dtype=torch.int64, device=device)
    keep = torch.zeros((d.shape[0],), dtype=torch.uint8, device=device)
    count = torch.zeros((n,), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.ttl_compress_mask(_lib.ptr(d), _lib.ptr(o), n, float(tol_error), float(max_segment_length),
                                         _lib.ptr(keep), _lib.ptr(count), _lib.stream_ptr(device)),
                   'ttl_compress_mask')
    new_offsets = torch.zeros((n + 1,), dtype=torch.int64, device=device)
    torch.cumsum(count, 0, out=new_offsets[1:])
    return d[keep.bool()], new_offsets


def select_packed(data, offsets, keep=None, scores=None, threshold=0.0):
    """Ordered selection of packed streamlines on their device (``ttl_select_streamlines`` +
    ``ttl_gather_streamlines``): streamline i is kept when ``keep[i]`` (uint8 / bool, None = all) and
    ``scores[i] >= threshold`` (float32, compared in float32; None = no score test; NaN is never kept).
    Returns (data', offsets', index) as CUDA tensors: the kept points bit for bit, their offsets and the
    int64 source row of every kept streamline.  One device-to-host copy of the two sizes."""
    device = _dev(data.device)
    lib = _lib.load()
    data, offsets = _to_device(data, offsets, device)
    n = int(offsets.shape[0]) - 1
    sp = _lib.stream_ptr(device)
    if keep is not None:
        keep = keep.to(device, dtype=torch.uint8).contiguous()
    if scores is not None:
        scores = scores.to(device, dtype=torch.float32).contiguous()
    nbytes = int(lib.ttl_select_workspace_bytes(max(n, 0)))
    work = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=device)
    out_off = torch.empty((max(n, 0) + 1,), dtype=torch.int64, device=device)
    index = torch.empty((max(n, 0),), dtype=torch.int64, device=device)
    result = torch.empty((2,), dtype=torch.int64, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.ttl_select_streamlines(_lib.ptr(offsets), max(n, 0), _lib.ptr(keep), _lib.ptr(scores),
                                              float(threshold), _lib.ptr(work), nbytes, _lib.ptr(out_off),
                                              _lib.ptr(index), _lib.ptr(result), sp), 'ttl_select_streamlines')
        m, total = (int(v) for v in result.cpu())
        out = torch.empty((total, 3), dtype=torch.float32, device=device)
        _lib.check(lib.ttl_gather_streamlines(_lib.ptr(data), _lib.ptr(offsets), _lib.ptr(index), _lib.ptr(out_off),
                                              m, _lib.ptr(out), sp), 'ttl_gather_streamlines')
    return out, out_off[:m + 1], index[:m]


def tract_maps_packed(data, offsets, dims, density=None, endpoints=None):
    """Streamline density and endpoint maps of packed voxel-space streamlines (``ttl_tract_maps``), added in
    place into int32 CUDA tensors of shape ``dims`` (X, Y, Z) on the points' device; either may be None, not
    both.  The voxel of a point is ``floor(p + 0.5)`` per axis; ``density[v]`` counts the streamlines with a
    point in v, ``endpoints[v]`` their first and last points in v.  Returns the number of points outside the
    grid (one small device-to-host copy)."""
    device = _dev(data.device)
    lib = _lib.load()
    data, offsets = _to_device(data, offsets, device)
    dims = tuple(int(d) for d in dims)
    if density is None and endpoints is None:
        raise ValueError('tract_maps_packed needs a density map, an endpoint map or both')
    for m in (density, endpoints):
        if m is not None and (m.device != device or m.dtype != torch.int32 or tuple(m.shape) != dims
                              or not m.is_contiguous()):
            raise ValueError('maps must be contiguous int32 tensors of shape %r on %s' % (dims, device))
    n = int(offsets.shape[0]) - 1
    skipped = torch.zeros((1,), dtype=torch.int64, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.ttl_tract_maps(_lib.ptr(data), _lib.ptr(offsets), max(n, 0), *dims, _lib.ptr(density),
                                      _lib.ptr(endpoints), _lib.ptr(skipped), _lib.stream_ptr(device)),
                   'ttl_tract_maps')
        return int(skipped.item())


CONNECTOME_MAX_LABEL = 16383       # K <= TTL_CONNECTOME_MAX_LABELS (include/ttl_b200.h)
CONNECTOME_MAX_RADIUS_VOX = 8.0    # TTL_CONNECTOME_MAX_RADIUS


def radius_voxels(radius_mm, affine):
    """A connectivity search radius in mm -> voxels of the grid of ``affine``, the voxel size taken as
    ``track_to_file`` takes it (the mean of |diagonal| of the vox -> RAS mm affine).  Raises ValueError for a
    negative or non-finite radius, or one of more than 8 voxels."""
    radius_mm = float(radius_mm)
    if not 0.0 <= radius_mm < float('inf'):
        raise ValueError('the connectivity radius must be a finite number of mm >= 0, not %r' % radius_mm)
    vox_size = float(np.mean(np.abs(np.asarray(affine, dtype=np.float64))[np.diag_indices(4)][:3]))
    r = radius_mm / vox_size
    if not r <= CONNECTOME_MAX_RADIUS_VOX:
        raise ValueError('a connectivity radius of %g mm is %g voxels of %g mm: at most %g voxels are searched'
                         % (radius_mm, r, vox_size, CONNECTOME_MAX_RADIUS_VOX))
    return r


def unlabelled_endpoints(matrix):
    """The number of endpoints given label 0 in a connectivity matrix (numpy): one count in row 0 each, two
    for a streamline with both ends at 0."""
    m = np.asarray(matrix)
    return 2 * int(m[0, 0]) + int(m[0, 1:].sum(dtype=np.int64))


def connectome_packed(data, offsets, labels, matrix=None, radius_vox=0.0, pairs=False):
    """Structural connectivity of packed voxel-space streamlines over ``labels``, an int32 CUDA volume
    (X, Y, Z) on the points' device (``ttl_connectome``).  An endpoint's label is that of its own voxel
    ``floor(p + 0.5)`` when labelled, else that of the nearest labelled voxel within ``radius_vox`` voxels
    (ties to the smaller linear index), else 0.  A streamline with end labels (a, b) is added in place into
    ``matrix`` (int32 CUDA [K, K], K = max label + 1): 1 at [a, a] when a == b, else 1 at [a, b] and at [b, a].
    With ``pairs``, returns the int32 [n, 2] CUDA tensor of the labels of every streamline's first and last
    points, else None.  ``matrix`` may be None when ``pairs`` is set (K is then ``labels.max() + 1``)."""
    device = _dev(data.device)
    lib = _lib.load()
    data, offsets = _to_device(data, offsets, device)
    if matrix is None and not pairs:
        raise ValueError('connectome_packed needs a matrix, pairs or both')
    if (not isinstance(labels, torch.Tensor) or labels.device != device or labels.dtype != torch.int32
            or labels.dim() != 3 or not labels.is_contiguous()):
        raise ValueError('labels must be a contiguous int32 tensor (X, Y, Z) on %s' % device)
    if matrix is not None:
        if (matrix.device != device or matrix.dtype != torch.int32 or matrix.dim() != 2
                or matrix.shape[0] != matrix.shape[1] or not matrix.is_contiguous()):
            raise ValueError('matrix must be a contiguous square int32 tensor on %s' % device)
        K = int(matrix.shape[0])
    else:
        K = int(labels.max().item()) + 1 if labels.numel() else 1
    n = max(int(offsets.shape[0]) - 1, 0)
    out = torch.zeros((n, 2), dtype=torch.int32, device=device) if pairs else None
    with torch.cuda.device(device):
        _lib.check(lib.ttl_connectome(_lib.ptr(data), _lib.ptr(offsets), n, _lib.ptr(labels), *labels.shape, K,
                                      float(radius_vox), _lib.ptr(matrix), _lib.ptr(out), _lib.stream_ptr(device)),
                   'ttl_connectome')
    return out


SAMPLE_MAX_METRICS = 8             # TTL_SAMPLE_MAX_METRICS (include/ttl_b200.h)
SUMS_MAX_SHIFT = 62                # TTL_CONNECTOME_SUMS_MAX_SHIFT


def sample_metrics_packed(data, offsets, volumes):
    """Per-streamline means of scalar maps along packed voxel-space streamlines (``ttl_sample_metrics``).
    ``volumes``: a contiguous float32 CUDA tensor (X, Y, Z, C), C in [1, 8], on the points' device.  A point is
    sampled when ``tract_maps_packed`` counts it (its voxel ``floor(p + 0.5)`` is in the grid); its value is the
    fp64 trilinear interpolation with the corner indices clamped to the grid (scipy ``map_coordinates(order=1)``
    inside [0, n-1]).  Returns (means, skipped): float32 CUDA [n, C], the fp64 mean of the sampled values rounded
    once to float32 (NaN when no point is sampled), and the number of points not sampled (one small
    device-to-host copy).  A streamline's means do not depend on its batch or its position in it."""
    device = _dev(data.device)
    lib = _lib.load()
    data, offsets = _to_device(data, offsets, device)
    if (not isinstance(volumes, torch.Tensor) or volumes.device != device or volumes.dtype != torch.float32
            or volumes.dim() != 4 or not volumes.is_contiguous()
            or not 1 <= int(volumes.shape[3]) <= SAMPLE_MAX_METRICS):
        raise ValueError('volumes must be a contiguous float32 tensor (X, Y, Z, C), C in [1, %d], on %s'
                         % (SAMPLE_MAX_METRICS, device))
    n = max(int(offsets.shape[0]) - 1, 0)
    C = int(volumes.shape[3])
    means = torch.empty((n, C), dtype=torch.float32, device=device)
    skipped = torch.zeros((1,), dtype=torch.int64, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.ttl_sample_metrics(_lib.ptr(data), _lib.ptr(offsets), n, _lib.ptr(volumes), C,
                                          *volumes.shape[:3], _lib.ptr(means), _lib.ptr(skipped),
                                          _lib.stream_ptr(device)), 'ttl_sample_metrics')
        return means, int(skipped.item())


def metric_shift(bound):
    """The fixed-point shift S of edge sums for values with |v| <= ``bound``: S = clamp(31 - e, 0, 62) where
    bound < 2^e, so that every |round(v * 2^S)| <= 2^31 and any 2^31 streamlines sum within +-2^62 in int64.
    Raises ValueError for a negative or non-finite bound, or one >= 2^31."""
    bound = float(bound)
    if not 0.0 <= bound < 2.0 ** 31:
        raise ValueError('edge values bounded by %r cannot be summed exactly in int64: the largest |value| must be '
                         'finite and below 2^31' % bound)
    return min(max(31 - math.frexp(bound)[1], 0), SUMS_MAX_SHIFT)


def connectome_sums_packed(pairs, values, shifts, sums, counts):
    """Metric-weighted connectivity (``ttl_connectome_sums``), added in place.  ``pairs``: int32 CUDA [n, 2], the
    end labels of ``connectome_packed(pairs=True)``; ``values``: float32 CUDA [n, C]; ``shifts``: C ints
    (``metric_shift``).  A finite value v of column c adds round(v * 2^shifts[c]) to ``sums[c, a, b]`` (int64 CUDA
    [C, K, K]) and 1 to ``counts[c, a, b]`` (int32 CUDA [C, K, K]), and the same at [b, a] when a != b; NaN adds
    nothing.  The planes are exact integer sums: they do not depend on the order of streamlines or calls."""
    device = _dev(values.device if isinstance(values, torch.Tensor) else None)
    lib = _lib.load()
    if (not isinstance(values, torch.Tensor) or values.device != device or values.dtype != torch.float32 or values.dim() != 2
            or not values.is_contiguous()):
        raise ValueError('values must be a contiguous float32 tensor [n, C] on %s' % device)
    n, C = (int(s) for s in values.shape)
    if (not isinstance(pairs, torch.Tensor) or pairs.device != device or pairs.dtype != torch.int32
            or tuple(pairs.shape) != (n, 2) or not pairs.is_contiguous()):
        raise ValueError('pairs must be a contiguous int32 tensor [%d, 2] on %s' % (n, device))
    for name, t, dtype in (('sums', sums, torch.int64), ('counts', counts, torch.int32)):
        if (not isinstance(t, torch.Tensor) or t.device != device or t.dtype != dtype or t.dim() != 3
                or t.shape[0] != C or t.shape[1] != t.shape[2] or not t.is_contiguous()):
            raise ValueError('%s must be a contiguous %s tensor [%d, K, K] on %s' % (name, dtype, C, device))
    if sums.shape != counts.shape:
        raise ValueError('sums and counts must have the same shape')
    sh = np.ascontiguousarray(np.asarray(shifts, dtype=np.int64).reshape(-1))
    if sh.shape != (C,) or sh.min(initial=0) < 0 or sh.max(initial=0) > SUMS_MAX_SHIFT:
        raise ValueError('shifts must be %d integers in [0, %d]' % (C, SUMS_MAX_SHIFT))
    sh = sh.astype(np.int32)
    with torch.cuda.device(device):
        _lib.check(lib.ttl_connectome_sums(_lib.ptr(pairs), n, _lib.ptr(values), C, int(sums.shape[1]),
                                           sh.ctypes.data, _lib.ptr(sums), _lib.ptr(counts),
                                           _lib.stream_ptr(device)), 'ttl_connectome_sums')


def edge_means(sums, counts, shifts):
    """The mean value of every edge from ``connectome_sums_packed``'s planes: float64 numpy [C, K, K],
    (sums * 2^-shift) / counts, NaN where the count is 0."""
    s = np.asarray(sums.cpu() if isinstance(sums, torch.Tensor) else sums, dtype=np.int64)
    c = np.asarray(counts.cpu() if isinstance(counts, torch.Tensor) else counts, dtype=np.int64)
    sh = np.asarray(shifts, dtype=np.int32).reshape(-1, 1, 1)
    with np.errstate(invalid='ignore', divide='ignore'):
        out = np.ldexp(s.astype(np.float64), -sh) / c
    out[c == 0] = np.nan
    return out
