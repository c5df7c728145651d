"""Per-streamline post-processing of a packed tractogram on the device (reference:
tracking/tracker.py:118-125): dipy ``length`` for the min/max length filter and dipy
``compress_streamlines`` for ``--compress``.  Packed layout: ``data`` [total, 3] float32 and
``offsets`` [n + 1] int64 (streamline i = data[offsets[i]:offsets[i+1]])."""
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
