"""TRK (TrackVis v2) and TCK (MRtrix) writers / readers for packed streamlines -- the tractogram
formats ``ttl_track.py`` writes (reference: runners/ttl_track.py:179-186 through nibabel).

Space conventions written here (the intent of tracking/tracker.py:127-136):
  * .trk stores "voxmm": (voxel coordinate + 0.5) * voxel size, corner origin, plus the
    vox->RAS mm affine in the header;
  * .tck stores RAS mm: voxel coordinates through the vox->RAS mm affine.
"""
import struct

import numpy as np


def detect_format(path):
    p = str(path).lower()
    if p.endswith('.trk'):
        return 'trk'
    if p.endswith('.tck'):
        return 'tck'
    raise ValueError('Invalid output streamline file format (must be trk or tck): {0}'.format(path))


def _voxel_order(affine):
    lab = (('L', 'R'), ('P', 'A'), ('I', 'S'))
    out = ''
    R = np.asarray(affine)[:3, :3]
    for j in range(3):
        i = int(np.argmax(np.abs(R[:, j])))
        out += lab[i][1] if R[i, j] > 0 else lab[i][0]
    return out


class TrkWriter(object):
    """Streams (data, offsets) batches to a .trk file; the streamline count is patched on close.
    Per-streamline properties: ``seeds_x/y/z`` (``save_seeds``), then ``oracle_score`` (``save_scores``), then
    ``start_label`` and ``end_label`` (``save_labels``: connectivity labels, integers held exactly in float32), then
    ``mean_NAME`` for every name of ``metric_names`` (per-streamline metric means).  The header has room for 10
    properties: more raise ValueError."""

    MAX_PROPERTIES = 10

    def __init__(self, path, dims, voxel_sizes, affine, save_seeds=False, save_scores=False, save_labels=False,
                 metric_names=()):
        names = (((b'seeds_x', b'seeds_y', b'seeds_z') if save_seeds else ()) + ((b'oracle_score',) if save_scores else ())
                 + ((b'start_label', b'end_label') if save_labels else ())
                 + tuple(b'mean_' + str(m).encode() for m in metric_names))
        if len(names) > self.MAX_PROPERTIES:
            raise ValueError('a .trk file holds at most %d per-streamline properties, not %d'
                             % (self.MAX_PROPERTIES, len(names)))
        if any(len(name) > 19 for name in names):
            raise ValueError('a .trk property name has at most 19 bytes: %r' % [n for n in names if len(n) > 19])
        self.f = open(path, 'wb')
        self.n = 0
        self.save_seeds = save_seeds
        self.save_scores = save_scores
        self.save_labels = save_labels
        self.n_metrics = len(metric_names)
        hdr = bytearray(1000)
        hdr[0:6] = b'TRACK\x00'
        struct.pack_into('<3h', hdr, 6, *[int(d) for d in dims])
        struct.pack_into('<3f', hdr, 12, *[float(v) for v in voxel_sizes])
        struct.pack_into('<3f', hdr, 24, 0.0, 0.0, 0.0)
        struct.pack_into('<h', hdr, 36, 0)                                   # n_scalars
        struct.pack_into('<h', hdr, 238, len(names))                         # n_properties
        for i, name in enumerate(names):
            hdr[240 + 20 * i:240 + 20 * i + len(name)] = name
        struct.pack_into('<16f', hdr, 440, *np.asarray(affine, dtype=np.float32).reshape(-1))
        vo = _voxel_order(affine).encode()
        hdr[948:948 + len(vo)] = vo
        struct.pack_into('<i', hdr, 988, 0)                                  # n_count, patched later
        struct.pack_into('<i', hdr, 992, 2)                                  # version
        struct.pack_into('<i', hdr, 996, 1000)                               # hdr_size
        self.f.write(bytes(hdr))

    def write(self, data, offsets, seeds=None, scores=None, labels=None, means=None):
        n = len(offsets) - 1
        if n <= 0:
            return
        lens = np.diff(offsets).astype(np.int64)
        n_prop = ((3 if self.save_seeds else 0) + (1 if self.save_scores else 0) + (2 if self.save_labels else 0)
                  + self.n_metrics)
        total = int(lens.sum()) * 3 + n * (1 + n_prop)
        out = np.empty(total, dtype='<f4')
        # positions of the int32 counts inside the float buffer
        starts = np.concatenate(([0], np.cumsum(lens * 3 + 1 + n_prop)[:-1])).astype(np.int64)
        out.view('<i4')[starts] = lens.astype(np.int32)
        idx = np.repeat(starts + 1 - offsets[:-1] * 3, lens * 3) + np.arange(int(lens.sum()) * 3)
        out[idx] = np.asarray(data, dtype=np.float32).reshape(-1)
        if self.save_seeds:
            ps = starts + 1 + lens * 3
            for c in range(3):
                out[ps + c] = np.asarray(seeds, dtype=np.float32)[:, c]
        if self.save_scores:
            out[starts + lens * 3 + 1 + (3 if self.save_seeds else 0)] = np.asarray(scores, dtype=np.float32).reshape(-1)
        if self.save_labels:
            lab = np.asarray(labels).reshape(-1, 2).astype(np.float32)
            out[starts + lens * 3 + n_prop - 1 - self.n_metrics] = lab[:, 0]
            out[starts + lens * 3 + n_prop - self.n_metrics] = lab[:, 1]
        if self.n_metrics:
            m = np.asarray(means, dtype=np.float32).reshape(n, self.n_metrics)
            for c in range(self.n_metrics):
                out[starts + lens * 3 + n_prop - self.n_metrics + 1 + c] = m[:, c]
        self.f.write(out.tobytes())
        self.n += n

    def close(self):
        self.f.seek(988)
        self.f.write(struct.pack('<i', self.n))
        self.f.close()


class TckWriter(object):
    def __init__(self, path):
        self.f = open(path, 'wb')
        self.n = 0
        self._write_header(0)

    def _write_header(self, count):
        lines = ['mrtrix tracks', 'datatype: Float32LE', 'count: %010d' % count]
        hdr = '\n'.join(lines) + '\n'
        offset = len(hdr) + len('file: . ') + 5 + len('\nEND\n')
        text = hdr + 'file: . %05d' % offset + '\nEND\n'
        assert len(text) == offset
        self.f.seek(0)
        self.f.write(text.encode())
        self.offset = offset

    def write(self, data, offsets, seeds=None, scores=None, labels=None, means=None):
        """``seeds``, ``scores``, ``labels`` and ``means`` are accepted for TrkWriter's signature: .tck has no
        per-streamline data."""
        n = len(offsets) - 1
        if n <= 0:
            return
        lens = np.diff(offsets).astype(np.int64)
        total = int(lens.sum()) + n
        out = np.full((total, 3), np.nan, dtype='<f4')
        starts = offsets[:-1] + np.arange(n)
        idx = np.repeat(starts - offsets[:-1], lens) + np.arange(int(lens.sum()))
        out[idx] = np.asarray(data, dtype=np.float32).reshape(-1, 3)
        self.f.seek(0, 2)
        self.f.write(out.tobytes())
        self.n += n

    def close(self):
        self.f.seek(0, 2)
        self.f.write(np.full((1, 3), np.inf, dtype='<f4').tobytes())
        self._write_header(self.n)
        self.f.close()


def read_trk(path, spans=False):
    """-> (data [sum L,3] float32 in voxmm, offsets, header dict).  ``spans=True``: also the byte span
    [start, end) of every record in the file, as a fourth item (int64 arrays (start, end))."""
    with open(path, 'rb') as f:
        raw = f.read()
    n_scalars = struct.unpack('<h', raw[36:38])[0]
    n_prop = struct.unpack('<h', raw[238:240])[0]
    n_count = struct.unpack('<i', raw[988:992])[0]
    hdr = {'dims': struct.unpack('<3h', raw[6:12]), 'voxel_sizes': struct.unpack('<3f', raw[12:24]),
           'affine': np.array(struct.unpack('<16f', raw[440:504])).reshape(4, 4), 'n_count': n_count,
           'voxel_order': raw[948:951].decode(), 'n_properties': n_prop, 'n_scalars': n_scalars,
           'property_names': [raw[240 + 20 * i:260 + 20 * i].split(b'\x00')[0].decode() for i in range(n_prop)]}
    body = np.frombuffer(raw, dtype='<f4', offset=1000)
    # the records are found by walking their counts (each position depends on the previous count); the
    # points are then what is left once the count and property words are masked out
    ints = memoryview(raw)[1000:1000 + (len(raw) - 1000) // 4 * 4].cast('i')
    w = 3 + n_scalars
    starts, lens = [0] * n_count, [0] * n_count
    pos = 0
    for i in range(n_count):
        L = ints[pos]
        starts[i] = pos
        lens[i] = L
        pos += 1 + L * w + n_prop
    starts, lens = np.asarray(starts, dtype=np.int64), np.asarray(lens, dtype=np.int64)
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    prop_at = starts + 1 + lens * w
    is_point = np.ones((pos,), dtype=bool)
    is_point[starts] = False
    for k in range(n_prop):
        is_point[prop_at + k] = False
    data = np.ascontiguousarray(body[:pos][is_point].reshape(-1, w)[:, :3])
    hdr['properties'] = body[prop_at[:, None] + np.arange(n_prop)] if n_count else np.asarray([])
    if spans:
        return data, offsets, hdr, (1000 + 4 * starts, 1000 + 4 * (prop_at + n_prop))
    return data, offsets, hdr


def read_tck(path, spans=False):
    """-> (data [sum L,3] float32, offsets, header dict).  ``spans=True``: also the byte span [start, end)
    of every record, its NaN delimiter included, as a fourth item."""
    with open(path, 'rb') as f:
        raw = f.read()
    head = raw[:raw.index(b'END\n')].decode()
    offset = int([ln for ln in head.split('\n') if ln.startswith('file:')][0].split()[-1])
    count = int([ln for ln in head.split('\n') if ln.startswith('count:')][0].split()[-1])
    body = np.frombuffer(raw, dtype='<f4', offset=offset).reshape(-1, 3)
    is_nan = np.isnan(body[:, 0])
    is_inf = np.isinf(body[:, 0])
    ends = np.nonzero(is_nan)[0]
    lens = np.diff(np.concatenate(([-1], ends))) - 1
    data = body[~(is_nan | is_inf)]
    offsets = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    assert len(lens) == count
    if spans:
        return data, offsets, {'count': count}, (offset + 12 * (ends - lens), offset + 12 * (ends + 1))
    return data, offsets, {'count': count}
