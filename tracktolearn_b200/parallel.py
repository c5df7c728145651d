"""Multi-GPU plumbing for tracking: seed sharding and the final tractogram gather.

The path shards by seed (SURVEY.md section 8(e)): every rank holds a replica of the volume,
mask and actor, tracks its own contiguous slice of the (globally shuffled) seeds and there is
no collective on the data path.  The only exchange is at the end: ranks send their packed
streamlines to rank 0, which concatenates them in rank order -- the same order a single GPU
would have produced.  Works with any ``torch.distributed`` backend (NCCL on GPUs, gloo in the
CPU tests): only host logic lives here.
"""
import numpy as np
import torch
import torch.distributed as dist

from tracktolearn_b200.tracking.tractogram import Tractogram


def shard_bounds(n, rank, world):
    """Contiguous slice [start, end) of n items for `rank`; sizes differ by at most one and
    concatenating the slices in rank order gives back 0..n."""
    base, rem = divmod(n, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def shard_seeds(seeds, rank=None, world=None):
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    s, e = shard_bounds(len(seeds), rank, world)
    return seeds[s:e]


def sharded_scores(n_items, score_chunk, device=None):
    """Per-item scores computed by all ranks together (SURVEY.md section 8(e), oracle scoring): rank k
    scores the contiguous chunk ``shard_bounds(n_items, k, world)`` with ``score_chunk(start, end) ->
    float32 tensor [end - start]`` and one ``all_gather_into_tensor`` of the (padded) chunks hands every
    rank the full ``[n_items]`` tensor, in item order.  Without torch.distributed: ``score_chunk(0, n)``."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        return score_chunk(0, n_items)
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = device if device is not None else _device_for_backend()
    s, e = shard_bounds(n_items, rank, world)
    pad = -(-n_items // world)                       # chunk sizes differ by at most one
    mine = torch.zeros((pad,), dtype=torch.float32, device=dev)
    if e > s:
        mine[:e - s] = score_chunk(s, e).to(dev, dtype=torch.float32).reshape(-1)
    full = torch.empty((world * pad,), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(full, mine)
    parts = []
    for r in range(world):
        rs, re = shard_bounds(n_items, r, world)
        parts.append(full[r * pad:r * pad + (re - rs)])
    return torch.cat(parts) if parts else full[:0]


def _device_for_backend():
    if dist.get_backend() == 'nccl':
        return torch.device('cuda', torch.cuda.current_device())
    return torch.device('cpu')


_PINNED = {}


def _pinned(nbytes):
    """Grow-only pinned staging buffer (a fresh 1 GB cudaHostAlloc per gather costs more than the
    transfer it serves)."""
    cur = _PINNED.get('buf')
    if cur is None or cur.numel() < nbytes:
        cur = torch.empty((int(nbytes * 1.25) + 4096,), dtype=torch.uint8, pin_memory=True)
        _PINNED['buf'] = cur
    return cur


def _pinned_named(name, nbytes):
    cur = _PINNED.get(name)
    if cur is None or cur.numel() < nbytes:
        cur = torch.empty((int(nbytes * 1.25) + 4096,), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
        _PINNED[name] = cur
    return cur


class _HostArena(object):
    """A block of host memory shared by the ranks of ONE node (a file in /dev/shm mapped by every rank)
    and page-locked in every rank's CUDA context (cudaHostRegister), grown on demand and kept.  Every
    rank's GPU can DMA into it over its own PCIe link, which is what makes the single-node tractogram
    gather scale: through NCCL the 4 GB of an 8-GPU run all cross rank 0's link (411 ms end to end for
    6.4 M streamlines); into the arena they cross eight links at once."""

    def __init__(self):
        self.buf = None
        self.nbytes = 0
        self.generation = 0
        self.failed = False

    def _release(self):
        if self.buf is not None and torch.cuda.is_available():
            try:
                torch.cuda.cudart().cudaHostUnregister(self.buf.data_ptr())
            except Exception:
                pass
        self.buf = None
        self.nbytes = 0

    def ensure(self, nbytes):
        """All ranks call this with the same `nbytes`.  Returns the uint8 tensor over the shared block, or
        None -- on EVERY rank -- when any rank could not set it up (no /dev/shm, too small, registration
        refused): the caller then takes the NCCL route."""
        if self.failed:
            return None
        if self.buf is not None and self.nbytes >= nbytes:
            return self.buf
        import os
        self._release()
        rank = dist.get_rank()
        self.generation += 1
        size = int(nbytes * 1.25) + (1 << 20)
        token = [None]
        if rank == 0:
            try:
                path = '/dev/shm/ttl_b200_arena_%d_%d_%d' % (os.getpid(), self.generation,
                                                             int.from_bytes(os.urandom(4), 'little'))
                with open(path, 'wb') as f:
                    f.truncate(size)
                token[0] = path
            except Exception:
                token[0] = None
        dist.broadcast_object_list(token, src=0)
        path = token[0]
        buf, ok = None, path is not None
        if ok:
            try:
                buf = torch.from_file(path, shared=True, size=size, dtype=torch.uint8)
                if torch.cuda.is_available():
                    rc = torch.cuda.cudart().cudaHostRegister(buf.data_ptr(), size, 1)      # cudaHostRegisterPortable
                    ok = int(rc) == 0
            except Exception:
                ok = False
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=_device_for_backend())
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)          # also the barrier before the file is unlinked
        if rank == 0 and path is not None:
            try:
                os.unlink(path)      # the mappings keep the pages alive
            except OSError:
                pass
        if int(flag.item()) == 0:
            if buf is not None and ok and torch.cuda.is_available():
                try:
                    torch.cuda.cudart().cudaHostUnregister(buf.data_ptr())
                except Exception:
                    pass
            self.failed = True
            return None
        self.buf, self.nbytes = buf, size
        return buf


_ARENA = _HostArena()


def _single_node():
    import os
    try:
        return int(os.environ.get('LOCAL_WORLD_SIZE', '0')) == dist.get_world_size()
    except Exception:
        return False


def _gather_via_arena(parts, dst, copy):
    """parts: [(tensor [rows, width] on this rank's device or host, width, dtype, name)].  One all_gather of
    the row counts (NCCL), then every rank copies ITS rows into its slice of the shared pinned arena (D2H over
    its own PCIe link), one barrier, and `dst` reads the result in place."""
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = _device_for_backend()
    counts_mine = torch.tensor([int(p[0].shape[0]) for p in parts], dtype=torch.int64, device=dev)
    all_counts = [torch.zeros_like(counts_mine) for _ in range(world)]
    dist.all_gather(all_counts, counts_mine)
    counts = torch.stack(all_counts).cpu().numpy()                  # [world, n_parts]
    # arena layout: part after part, ranks in order inside a part, every region 64-byte aligned
    layout, off = [], 0
    for j, (_, width, dtype, _) in enumerate(parts):
        es = torch.empty((), dtype=dtype).element_size() * width
        starts = []
        for r in range(world):
            starts.append(off)
            off += int(counts[r, j]) * es
        layout.append((starts, es))
        off = (off + 63) // 64 * 64
    arena = _ARENA.ensure(max(off, 64))
    if arena is None:
        return 'unavailable'
    for j, (mine, width, dtype, _) in enumerate(parts):
        n = int(mine.shape[0])
        if n == 0:
            continue
        starts, es = layout[j]
        view = arena[starts[rank]:starts[rank] + n * es].view(dtype).view(n, width)
        view.copy_(mine, non_blocking=True)
    if torch.cuda.is_available():
        torch.cuda.current_stream().synchronize()
    dist.barrier()
    if rank != dst:
        return None
    out = []
    for j, (_, width, dtype, _) in enumerate(parts):
        starts, es = layout[j]
        total = int(counts[:, j].sum())
        # the ranks' slices of a part are contiguous (no padding inside a part)
        a = arena[starts[0]:starts[0] + total * es].view(dtype).view(total, width).numpy()
        out.append(a.copy() if copy else a)
    return out


def gather_packed(points, lengths, seeds, flags, dst=0, copy=True, via='auto', scores=None):
    """Gather packed streamlines on rank `dst` in rank order.

    ``via``: 'nccl' -- the data travels through NCCL to `dst`'s GPU and over its PCIe link (below);
    'host' -- every rank copies its part into a shared pinned host arena over its own link (one node
    only; NCCL carries the sizes and the barrier); 'auto' -- 'host' when all ranks are on this node and
    the backend is NCCL, else 'nccl'.

    ``points`` [n_pts, 3] float32, ``lengths`` [n] int64, ``seeds`` [n, 3] float64, ``flags`` [n] int64:
    tensors on this rank's device for the backend (CUDA under NCCL -- e.g. straight from
    ``env.get_streamlines_device()``, no host round trip -- CPU under gloo).  One all_gather of the
    sizes, then every rank sends exactly its rows into its slice of `dst`'s buffers (batched
    point-to-point: device-to-device over NVLink under NCCL) and `dst` makes one D2H copy per array
    into grow-only pinned memory.  With ``copy=False`` the returned arrays are views of that pinned
    memory, valid until the next gather.  ``scores`` [n] float32 (optional): per-streamline oracle scores,
    carried along and returned as ``data_per_streamline['oracle_score']``.  Returns a Tractogram on `dst`,
    None elsewhere."""
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = _device_for_backend()
    if via == 'auto':
        import os
        via = 'host' if (dist.get_backend() == 'nccl' and _single_node()
                         and os.environ.get('TTL_GATHER', 'host') != 'nccl') else 'nccl'
    if via == 'host':
        # seeds usually live on the host already: they go to the arena by a plain memcpy
        parts = [(points.to(dtype=torch.float32).reshape(-1, 3), 3, torch.float32, 'pts'),
                 (lengths.to(dtype=torch.int64).reshape(-1, 1), 1, torch.int64, 'len'),
                 (seeds.to(dtype=torch.float64).reshape(-1, 3), 3, torch.float64, 'seeds'),
                 (flags.to(dtype=torch.int64).reshape(-1, 1), 1, torch.int64, 'flags')]
        if scores is not None:
            parts.append((scores.to(dtype=torch.float32).reshape(-1, 1), 1, torch.float32, 'scores'))
        arrs = _gather_via_arena(parts, dst, copy)
        if arrs is None:
            return None
        if not isinstance(arrs, str):
            return _packed_tractogram(arrs)
        # the arena could not be set up on some rank (every rank knows): the NCCL route below
    parts = [(points.to(dev, dtype=torch.float32).reshape(-1, 3).contiguous(), 3, torch.float32, 'pts'),
             (lengths.to(dev, dtype=torch.int64).reshape(-1, 1).contiguous(), 1, torch.int64, 'len'),
             (seeds.to(dev, dtype=torch.float64).reshape(-1, 3).contiguous(), 3, torch.float64, 'seeds'),
             (flags.to(dev, dtype=torch.int64).reshape(-1, 1).contiguous(), 1, torch.int64, 'flags')]
    if scores is not None:
        parts.append((scores.to(dev, dtype=torch.float32).reshape(-1, 1).contiguous(), 1, torch.float32, 'scores'))
    n_sl, n_pts = int(parts[1][0].shape[0]), int(parts[0][0].shape[0])
    sizes = torch.tensor([n_sl, n_pts], dtype=torch.int64, device=dev)
    all_sizes = [torch.zeros_like(sizes) for _ in range(world)]
    dist.all_gather(all_sizes, sizes)
    all_sizes = torch.stack(all_sizes).cpu().numpy()
    n_per, p_per = all_sizes[:, 0], all_sizes[:, 1]
    ops, bufs = [], []
    for mine, width, dtype, name in parts:
        counts = p_per if name == 'pts' else n_per
        if rank == dst:
            buf = torch.empty((int(counts.sum()), width), dtype=dtype, device=dev)
            o = 0
            for r in range(world):
                c = int(counts[r])
                if r == dst:
                    buf[o:o + c].copy_(mine)
                elif c > 0:
                    ops.append(dist.P2POp(dist.irecv, buf[o:o + c], r))
                o += c
            bufs.append(buf)
        elif int(counts[rank]) > 0:
            ops.append(dist.P2POp(dist.isend, mine, dst))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    if rank != dst:
        return None
    host = []
    for buf, (_, _, dtype, name) in zip(bufs, parts):
        if buf.is_cuda:
            nbytes = buf.numel() * buf.element_size()
            h = _pinned_named(name, nbytes)[:nbytes].view(dtype).view(buf.shape)
            h.copy_(buf, non_blocking=True)
            host.append(h)
        else:
            host.append(buf)
    if bufs and bufs[0].is_cuda:
        torch.cuda.current_stream(bufs[0].device).synchronize()
    return _packed_tractogram([h.numpy().copy() if copy else h.numpy() for h in host])


def _packed_tractogram(arrs):
    """[points, lengths, seeds, flags(, scores)] host arrays in gather_packed's part order -> Tractogram."""
    data, lens, gseeds, gflags = arrs[:4]
    offsets = np.concatenate(([0], np.cumsum(lens[:, 0]))).astype(np.int64)
    per = {'seeds': gseeds, 'flags': gflags[:, 0]}
    if len(arrs) > 4:
        per['oracle_score'] = arrs[4][:, 0]
    return Tractogram(data=data, offsets=offsets, data_per_streamline=per)


def gather_tractogram(local, dst=0, copy=True, via='auto'):
    """Gather host-side packed tractograms (``Tractogram``) on rank `dst` in rank order; returns the
    merged Tractogram on `dst` and None elsewhere.  Prefer ``gather_env_streamlines`` when the
    streamlines are still on the device."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return local
    n_sl = len(local)
    return gather_packed(
        torch.as_tensor(np.ascontiguousarray(local.data, dtype=np.float32)).reshape(-1, 3),
        torch.as_tensor(np.diff(local.offsets).astype(np.int64)),
        torch.as_tensor(np.ascontiguousarray(local.data_per_streamline.get('seeds', np.zeros((n_sl, 3))),
                                             dtype=np.float64)).reshape(-1, 3),
        torch.as_tensor(np.asarray(local.data_per_streamline.get('flags', np.zeros(n_sl))).astype(np.int64)),
        dst=dst, copy=copy, via=via)


def gather_env_streamlines(env, dst=0, copy=True, via='auto'):
    """The final exchange of a multi-GPU tracking run, from the device: this rank's packed streamlines
    (``env.get_streamlines_device()``), seeds and flags go to rank `dst` without touching the host on
    the sending side.  Single process: the env's own tractogram."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return env.get_streamlines(copy=copy)
    pts, offsets = env.get_streamlines_device()
    n = int(offsets.shape[0]) - 1
    seeds = torch.as_tensor(np.ascontiguousarray(env.initial_points, dtype=np.float64)).reshape(-1, 3)
    return gather_packed(pts, offsets[1:] - offsets[:-1], seeds, env._batch.flags[:n].to(torch.int64),
                         dst=dst, copy=copy, via=via)
