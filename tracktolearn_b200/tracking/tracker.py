"""Tracker (reference: tracking/tracker.py:18-259).

``track`` keeps the reference's generator contract -- shuffle seeds, track batch after batch,
keep streamlines whose length is within [min_length, max_length] mm, move them to TRK or TCK
space, yield ``TractogramItem`` -- but by default it drives the env as a *streaming* tracker:
``n_actor`` streamlines are alive at once and slots freed by stopped streamlines take the next
seeds on the device, so the GPU stays full while the tail of long streamlines finishes.
At ``prob = 0`` every streamline depends only on its own seed, so the output is the same as
batch-by-batch tracking (tests/test_tracker_gpu.py).  At ``prob > 0`` that holds with a
``policy_seed``: the policy's eps is then drawn per (seed, seed index, point count) on the device
(ttl_policy); without one, eps comes from torch.randn in alive-list order and tracking goes batch by batch.
"""
import numpy as np
import torch

from tracktolearn_b200.tracking.tractogram import Tractogram, TractogramItem


def streamline_lengths(data, offsets):
    """dipy ``length`` for every packed streamline: sum of segment norms, in double."""
    n = len(offsets) - 1
    out = np.zeros(n, dtype=np.float64)
    if len(data) < 2 or n == 0:
        return out
    d = np.diff(data.astype(np.float64), axis=0)
    seg = np.sqrt((d * d).sum(-1))
    cs = np.concatenate(([0.0], np.cumsum(seg)))
    first, last = offsets[:-1], offsets[1:] - 1
    ok = last > first
    out[ok] = cs[last[ok]] - cs[first[ok]]
    return out


class Tracker(object):

    def __init__(self, alg, n_actor, prob=0., compress=0.0, min_length=20, max_length=200,
                 save_seeds=False, streaming=True, rows_per_pass=None, policy_seed=None):
        self.alg = alg
        self.n_actor = n_actor
        self.prob = prob
        self.policy_seed = policy_seed
        self.compress = compress
        self.min_length = min_length
        self.max_length = max_length
        self.save_seeds = save_seeds
        self.streaming = streaming
        self.rows_per_pass = rows_per_pass
        self.maps_skipped = 0       # points outside the grid in the maps of the last track_to_file
        self.connectome_unlabelled = 0      # endpoints given label 0 in the matrix of the last track_to_file
        self.metrics_unsampled = 0          # streamlines with no sampled point in the last track_to_file

    # ----------------------------------------------------------------------------------
    def _passes(self, env):
        n_seeds = len(env.seeds)
        if not self.streaming or (self.prob != 0. and self.policy_seed is None):
            for start in range(0, n_seeds, self.n_actor):
                yield start, min(start + self.n_actor, n_seeds), None
            return
        rows = self.rows_per_pass
        if rows is None:
            # streamline buffer budget: rows * (max_nb_steps+1) * 12 bytes <= ~24 GB of the 180 GB of
            # HBM3e (1M seeds at 799 points = 9.6 GB is one pass, hence one low-occupancy tail)
            rows = max(self.n_actor, int(24e9 // ((env.max_nb_steps + 1) * 12)))
        for start in range(0, n_seeds, rows):
            yield start, min(start + rows, n_seeds), self.n_actor

    def _check_range(self, env):
        """The fp16 tier saturates values outside +-65504 instead of producing infinities; a tractogram
        computed from saturated numbers would be silently wrong, so stop and say what to do."""
        actor = self.alg.agent.actor
        if getattr(actor, 'precision', None) != 'fp16':
            return
        if actor.overflowed() or env.operand_saturated():
            from tracktolearn_b200 import _lib
            raise _lib.TTLError('a state or activation value exceeded the fp16 range (65504) during tracking; '
                                're-run with precision="tf32" (--precision tf32)')

    def _run_pass(self, env, start, end, slots):
        """Track seeds [start, end) of the env: one streaming pass (or one plain batch)."""
        if slots is None or slots >= end - start:
            state = env.reset(start, end)
        else:
            # a tensor-core actor reads its operand rows only: do not materialise the fp32 state
            prec = getattr(self.alg.agent.actor, 'precision', 'fp32')
            tc_actor = prec in ('bf16', 'fp16', 'tf32')
            state = env.reset_streaming(start, end, slots, fp32_state=not tc_actor,
                                        operand=prec if tc_actor else None)
        self.alg.validation_episode(state, env, self.prob, policy_seed=self.policy_seed)
        self._check_range(env)

    def track_packed(self, env, copy=True):
        """Yields a Tractogram with voxel-space packed streamlines (+ seeds, flags) per pass;
        no length filter, no space change.  ``copy=False``: each batch aliases the env's pinned
        staging buffers and must be consumed before the next one is requested."""
        self.alg.agent.eval()
        for start, end, slots in self._passes(env):
            self._run_pass(env, start, end, slots)
            yield env.get_streamlines(copy=copy)

    def track_gathered(self, env, copy=True):
        """``track_packed`` for one process per GPU (torchrun): every rank tracks ITS seeds (the caller
        sharded ``env.seeds``, parallel.shard_seeds) and after each pass the packed streamlines of all
        ranks are gathered on rank 0 in rank order -- the order one GPU would have produced
        (tracker.py:106-145 collects batch after batch the same way).  Yields the merged Tractogram on
        rank 0 and None elsewhere; without torch.distributed it is ``track_packed``.  All ranks must make
        the same number of passes.  With device-drawn noise (``noise_rng='device'``) the caller also sets
        ``env.seed_offset`` to the index of its first seed in the unsharded list (``parallel.shard_bounds``),
        so that every seed gets the noise one GPU would give it."""
        from tracktolearn_b200 import parallel
        self.alg.agent.eval()
        for start, end, slots in self._passes(env):
            self._run_pass(env, start, end, slots)
            yield parallel.gather_env_streamlines(env, copy=copy)

    def track(self, env, tracts_format='trk'):
        """Reference: tracking/tracker.py:62-150.  ``tracts_format``: 'trk' / 'tck' (or the
        nibabel TrkFile / TckFile classes).  Returns a generator of TractogramItem."""
        affine = env.affine_vox2rasmm
        np.random.shuffle(env.seeds)      # tracker.py:94
        is_trk = 'trk' in str(tracts_format).lower()

        def tracking_generator():
            vox_size = np.mean(np.abs(affine)[np.diag_indices(4)][:3])
            scaled_min_length = self.min_length / vox_size
            scaled_max_length = self.max_length / vox_size
            compress_th_vox = self.compress / vox_size        # tracker.py:103: --compress is in mm
            for batch in self.track_packed(env):
                lens = streamline_lengths(batch.data, batch.offsets)
                keep = (scaled_min_length <= lens) & (lens <= scaled_max_length)
                seeds = batch.data_per_streamline['seeds']
                data, offsets = batch.data, batch.offsets
                if self.compress:     # tracker.py:123-125, on the device for the whole batch
                    data, offsets = self._compress(env, data, offsets, compress_th_vox)
                for i in np.nonzero(keep)[0]:
                    s = np.array(data[offsets[i]:offsets[i + 1]])
                    if is_trk:
                        s += 0.5
                        s *= vox_size
                    else:
                        s = np.dot(s, affine[:3, :3]) + affine[:3, 3]
                    seed_dict = {'seeds': seeds[i] - 0.5} if self.save_seeds else {}
                    yield TractogramItem(s, seed_dict, {})

        return tracking_generator()

    def _compress(self, env, data, offsets, tol_vox):
        """dipy ``compress_streamlines(streamline, compress_th_vox)`` (tracker.py:103,123-125: the
        tolerance given in mm divided by the voxel size, the streamlines being in voxel space) for a
        packed batch, on the env's device; returns host arrays."""
        from tracktolearn_b200.tracking.postprocess import compress_packed
        d, o = compress_packed(data, offsets, tol_error=float(tol_vox), device=env.device)
        return d.cpu().numpy(), o.cpu().numpy()

    def track_to_file(self, env, path, dims, voxel_sizes, oracle=None, oracle_threshold=0.5, save_scores=False,
                      density_path=None, endpoints_path=None, labels=None, connectivity_path=None,
                      connectivity_radius=0.0, save_labels=False, metrics=None, metric_names=(),
                      save_metric_means=False, metric_connectivity_prefix=None, length_connectivity_path=None):
        """What ``ttl_track.py`` does with ``track`` + ``nib.streamlines.save`` (runners/ttl_track.py:
        172-186), on packed arrays and on the device: dipy ``length`` and the min/max filter
        (tracker.py:118-121), ``compress_streamlines`` (:123-125), voxel -> file space (:127-136);
        only the kept, transformed float32 points cross PCIe, into pinned memory, and go to a
        streaming .trk / .tck writer.  Returns the number of streamlines kept.

        ``oracle`` (an ``OracleSingleton``): after the length filter, every streamline is scored by
        TractOracle-Net on its voxel-space points -- the coordinates the in-step ORACLE criterion scores --
        and kept when its score is >= ``oracle_threshold`` (the criterion stops below 0.5).  Scoring
        comes before ``--compress``, so a score does not depend on it.  Each rank scores its own
        streamlines: a streamline's score does not depend on the batch it is scored in, so the file is
        the same for every GPU count.  ``save_scores`` (.trk only) writes the scores as the
        per-streamline property ``oracle_score``.

        ``density_path`` / ``endpoints_path`` (.nii / .nii.gz): the streamline density and endpoint maps of the
        streamlines written, on the env's voxel grid (``postprocess.tract_maps_packed``), taken from their
        voxel-space points after the length and oracle filters and before ``--compress``; summed over the
        ranks onto rank 0, which writes them as int32 NIfTI with ``env.affine_vox2rasmm``.  The number of
        points outside the grid is kept in ``self.maps_skipped``.

        ``labels`` (an int32 volume of the env's grid on its device, ``ttl_connectivity.load_labels``): the
        structural connectivity of the streamlines written (``postprocess.connectome_packed``), from the same
        points as the maps, each endpoint labelled from its own voxel or the nearest labelled voxel within
        ``connectivity_radius`` mm.  ``connectivity_path`` (.npy): the int32 matrix [K, K], K = max label + 1,
        summed over the ranks onto rank 0, which writes it with ``np.save``; the number of endpoints given label
        0 is kept in ``self.connectome_unlabelled``.  ``save_labels`` (.trk only) writes every streamline's end
        labels as the per-streamline properties ``start_label`` and ``end_label``, after ``oracle_score``.

        ``metrics`` (a float32 volume (X, Y, Z, C) of the env's grid on its device, ``ttl_connectivity.load_metrics``)
        with ``metric_names`` (C names): tractometry of the streamlines written, from the same points as the maps
        (``postprocess.sample_metrics_packed``): every streamline's mean of each metric over its sampled points.
        ``save_metric_means`` (.trk only) writes them as the per-streamline properties ``mean_NAME``, after the
        labels.  With ``labels``, ``metric_connectivity_prefix`` writes PREFIX + NAME + '.npy' per metric and
        ``length_connectivity_path`` one .npy: the mean metric / mean length in mm of the streamlines of every edge,
        float64 [K, K], NaN where the count matrix is 0.  They are summed exactly (``postprocess.metric_shift``,
        ``connectome_sums_packed``) over the ranks onto rank 0, so they do not depend on batch order, passes,
        ``n_actor`` or GPU count.  The number of streamlines with no sampled point is kept in
        ``self.metrics_unsampled``."""
        from tracktolearn_b200.io.streamlines import TckWriter, TrkWriter, detect_format
        from tracktolearn_b200.tracking.postprocess import (compress_packed, connectome_packed, connectome_sums_packed,
                                                            edge_means, lengths_packed, metric_shift, radius_voxels,
                                                            sample_metrics_packed, select_packed, tract_maps_packed,
                                                            unlabelled_endpoints)
        import torch.distributed as dist
        from tracktolearn_b200 import parallel
        fmt = detect_format(path)
        if save_scores and oracle is None:
            raise ValueError('save_scores needs an oracle')
        if save_scores and fmt != 'trk':
            raise ValueError('.tck files cannot hold per-streamline data: save oracle scores to a .trk file')
        grid = (env._volume.X, env._volume.Y, env._volume.Z)
        weighted = metric_connectivity_prefix is not None or length_connectivity_path is not None
        if (connectivity_path is not None or save_labels or weighted) != (labels is not None):
            raise ValueError('a connectivity output needs labels, and labels need a connectivity output')
        if save_labels and fmt != 'trk':
            raise ValueError('.tck files cannot hold per-streamline data: save connectivity labels to a .trk file')
        if labels is not None:
            if tuple(labels.shape) != grid or labels.dtype != torch.int32:
                raise ValueError('labels must be an int32 volume of shape %r' % (grid,))
            radius_vox = radius_voxels(connectivity_radius, env.affine_vox2rasmm)
        if (save_metric_means or metric_connectivity_prefix is not None) != (metrics is not None):
            raise ValueError('a metric output needs metrics, and metrics need a metric output')
        if save_metric_means and fmt != 'trk':
            raise ValueError('.tck files cannot hold per-streamline data: save metric means to a .trk file')
        shifts = []
        if metrics is not None:
            metric_names = [str(m) for m in metric_names]
            if (metrics.dim() != 4 or tuple(metrics.shape[:3]) != grid or metrics.dtype != torch.float32
                    or int(metrics.shape[3]) != len(metric_names)):
                raise ValueError('metrics must be a float32 volume of shape %r + (%d,)' % (grid, len(metric_names)))
            if metric_connectivity_prefix is not None:
                shifts += [metric_shift(b) for b in metrics.abs().amax(dim=(0, 1, 2)).cpu().tolist()]
        if length_connectivity_path is not None:      # kept lengths are <= max_length, up to float32 rounding
            shifts.append(metric_shift(float(self.max_length) * 1.001))
        affine = np.asarray(env.affine_vox2rasmm, dtype=np.float64)
        np.random.shuffle(env.seeds)      # tracker.py:94
        # One process per GPU (torchrun): every rank shuffled the same seed list with the same RNG state;
        # it keeps its contiguous slice, tracks and post-processes it on its own device, and rank 0
        # receives the packed results over NCCL and writes them in rank order -- the order one GPU
        # produces (SURVEY 8(e)).
        world = dist.get_world_size() if dist.is_initialized() else 1
        rank = dist.get_rank() if dist.is_initialized() else 0
        if world > 1:
            # device-drawn noise and policy samples are keyed by the index in the common shuffled list: tell
            # the env where its slice starts, so that every seed gets the draws it gets on one GPU
            env.seed_offset = parallel.shard_bounds(len(env.seeds), rank, world)[0]
            env.seeds = parallel.shard_seeds(env.seeds, rank, world)
        vox_size = np.mean(np.abs(affine)[np.diag_indices(4)][:3])
        lo, hi = self.min_length / vox_size, self.max_length / vox_size
        writer = None
        if rank == 0:
            writer = (TrkWriter(path, dims, voxel_sizes, affine, self.save_seeds, save_scores=save_scores,
                                save_labels=save_labels, metric_names=metric_names if save_metric_means else ())
                      if fmt == 'trk' else TckWriter(path))
        self.alg.agent.eval()
        n_passes = len(list(self._passes(env)))
        if world > 1:       # ranks may differ by one seed: agree on the number of passes
            t = torch.tensor([n_passes], device=env.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            n_passes = int(t.item())
        passes = list(self._passes(env))
        density = endpoints = None
        if density_path is not None:
            density = torch.zeros(grid, dtype=torch.int32, device=env.device)
        if endpoints_path is not None:
            endpoints = torch.zeros(grid, dtype=torch.int32, device=env.device)
        skipped = 0
        matrix = None
        if connectivity_path is not None or weighted:
            K = int(labels.max().item()) + 1
        if connectivity_path is not None:
            matrix = torch.zeros((K, K), dtype=torch.int32, device=env.device)
        sums = counts = unsampled = None
        if weighted:
            sums = torch.zeros((len(shifts), K, K), dtype=torch.int64, device=env.device)
            counts = torch.zeros((len(shifts), K, K), dtype=torch.int32, device=env.device)
        if metrics is not None:
            unsampled = torch.zeros((1,), dtype=torch.int64, device=env.device)
        try:
            for ip in range(n_passes):
                out = torch.zeros((0, 3), dtype=torch.float32, device=env.device)
                new_off = torch.zeros((1,), dtype=torch.int64, device=env.device)
                seeds_kept = np.zeros((0, 3))
                scores_kept = torch.zeros((0,), dtype=torch.float32, device=env.device)
                pairs = torch.zeros((0, 2), dtype=torch.int32, device=env.device)
                means = torch.zeros((0, len(metric_names)), dtype=torch.float32, device=env.device)
                if ip < len(passes) and passes[ip][1] > passes[ip][0]:
                    self._run_pass(env, *passes[ip])
                    pts, offsets = env.get_streamlines_device()
                    lens = lengths_packed(pts, offsets)
                    data, new_off, index = select_packed(pts, offsets, keep=(lens >= lo) & (lens <= hi))
                    if oracle is not None:
                        scores = oracle.predict_device(data, new_off, distributed=False)
                        data, new_off, sel = select_packed(data, new_off, scores=scores, threshold=oracle_threshold)
                        index, scores_kept = index[sel], scores[sel]
                    if density is not None or endpoints is not None:
                        skipped += tract_maps_packed(data, new_off, grid, density, endpoints)
                    if labels is not None:
                        pairs = connectome_packed(data, new_off, labels, matrix, radius_vox,
                                                  pairs=save_labels or weighted)
                    if metrics is not None:
                        means, _ = sample_metrics_packed(data, new_off, metrics)
                        unsampled += torch.isnan(means[:, 0]).sum()
                    if weighted:
                        cols = [means] if metric_connectivity_prefix is not None else []
                        if length_connectivity_path is not None:
                            cols.append((lens[index] * float(vox_size)).to(torch.float32).reshape(-1, 1))
                        connectome_sums_packed(pairs, torch.cat(cols, 1).contiguous(), shifts, sums, counts)
                    if self.compress:     # after the length filter, before the space change (tracker.py:120-129)
                        data, new_off = compress_packed(data, new_off, tol_error=float(self.compress) / float(vox_size))
                    d64 = data.to(torch.float64)
                    if fmt == 'trk':
                        out = ((d64 + 0.5) * float(vox_size)).to(torch.float32)
                    else:                 # s . affine[:3,:3] + affine[:3,3] (tracker.py:133-136), term by term
                        A = affine
                        cols = [d64[:, 0] * A[0, c] + d64[:, 1] * A[1, c] + d64[:, 2] * A[2, c] + A[c, 3]
                                for c in range(3)]
                        out = torch.stack(cols, 1).to(torch.float32)
                    seeds_kept = np.asarray(env.initial_points)[index.cpu().numpy()] - 0.5
                if world > 1:
                    n_kept = int(new_off.shape[0]) - 1
                    merged = parallel.gather_packed(out, new_off[1:] - new_off[:-1], torch.as_tensor(seeds_kept),
                                                    torch.zeros((n_kept,), dtype=torch.int64), copy=False,
                                                    scores=scores_kept if save_scores else None,
                                                    labels=pairs if save_labels else None,
                                                    means=means if save_metric_means else None)
                    if rank == 0 and len(merged) > 0:
                        per = merged.data_per_streamline
                        writer.write(merged.data, merged.offsets, per['seeds'], per.get('oracle_score'),
                                     np.stack((per['start_label'], per['end_label']), 1) if save_labels else None,
                                     per.get('metric_means'))
                    continue
                if int(new_off.shape[0]) <= 1:
                    continue
                h_data = env._pinned('file_pts', out.numel(), torch.float32)
                h_off = env._pinned('file_off', new_off.numel(), torch.int64)
                h_data.copy_(out.reshape(-1), non_blocking=True)
                h_off.copy_(new_off, non_blocking=True)
                torch.cuda.current_stream(env.device).synchronize()
                writer.write(h_data.numpy().reshape(-1, 3), h_off.numpy(), seeds_kept,
                             scores_kept.cpu().numpy() if save_scores else None,
                             pairs.cpu().numpy() if save_labels else None,
                             means.cpu().numpy() if save_metric_means else None)
        finally:
            if writer is not None:
                writer.close()
        self.connectome_unlabelled = self.metrics_unsampled = 0
        if any(m is not None for m in (density, endpoints, matrix, sums, unsampled)):
            skipped = parallel.reduce_maps([density, endpoints, matrix, sums, counts, unsampled], skipped)
            if rank == 0:
                from tracktolearn_b200.io import nifti
                for p, m in ((density_path, density), (endpoints_path, endpoints)):
                    if m is not None:
                        nifti.save(p, m.cpu().numpy(), env.affine_vox2rasmm)
                if matrix is not None:
                    m = matrix.cpu().numpy()
                    np.save(connectivity_path, m)
                    self.connectome_unlabelled = unlabelled_endpoints(m)
                if sums is not None:
                    mean = edge_means(sums, counts, shifts)
                    if metric_connectivity_prefix is not None:
                        for c, name in enumerate(metric_names):
                            np.save(metric_connectivity_prefix + name + '.npy', mean[c])
                    if length_connectivity_path is not None:
                        np.save(length_connectivity_path, mean[-1])
                if unsampled is not None:
                    self.metrics_unsampled = int(unsampled.item())
        self.maps_skipped = skipped
        n = writer.n if writer is not None else 0
        if world > 1:
            t = torch.tensor([n], device=env.device)
            dist.broadcast(t, 0)
            n = int(t.item())
        return n

    def track_and_train(self, env):
        """Reference: tracking/tracker.py:152-202.  One training "epoch": ``n_actor`` streamlines from
        random seeds (``env.nreset``), the rollout + update loop of the algorithm (``alg._episode``:
        sample actions, step, push transitions to the replay buffer, one gradient update per env step),
        then the streamlines it produced.  Returns (tractogram, mean losses, reward, mean reward factors)."""
        from collections import defaultdict
        self.alg.agent.train()
        mean_losses = defaultdict(list)
        mean_reward_factors = defaultdict(list)
        state = env.nreset(self.n_actor)
        reward, losses, length, reward_factors = self.alg._episode(state, env)
        train_tractogram = env.get_streamlines()
        for step_losses in (losses if isinstance(losses, (list, tuple)) else [losses]):
            for k, v in step_losses.items():
                mean_losses[k].append(float(v))
        for k, v in (reward_factors or {}).items():
            mean_reward_factors[k].append(float(v))
        return train_tractogram, mean_losses, reward, mean_reward_factors

    def track_and_validate(self, env):
        """Reference: tracking/tracker.py:204-259 (batch by batch, with rewards)."""
        self.alg.agent.eval()
        tractogram = None
        cummulative_reward = 0
        for start in range(0, len(env.seeds), self.n_actor):
            end = min(start + self.n_actor, len(env.seeds))
            state = env.reset(start, end)
            reward = self.alg.validation_episode(state, env, self.prob, policy_seed=self.policy_seed)
            t = env.get_streamlines()
            if tractogram is None and len(t) > 0:
                tractogram = t
            elif len(t) > 0:
                tractogram += t
            cummulative_reward += reward
        return tractogram, cummulative_reward
