/*
 * ttl_b200.h -- C ABI of libttl_b200.so, the B200 (sm_100a) implementation of the
 * TrackToLearn batched tracking step, SAC actor forward and TractOracle-Net scoring.
 *
 * The reference (levje/TrackToLearn) is pure Python and has no FFI; its boundary for this
 * path is the duck-typed class API of TrackingEnvironment / SACActorCritic /
 * OracleSingleton.  Each entry point below names the reference method(s) it replaces
 * (paths relative to /root/reference/TrackToLearn).  The Python classes in
 * tracktolearn_b200/ keep those names and call these functions through ctypes; a
 * maintainer of the reference would bind them the same way (INTEGRATION.md).
 *
 * Conventions: every pointer is a DEVICE pointer unless the name ends in _host; nothing is
 * allocated or freed behind the caller's back except the opaque plan objects
 * (ttl_actor_plan_*, ttl_oracle_plan_*); every function enqueues work on `stream`
 * (a cudaStream_t passed as void*) and returns 0 or a cudaError_t / negative ttl error;
 * no function synchronises the stream.  There is no CPU fallback.
 */
#ifndef TTL_B200_H
#define TTL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTL_ABI_VERSION 5

/* StoppingFlags, environments/stopping_criteria.py:10-20 */
#define TTL_STOPPING_MASK 1
#define TTL_STOPPING_LENGTH 2
#define TTL_STOPPING_CURVATURE 4
#define TTL_STOPPING_ORACLE 64

#define TTL_OPERAND_BF16 0
#define TTL_OPERAND_FP16 1
#define TTL_OPERAND_TF32 2

#define TTL_ERR_BAD_ARG (-1)
#define TTL_ERR_UNSUPPORTED (-2)
#define TTL_ERR_DRIVER (-3)

/* Subject data resident in HBM (environments/env.py:143-260, load_subject). */
typedef struct ttl_volume {
  const float* sh;         /* [X][Y][Z][CP] fp32 SH coefficients, channel-padded, z fastest */
  int32_t X, Y, Z;         /* SH volume dims */
  int32_t C;               /* real coefficient count (45 for order 8) */
  int32_t CP;              /* padded channel stride in floats, multiple of 4 */
  const double* mask_coef; /* [MX][MY][MZ] f64 cubic B-spline coefficients of the tracking mask
                              (scipy spline_filter output, stopping_criteria.py:58-59) */
  int32_t MX, MY, MZ;
  const float* peaks;      /* [PX][PY][PZ][15] fp32 or NULL (local_reward.py:23-27) */
  int32_t PX, PY, PZ;
} ttl_volume;

/* Tracking parameters (environments/env.py:108-138,196-213). */
typedef struct ttl_params {
  double step_vox;          /* step size in voxels, np.float64 (datasets/utils.py:88-124) */
  double mask_threshold;    /* binary_stopping_threshold */
  double alignment_weighting;
  float theta_rad;          /* float32(deg2rad(theta)), numpy-1.23 comparison precision */
  int32_t max_nb_steps;     /* int(max_length / step_size_mm) */
  int32_t n_dirs;           /* previous directions in the state (100) */
  int32_t dir_f64;          /* 1: NoisyTrackingEnvironment arithmetic (float64 directions,
                               noisy_tracking_env.py:63-77); 0: float32 (TrackingEnvironment) */
  int32_t compute_reward;   /* 1: alignment reward (reward.py:46-79, local_reward.py:29-107) */
  int32_t state_stopped;    /* 1: also build the state rows of streamlines that stop this step
                               (the reference does, tracking_env.py:214-215); 0: skip them */
  int32_t refill;           /* 1: streaming tracker -- slots freed by stopped streamlines are given
                               to the next unseeded rows of the batch in the same step (results per
                               seed are unchanged at prob = 0; excludes state_stopped) */
} ttl_params;

/* Per-batch mutable state in HBM (tracking_env.py:91-133 allocates the equivalent). */
typedef struct ttl_batch {
  int32_t n;               /* streamlines (seeds) in this batch */
  int32_t n_slots;         /* streamlines tracked at once (n_actor); == n without refill */
  int32_t capacity;        /* rows allocated in every per-row buffer */
  int32_t max_pts;         /* points per row = max_nb_steps + 1 */
  int32_t ld_state;        /* floats per state row (>= state size, multiple of 4) */
  int32_t state_size;      /* 7*C + 3*n_dirs (615) */
  float* points;           /* [capacity][max_pts][3] fp32 streamline coordinates (voxel space) */
  int32_t* flags;          /* [capacity] StoppingFlags per global row */
  int32_t* lengths;        /* [capacity] points per global row, set when the row stops */
  int32_t* npts;           /* [capacity] running point count of every row (1 after reset) */
  uint8_t* dones;          /* [capacity] */
  int32_t* alive[2];       /* ping-pong lists of alive global rows, ascending */
  int32_t* ctrl;           /* [16] device ints: [0],[1] alive count of alive[0],alive[1];
                              [2] steps taken; [3] alive count before the last step;
                              [4],[5] int64 streamline-steps so far; [6] next unseeded row;
                              [8] survivors of the last step; [9] rows refilled in the last step;
                              [10] first row refilled in the last step; [12],[13] ping-pong copies of
                              [6] used by the step kernels; others reserved */
  uint8_t* stop;           /* [n_slots+16] per rank (position in the alive list): stopped this step */
  int32_t* dest;           /* [n_slots] per rank: row of state[next] that holds its new state */
  int32_t* step_flags;     /* [n_slots] per rank: flags raised this step */
  float* reward;           /* [n_slots] per rank */
  float* state[2];         /* ping-pong [n_slots][ld_state] fp32 state rows.  state[cur] rows
                              [0, n_alive) are the states of alive[cur] in order. */
  void* state_bf16[2];     /* ping-pong [n_slots][ld_bf16] operand rows: the state rows in the actor's
                              operand type (operand_fmt below; "bf16" in the names is historical),
                              zero padded to ld_bf16 = round_up(state_size, 64) elements, 16-byte
                              aligned: the actor's first-layer TMA operand, written by the same kernel
                              that writes state[] */
  int32_t ld_bf16;
  int32_t max_groups;      /* entries in grp_stops: ceil(n_slots / 32) + 1 */
  int32_t* grp_stops;      /* [max_groups] streamlines stopped this step per group of 32 ranks */
  int32_t* sg_stops;       /* [2][ceil(max_groups / 64)] ping-pong: stops per super-group of 64 groups,
                              accumulated by the stop kernels, consumed and cleared by the state kernel */
  int32_t bf16_layout;     /* column order of state_bf16 rows: 0 = the reference's
                              [7*C | 3*n_dirs | 0..]; 1 = channel-padded [7*CP | 3*n_dirs | 0..]
                              (every neighbourhood point starts on a 16-byte boundary; the actor's
                              first-layer weights are permuted to match, ttl_actor_plan_set_layout).
                              state[] may be NULL with layout 1: the fp32 rows are then not
                              materialised (SURVEY.md section 7, step 7) */
  float* rank_rec[2];      /* ping-pong [n_slots+16][8] fp32 words, one 32-byte record per rank of
                              alive[k]: {row (int bits), points so far (int bits), tip xyz, the point
                              before the tip xyz (zeros when there is none)}.  Written by reset and by
                              the state kernel of every step; the next step reads it instead of
                              chasing alive[] -> npts[] -> points[] (tracking_env.py:181-188 re-slices
                              the streamline buffer for the same purpose) */
  float* step_tip;         /* [n_slots+16][4] per rank of alive[cur]: the point added this step */
  int32_t operand_fmt;     /* element type of state_bf16 rows: TTL_OPERAND_BF16 / _FP16 (2 bytes) or
                              TTL_OPERAND_TF32 (fp32 words rounded to tf32; bf16_layout 1 only).  FP16 rows
                              saturate at +-65504: a state value is a convex combination of SH coefficients
                              or a step vector, so the caller checks the volume's range once */
  const int32_t* order;    /* NULL, or a permutation [n] of the rows: the order in which seeds take slots
                              (slot k of reset gets row order[k]; refills continue from there).  Rows
                              keep their identity -- results, flags and the output order are per row --
                              so this only decides which streamlines sit next to each other in the alive
                              list.  The streaming tracker passes the seeds' voxel raster order: the
                              reference shuffles its seeds (tracker.py:94), which makes every warp of
                              the gather touch unrelated voxels; neighbours in the list then share
                              cache lines.  Must be NULL for the reference protocol (ascending
                              continue_idx, tracking_env.py:123). */
} ttl_batch;

/* ---- one-time / load-time helpers ------------------------------------------------------ */

/* [V][C] -> [V][CP] channel padding (zero fill) of the SH volume (env.py:179-180 uploads the
 * unpadded volume; the padding makes every voxel a whole number of float4). */
int ttl_pad_channels(const float* src, float* dst, int64_t n_voxels, int32_t C, int32_t CP,
                     void* stream);

/* Peak extraction at load time (environments/env.py:405-432, the reference's only SH-to-SF
 * projection): per voxel with a non-zero coefficient sum, SF = sh . basis^T on n_vertices sphere
 * directions (double), values below absolute_threshold zeroed, dipy peak_directions (local maxima over
 * the sphere's edges given as a padded neighbour table [n_vertices][max_degree], -1 = none; relative
 * threshold; min_separation_deg between kept peaks), the first npeaks directions scaled by
 * value / first value -> out_peaks [n_voxels][npeaks * 3] fp32 (zeros elsewhere).
 * sh [n_voxels][ld] fp32 with C <= 64 coefficients; basis [n_vertices][C], vertices [n_vertices][3] f64. */
int ttl_peaks_from_sh(const float* sh, int64_t n_voxels, int32_t C, int32_t ld, const double* basis,
                      const double* vertices, const int32_t* neighbours, int32_t n_vertices,
                      int32_t max_degree, double relative_threshold, double absolute_threshold,
                      double min_separation_deg, int32_t npeaks, float* out_peaks, void* stream);

/* ---- TrackingEnvironment ------------------------------------------------------------------ */

/* TrackingEnvironment.reset / nreset (tracking_env.py:47-133): seeds [n][3] float64 voxel
 * coordinates -> first points, zeroed flags, lengths 1, alive = 0..min(n,n_slots)-1 and the
 * initial state rows in state[0].  After this call cur = 0. */
int ttl_env_reset(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b,
                  const double* seeds, void* stream);

/* Tracking noise drawn inside the step kernel (NoisyTrackingEnvironment with noise_rng = 'device').
 * Row i of the batch, with g = row_base + i and L = its point count before the step (1 on the first
 * step), gets noise_c = sigma * z_c for c = 0, 1, 2, where
 *   (w0, w1, w2, w3) = Philox4x32-10(counter = (lo32(g), hi32(g), L, c), key = (lo32(seed), hi32(seed)))
 *   u1 = (((w1 << 32 | w0) >> 12) + 0.5) * 2^-52,  u2 = (((w3 << 32 | w2) >> 12) + 0.5) * 2^-52
 *   z_c = sqrt(-2 ln u1) * cos(2 pi u2)            (fp64; |z_c| <= 8.58)
 * added in fp64 to the action where ttl_env_step adds its `noise` array.  Each streamline's noise
 * depends only on (seed, g, L, c): not on the alive-list order, the slot count, refill or the process
 * that tracks it, so a run sharded over GPUs (row_base = the shard's first index in the
 * common seed list) produces what one GPU produces.  It is not the reference's RandomState stream.
 * The struct is a host structure read at call time (like ttl_params); a CUDA graph captures its values. */
typedef struct ttl_noise {
  double sigma;            /* N(0, sigma) per component */
  uint64_t seed;           /* Philox key */
  int64_t row_base;        /* global seed index of batch row 0 */
} ttl_noise;

/* The standard normals the step kernels use, for tests: out [n][3] f64, out[k][c] = z_c(nz->seed, g[k],
 * L[k]) for g [n] int64 and L [n] int32 (device arrays); nz->sigma and nz->row_base are ignored. */
int ttl_noise_normals(const ttl_noise* nz, const int64_t* g, const int32_t* L, int32_t n, double* out,
                      void* stream);

/* Stochastic policy sampled on the device (Tracker / validation_episode with prob > 0 and a policy seed).
 * Row i of the batch, with g = row_base + i (row_base as for ttl_noise: seed_offset + start after
 * reset / reset_streaming, 0 after nreset) and L = its point count before the step, takes for c = 0, 1, 2
 *   eps_c = fp32_rn(z(seed, g, L, 3 + c))        z = the ttl_noise normal above, counter words 3..5
 *   mu_c  = head output c     + bias[c]          the actor's fixed summation tree (ttl_step_action)
 *   ls_c  = head output 3 + c + bias[3 + c]
 *   std_c = expf(fminf(fmaxf(ls_c, -20.f), 2.f)) * prob
 *   a_c   = tanhf(fmaf(std_c, eps_c, mu_c))
 * which is the actor's own head arithmetic (MaxEntropyActor.forward, offpolicy.py:94-140) with eps_c in
 * place of torch.randn: the fused route (ttl_env_step with head partials and `pol`) and the actor-then-step
 * route fed by ttl_policy_eps give the same bits.  Counter words 3..5 keep eps independent of the tracking
 * noise (words 0..2) under one seed.  At prob = 0 the action is tanh(mu) bit for bit.  Each streamline's
 * sample depends only on (seed, g, L): not on the slot count, the alive-list order or the GPU count.  It is
 * not torch's random stream.  Host struct read at call time; a CUDA graph captures its values. */
typedef struct ttl_policy {
  uint64_t seed;           /* Philox key */
  int64_t row_base;        /* global seed index of batch row 0 */
  float prob;              /* std scale (Tracker's prob), >= 0 */
  int32_t pad;
} ttl_policy;

/* Where the actions of a step come from: exactly one of `actions` and `head_partial`.  Host structure read
 * at call time.
 * head_partial: the actor's fused head, the pointers ttl_actor_head_partial returns after a forward with
 * action == NULL -- [n_alive][n_tiles][8] fp32 per-column-tile partial sums of the 6-wide output layer
 * (tiles_per_256 = 256 / tile width of the launch that wrote them), head_bias [6].  The sums follow the same
 * fixed tree as the actor's own finishing pass, so this source and ttl_actor_forward* + an action buffer
 * give the same bits whatever the tile width; it saves one launch and the action round trip per step. */
typedef struct ttl_step_action {
  const float* actions;       /* [n_alive][lda] fp32 action buffer, or NULL */
  const float* head_partial;  /* or: fused head partial sums (ttl_actor_head_partial) */
  const float* head_bias;     /* [6], with head_partial */
  int32_t lda;                /* floats per action row, >= 3, with actions */
  int32_t n_tiles, tiles_per_256;
  int32_t pad;
} ttl_step_action;

/* TrackingEnvironment.step (tracking_env.py:135-221; NoisyTrackingEnvironment.step when
 * prm->dir_f64) for the alive rows of alive[cur]: action from `act`, optional noise added first.
 * Normalise+scale (env.py:493-502), first-step flip, grow, stopping flags (env.py:567-603,
 * utils.py:127-173, stopping_criteria.py:38-82), reward, ordered compaction into alive[cur^1] /
 * ctrl[cur^1], new state rows into state[cur^1] (survivors first, in order; then refilled rows if
 * prm->refill, or stopped rows if prm->state_stopped).
 *   noise   [n_alive][3] f64 drawn on the host, or NULL
 *   nz      the noise drawn on the device as described at ttl_noise: no host work, no copy and no extra
 *           launch per step.  prm->dir_f64 must be 1 (the noisy environment's float64 directions), else
 *           TTL_ERR_UNSUPPORTED
 *   pol     the stochastic policy sampled inside the propagate kernel (ttl_policy): head_partial must hold
 *           all six outputs (ttl_actor_forward* with action == NULL and probabilistic != 0)
 *   defer   1: stop before the state rows, so that TractOracle-Net can be consulted in between
 *           (OracleStoppingCriterion, stopping_criteria.py:113-154: stop where the score < 0.5 once the
 *           streamline has more than min_pts_stop points; OracleReward, oracle_reward.py:45-93: `bonus` for
 *           streamlines done this step with more than min_pts_reward points and score > 0.5):
 *             ttl_env_step, defer = 1     propagate + LENGTH/CURVATURE/MASK + alignment reward
 *             ttl_oracle_features_rows    resample(128)+diff of the alive streamlines   \  caller, between
 *             ttl_oracle_forward          scores [n_alive]                              /  the two calls
 *             ttl_env_step_finish         ORACLE flag, bonus, compaction bookkeeping, state rows
 * The combinations served (every other one is TTL_ERR_BAD_ARG):
 *   action from      noise            pol      defer
 *   actions          none / noise     -        0 or 1     the actor's head run on its own (with ttl_policy_eps
 *                    / nz                                 at prob > 0 and a policy seed)
 *   head_partial     none / nz        -        0          tanh(mu), the deterministic policy that tracking uses
 *                                                         (prob = 0: tracker.py:28, ttl_track.py:172-175;
 *                                                         offpolicy.py:126-128 with std * 0)
 *   head_partial     none / nz        pol      0          the stochastic policy
 * `n_upper` >= current alive count bounds the launch (the kernels read the true count from
 * ctrl[cur] on the device, so no host sync is needed between steps).
 * The caller flips cur afterwards: that flip is TrackingEnvironment.harvest (:223-245). */
int ttl_env_step(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                 const ttl_step_action* act, const double* noise, const ttl_noise* nz, const ttl_policy* pol,
                 int32_t defer, int32_t n_upper, void* stream);
int ttl_env_step_finish(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                        const float* scores, int32_t use_stop, int32_t min_pts_stop, int32_t min_pts_reward,
                        float bonus, int32_t n_upper, void* stream);

/* eps [rank][ld] fp32 (ld >= 3) for every rank of alive[cur], in rank order: the draws the fused route
 * makes, for the routes that run the actor's head on its own (ttl_actor_forward* with eps).  (row, L) come
 * from rank_rec[cur], the alive count from ctrl[cur]; ranks beyond it are not written. */
int ttl_policy_eps(const ttl_policy* pol, const ttl_batch* b, int32_t cur, int32_t n_upper, float* eps,
                   int32_t ld, void* stream);

/* state[cur^1][dest[r]] -> out[r] for r < n_rows: the `self.state[self.continue_idx]` that
 * step() returns, in the order of the pre-harvest alive list (tracking_env.py:217-218). */
int ttl_env_gather_step_state(const ttl_batch* b, int32_t cur, int32_t n_rows, float* out,
                              int32_t ld_out, void* stream);

/* _format_state alone (env.py:504-565) for arbitrary streamlines: points [n][L][3] fp32 ->
 * out [n][ld_out].  Used by parity tests and get_state_size. */
int ttl_format_state(const ttl_volume* vol, const ttl_params* prm, const float* points,
                     int32_t n, int32_t L, float* out, int32_t ld_out, void* stream);

/* _compute_stopping_flags alone (env.py:567-603) for arbitrary streamlines [n][L][3]:
 * out_flags [n] int32 (0 = continue). */
int ttl_stopping_flags(const ttl_volume* vol, const ttl_params* prm, const float* points,
                       int32_t n, int32_t L, int32_t* out_flags, double* out_mask_value,
                       float* out_reward, void* stream);

/* get_streamlines (tracking_env.py:247-294): effective lengths (last point dropped when the
 * CURVATURE or MASK bit is set) and their exclusive prefix sum: offsets [n+1] int64. */
int ttl_streamline_offsets(const ttl_batch* b, int64_t* offsets, void* stream);
/* ... then the ragged copy: out_points [offsets[n]][3] fp32. */
int ttl_pack_streamlines(const ttl_batch* b, const int64_t* offsets, float* out_points,
                         void* stream);

/* ---- tractogram output (tracking/tracker.py:118-125) ---------------------------------------- */

/* dipy `length` of n packed streamlines (points [total][3] fp32, offsets [n+1] int64): sum of the
 * segment norms in double -- the quantity tracker.py:120-121 compares with min/max length. */
int ttl_streamline_lengths(const float* points, const int64_t* offsets, int32_t n, double* out_lengths,
                           void* stream);
/* dipy `compress_streamlines(s, tol_error, max_segment_length)` (tracker.py:123-125, --compress) as a
 * per-point keep mask [total] and per-streamline kept-point counts [n]; the caller compacts. */
int ttl_compress_mask(const float* points, const int64_t* offsets, int32_t n, double tol_error,
                      double max_segment_length, uint8_t* keep, int32_t* count, void* stream);
/* Ordered compaction of n packed streamlines (offsets [n+1]): row i is kept when
 * (keep_in == NULL || keep_in[i] != 0) && (scores == NULL || scores[i] >= threshold), compared in
 * fp32; a NaN score is never kept.  Writes, in source order, out_offsets [m+1], out_index [m] (the
 * source row of every kept streamline) and result [2] = {m, out_offsets[m]} on the device, so one
 * small copy tells the host both sizes.  workspace: device, 256-byte aligned,
 * ttl_select_workspace_bytes(n) bytes (0 for n == 0). */
int64_t ttl_select_workspace_bytes(int32_t n);
int ttl_select_streamlines(const int64_t* offsets, int32_t n, const uint8_t* keep_in, const float* scores,
                           float threshold, void* workspace, int64_t workspace_bytes, int64_t* out_offsets,
                           int64_t* out_index, int64_t* result, void* stream);
/* out_points[out_offsets[k] ..] = points[offsets[index[k]] ..] for the m kept streamlines of
 * ttl_select_streamlines: the points copied bit for bit, one warp per streamline. */
int ttl_gather_streamlines(const float* points, const int64_t* offsets, const int64_t* index,
                           const int64_t* out_offsets, int32_t m, float* out_points, void* stream);

/* ---- SAC actor (algorithms/shared/offpolicy.py:61-140, shared/utils.py:41-51) -------------- */

#define TTL_ACTOR_MAX_LAYERS 8
/* Arithmetic of the hidden layers.  The reference runs them as fp32 GEMMs (offpolicy.py:94-140, no
 * autocast).  Relative half-ulp of the operands: bf16 2^-9, fp16 and tf32 2^-12 (11 significant bits);
 * measured output error against the fp32 reference on the 615-1024^3-6 network: bf16 ~4e-3 of the
 * output scale, fp16 / tf32 ~5e-4 (tests/test_actor_gpu.py). */
#define TTL_PRECISION_BF16 0   /* tcgen05 kind::f16, bf16 operands, fp32 TMEM accumulators */
#define TTL_PRECISION_FP32 1   /* CUDA-core fp32 reference-precision path */
#define TTL_PRECISION_FP16 2   /* tcgen05 kind::f16, fp16 operands: bf16's rate, tf32's precision, range
                                  +-65504 (stores saturate and raise ttl_actor_overflow) */
#define TTL_PRECISION_TF32 3   /* tcgen05 kind::tf32, fp32 words rounded to tf32: half the rate, fp32 range */

typedef struct ttl_actor_weights {
  int32_t n_layers;                         /* linear layers (4 for 1024-1024-1024) */
  int32_t in_dim[TTL_ACTOR_MAX_LAYERS];     /* true fan-in  (615,1024,1024,1024) */
  int32_t out_dim[TTL_ACTOR_MAX_LAYERS];    /* true fan-out (1024,1024,1024,6) */
  const float* w[TTL_ACTOR_MAX_LAYERS];     /* [out][in] fp32, nn.Linear layout */
  const float* b[TTL_ACTOR_MAX_LAYERS];     /* [out] fp32 */
} ttl_actor_weights;

typedef struct ttl_actor_plan ttl_actor_plan; /* opaque: packed operand weights, TMA maps, scratch */

/* Host-side: packs weights (operand type of `precision`, K padded to 64, N padded to 64) into
 * `workspace` (device, 1024-byte aligned, ttl_actor_workspace_bytes() bytes) and encodes the TMA
 * descriptors for batches of up to max_rows states.  Enqueues the packing kernels on `stream`. */
int64_t ttl_actor_workspace_bytes(const ttl_actor_weights* w, int32_t max_rows, int32_t precision);
int ttl_actor_plan_create(ttl_actor_plan** out, const ttl_actor_weights* w, int32_t max_rows,
                          int32_t precision, void* workspace, int64_t workspace_bytes, void* stream);
void ttl_actor_plan_destroy(ttl_actor_plan* plan);
int ttl_actor_precision(const ttl_actor_plan* plan);
/* A/B switches of the tensor-core layers (default 0): bit 0 = one launch per layer instead of one
 * persistent launch for the whole network; bits 8.. = pin the N tile to 256 / 128 / 64 (default: chosen
 * per launch from the row count).  Outputs are identical bit for bit in every combination. */
void ttl_actor_options(int32_t bits);
/* The fp32 weights the plan was created from changed in place (an optimiser step,
 * algorithms/sac_auto.py:220-232): repack the operand copies.  A few small launches. */
int ttl_actor_plan_refresh(ttl_actor_plan* plan, void* stream);

/* MaxEntropyActor.forward (offpolicy.py:94-140): state [n][ld_state] fp32 ->
 * action [n][3] = tanh(mu + exp(clamp(log_std,-20,2)) * probabilistic * eps), logp [n]
 * (may be NULL), pre [n][2*action] raw network output (may be NULL), in the plan's precision.
 * n is read from *n_rows_dev when that is non-NULL (no host sync), else n_rows_max.
 * eps [n][3] fp32 may be NULL when probabilistic == 0.  action == NULL (tensor-core tiers with the
 * output layer fused; eps, logp and pre NULL): stop after the last hidden layer, see ttl_actor_head_partial;
 * probabilistic != 0 then keeps the log_std partials too, for the policy ttl_env_step samples (the mu
 * partials are the bits the deterministic call leaves). */
int ttl_actor_forward(ttl_actor_plan* plan, const float* state, int32_t ld_state,
                      const int32_t* n_rows_dev, int32_t n_rows_max, float probabilistic,
                      const float* eps, float* action, float* logp, float* pre, void* stream);
/* Same (tensor-core tiers only) when the caller already holds the zero-padded operand rows that
 * ttl_env_step / ttl_env_reset write (ttl_batch.state_bf16, element type = ttl_batch.operand_fmt,
 * which must be the plan's): state_op [rows_alloc][ld] with ld == round_up(in_dim, 64).  Skips the
 * packing pass. */
int ttl_actor_forward_packed(ttl_actor_plan* plan, const void* state_op, int32_t ld,
                             int32_t rows_alloc, const int32_t* n_rows_dev, int32_t n_rows_max,
                             float probabilistic, const float* eps, float* action, float* logp,
                             float* pre, int32_t layout, void* stream);
/* With action == NULL (and logp == pre == NULL) ttl_actor_forward_packed stops after the last
 * tensor-core layer when the 6-wide output layer is fused into it: the per-tile partial sums of
 * mu / log_std stay in the plan's scratch and this call -- made AFTER the forward, the tile width is
 * chosen per launch -- returns where and in which geometry (see ttl_step_action):
 * partial [rows][n_tiles][8] fp32, tiles_per_256 = 256 / tile width.
 * TTL_ERR_UNSUPPORTED when the plan's output layer is not fused. */
int ttl_actor_head_partial(const ttl_actor_plan* plan, const float** partial, int32_t* n_tiles,
                           int32_t* tiles_per_256, const float** bias);
/* fp16 tier: 1 when a state or activation value was outside +-65504 and was saturated since the last
 * clearing call (synchronises `stream`).  The caller should then re-run in tf32. */
int ttl_actor_overflow(ttl_actor_plan* plan, int32_t* out_host, int32_t clear, void* stream);
/* Prepares the plan for ttl_batch.bf16_layout == 1: packs a copy of the first layer's weights
 * whose columns follow [n_points*CP | rest] (zero columns for the CP - C padding channels). */
int ttl_actor_plan_set_layout(ttl_actor_plan* plan, int32_t C, int32_t CP, int32_t n_points, void* stream);

/* Stand-alone dense layer used by the actor and exposed for tests:
 * C[m][ldc] = act(A[m][k] . W[n][k]^T + bias[n]) with A, W, C in the operand type of `precision`
 * (bf16 / fp16 / tf32-rounded fp32), tcgen05/TMEM/TMA; bn = 0 (auto) or the N tile 256 / 128 / 64.
 * k and n multiples of 64, ldc a multiple of 16, C 32-byte aligned. */
int ttl_gemm_tc(const void* A, const void* W, const float* bias, void* C, int32_t m, int32_t n,
                int32_t k, int32_t ldc, int32_t relu, const int32_t* m_dev, int32_t precision,
                int32_t bn, void* stream);
int ttl_gemm_bf16(const void* A, const void* W, const float* bias, void* C, int32_t m,
                  int32_t n, int32_t k, int32_t ldc, int32_t relu, const int32_t* m_dev,
                  void* stream);

/* ---- TractOracle-Net (oracles/oracle.py:39-89, transformer_oracle.py:77-92) ----------------- */

typedef struct ttl_oracle_weights {
  int32_t n_layers, n_head, d_model, d_ff, n_tokens; /* 4,4,32,2048,128 */
  const float* cls_token;   /* [3] */
  const float* emb_w;       /* [d][3] */
  const float* emb_b;       /* [d] */
  const float* pe;          /* [n_tokens][d] */
  const float* in_proj_w[8];  /* [3d][d] */
  const float* in_proj_b[8];  /* [3d] */
  const float* out_proj_w[8]; /* [d][d] */
  const float* out_proj_b[8]; /* [d] */
  const float* lin1_w[8];     /* [ff][d] */
  const float* lin1_b[8];     /* [ff] */
  const float* lin2_w[8];     /* [d][ff] */
  const float* lin2_b[8];     /* [d] */
  const float* norm1_w[8]; const float* norm1_b[8];
  const float* norm2_w[8]; const float* norm2_b[8];
  const float* head_w;      /* [d] */
  const float* head_b;      /* [1] */
} ttl_oracle_weights;

/* dipy set_number_of_points(s,128) + np.diff (oracle.py:52-54) on device: ragged points
 * [offsets[n]][3] fp32 -> dirs [n][127][3] fp32. */
int ttl_oracle_features(const float* points, const int64_t* offsets, int32_t n, float* dirs,
                        void* stream);
/* Same for the alive streamlines of a tracking batch (rows of alive[cur], npts points each):
 * dirs [n_alive][127][3]. */
int ttl_oracle_features_rows(const ttl_batch* b, int32_t cur, int32_t n_upper, float* dirs, void* stream);
/* TransformerOracle.forward: dirs [n][127][3] -> scores [n] fp32. */
int ttl_oracle_forward(const ttl_oracle_weights* w, const float* dirs, int32_t n, float* scores,
                       void* stream);

/* fp16 tensor-core tier (the reference's CUDA path autocasts to fp16, oracles/oracle.py:9,76):
 * linear1 / linear2 of every encoder layer run on tcgen05 with fp16 operands and fp32 TMEM
 * accumulators; attention, LayerNorm and the embedding stay fp32.  The plan holds fp16 copies of
 * the feed-forward weights in `workspace` (device, 1024-byte aligned,
 * ttl_oracle_workspace_bytes() bytes) and their TMA descriptors. */
typedef struct ttl_oracle_plan ttl_oracle_plan;
int64_t ttl_oracle_workspace_bytes(const ttl_oracle_weights* w);
int ttl_oracle_plan_create(ttl_oracle_plan** out, const ttl_oracle_weights* w, void* workspace,
                           int64_t workspace_bytes, void* stream);
void ttl_oracle_plan_destroy(ttl_oracle_plan* plan);
int ttl_oracle_forward_tc(ttl_oracle_plan* plan, const float* dirs, int32_t n, float* scores,
                          void* stream);

/* ---- introspection ------------------------------------------------------------------------ */
int ttl_abi_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t ttl_launch_count(void);
/* Per-kernel device timing: when enabled every launch is bracketed by CUDA events on its
 * stream; ttl_prof_report waits for them, writes {"kernel": [launches, total_ms], ...} (JSON)
 * into buf_host and clears the record.  Returns the bytes the full report needs. */
void ttl_prof_enable(int32_t on);
/* The kernels of a tracking step (actor layers, propagate/stop, state rows) are launched with the
 * programmatic stream-serialization attribute so that each is set up while its predecessor drains
 * (every one of them waits for its predecessor's completion before its first global access).
 * On by default; 0 switches back to plain stream-ordered launches. */
void ttl_pdl_enable(int32_t on);
int32_t ttl_prof_report(char* buf_host, int32_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* TTL_B200_H */
