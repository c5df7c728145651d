// Batched tracking-environment step for B200 (sm_100a).
//
// Replaces, on the device and without host round trips, what the reference does per step in
// numpy + dwi_ml + scipy (paths relative to /root/reference/TrackToLearn):
//   environments/env.py:493-502        _format_actions  (normalise, scale to the step size)
//   environments/tracking_env.py:165-183  first-step flip and streamline growth
//   environments/env.py:567-603        _compute_stopping_flags
//   environments/utils.py:127-173      is_too_long, is_too_curvy
//   environments/stopping_criteria.py:38-82  cubic B-spline tracking-mask criterion
//   environments/local_reward.py:29-107     peaks alignment reward
//   environments/tracking_env.py:192-202,223-245  continue_idx bookkeeping / harvest
//   environments/env.py:504-565        _format_state (7-point trilinear SH + previous dirs)
//
// Data layout in HBM: SH volume [X][Y][Z][CP] fp32 with the 45 coefficients padded to CP=48
// floats so a voxel is 12 aligned float4 (192 B) and the two z-corners of a trilinear cell
// are one contiguous 384 B run; streamline points [row][max_pts][3] fp32; state rows
// [rank][ld_state=616] fp32 so rows start 16-byte aligned.
//
// Two launches per step, none of which needs the host:
//   propagate_stop  4 lanes per alive streamline (byte/flag work, 64 fp64 spline taps split over the
//                   lanes); each CTA (32 ranks) publishes how many of its ranks stopped, per group and
//                   added into a counter per super-group of 64 groups -- no scan, no waiting
//   build_state     one warp per rank: derives its position in the compacted alive list from the
//                   super-group counters + the group counts of its super-group + a ballot over its
//                   group's stop flags (keeps the reference's ascending continue_idx order), gathers
//                   the 7x8 trilinear corner voxels as LDG.128 straight into registers (duplicates of
//                   the ~26-voxel footprint hit L1) and writes the fp32 row and / or the actor's
//                   operand row (bf16, fp16 or tf32-rounded fp32); one thread of the grid advances the
//                   control block (next alive count, slot refill, counters).
// The kernel boundary is the only synchronisation between the two.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "ttl_common.cuh"
#include "ttl_rng.cuh"

std::atomic<long long> g_ttl_launches{0};

namespace {

constexpr int kGroup = 32;          // ranks per compaction group == rows per propagate_stop CTA
constexpr int kLanesPerRow = 4;     // lanes that share one streamline's 64 spline taps
constexpr int kK1Threads = kGroup * kLanesPerRow;
constexpr int kSuper = 64;          // groups per super-group counter (ttl_batch.sg_stops)
__host__ __device__ __forceinline__ int super_count(int max_groups) { return (max_groups + kSuper - 1) / kSuper; }

// ------------------------------------------------------------------------------------------
// float helpers that refuse FMA contraction, so sums of products round like numpy's
// (no-FMA) einsum loops.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float dot3f(float ax, float ay, float az, float bx, float by, float bz) {
  return __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
}
__device__ __forceinline__ double dot3d(double ax, double ay, double az, double bx, double by,
                                        double bz) {
  return __dadd_rn(__dadd_rn(__dmul_rn(ax, bx), __dmul_rn(ay, by)), __dmul_rn(az, bz));
}

// scipy NI_GeometricTransform tap index reflection for the 'mirror' spline boundary.
__device__ __forceinline__ int mirror_idx(int idx, int n) {
  if (n <= 1) return 0;
  const int s2 = 2 * n - 2;
  if (idx < 0) {
    idx = s2 * (int)(-idx / s2) + idx;
    return idx <= 1 - n ? idx + s2 : -idx;
  }
  if (idx >= n) {
    idx -= s2 * (int)(idx / s2);
    if (idx >= n) idx = s2 - idx;
  }
  return idx;
}

// scipy get_spline_interpolation_weights(order 3)
__device__ __forceinline__ void bspline3(double y, double w[4]) {
  const double z = 1.0 - y;
  w[1] = __ddiv_rn(__dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(y, y), y - 2.0), 3.0), 4.0), 6.0);
  w[2] = __ddiv_rn(__dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(z, z), z - 2.0), 3.0), 4.0), 6.0);
  w[0] = __ddiv_rn(__dmul_rn(__dmul_rn(z, z), z), 6.0);
  w[3] = ((1.0 - w[0]) - w[1]) - w[2];
}

// stopping_criteria.py:79-82: map_coordinates(coef, p - 0.5, order=3, mode='constant',
// cval=0, prefilter=False).  0 for NaN/inf or anything outside [0, n-1].
__device__ double mask_spline_value(const ttl_volume& v, float px, float py, float pz) {
  const double c[3] = {(double)__fsub_rn(px, 0.5f), (double)__fsub_rn(py, 0.5f),
                       (double)__fsub_rn(pz, 0.5f)};
  const int dims[3] = {v.MX, v.MY, v.MZ};
  int start[3];
  double w[3][4];
  bool edge = false;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (!(c[a] >= 0.0 && c[a] <= (double)(dims[a] - 1))) return 0.0;
    const double fl = floor(c[a]);
    start[a] = (int)fl - 1;
    edge |= (start[a] < 0) || (start[a] + 3 >= dims[a]);
    bspline3(c[a] - fl, w[a]);
  }
  int xi[4], yi[4], zi[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    xi[t] = edge ? mirror_idx(start[0] + t, dims[0]) : start[0] + t;
    yi[t] = edge ? mirror_idx(start[1] + t, dims[1]) : start[1] + t;
    zi[t] = edge ? mirror_idx(start[2] + t, dims[2]) : start[2] + t;
  }
  double out = 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double* line = v.mask_coef + ((size_t)xi[i] * v.MY + yi[j]) * v.MZ;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        double t = __ldg(line + zi[k]);
        t = __dmul_rn(t, w[0][i]);
        t = __dmul_rn(t, w[1][j]);
        t = __dmul_rn(t, w[2][k]);
        out = __dadd_rn(out, t);
      }
    }
  }
  return out;
}

__device__ __forceinline__ double shfl_d(unsigned mask, double x, int src) {
  return __shfl_sync(mask, x, src);
}

// The same value computed by the 4 lanes that share a streamline.  The lanes split the work: lane a
// (a < 3) evaluates the four B-spline weights of axis a (6 fp64 divisions each) and broadcasts them,
// lane `sub` multiplies out the 16 taps of x-slab `sub`, then the running sum is handed from lane
// to lane so the 64 additions happen in exactly scipy's order (slab 0 first, z fastest).
// All 4 lanes return the value.
__device__ double mask_spline_value_quad(const ttl_volume& v, float px, float py, float pz, int sub,
                                         unsigned quad_mask, int lane) {
  const double c[3] = {(double)__fsub_rn(px, 0.5f), (double)__fsub_rn(py, 0.5f),
                       (double)__fsub_rn(pz, 0.5f)};
  const int dims[3] = {v.MX, v.MY, v.MZ};
  int start[3];
  double frac[3];
  bool edge = false;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (!(c[a] >= 0.0 && c[a] <= (double)(dims[a] - 1))) return 0.0;   // uniform across the quad
    const double fl = floor(c[a]);
    start[a] = (int)fl - 1;
    edge |= (start[a] < 0) || (start[a] + 3 >= dims[a]);
    frac[a] = c[a] - fl;
  }
  const int quad_base = lane & ~(kLanesPerRow - 1);
  // my axis' weights (lane 3 recomputes axis 2; its copy is not used)
  double wm[4];
  bspline3(sub == 0 ? frac[0] : (sub == 1 ? frac[1] : frac[2]), wm);
  double wx = 0.0, wy[4], wz[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const double x = shfl_d(quad_mask, wm[t], quad_base + 0);
    wx = (sub == t) ? x : wx;
    wy[t] = shfl_d(quad_mask, wm[t], quad_base + 1);
    wz[t] = shfl_d(quad_mask, wm[t], quad_base + 2);
  }
  const int xi = edge ? mirror_idx(start[0] + sub, dims[0]) : start[0] + sub;
  int yi[4], zi[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    yi[t] = edge ? mirror_idx(start[1] + t, dims[1]) : start[1] + t;
    zi[t] = edge ? mirror_idx(start[2] + t, dims[2]) : start[2] + t;
  }
  double prod[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double* line = v.mask_coef + ((size_t)xi * v.MY + yi[j]) * v.MZ;
#pragma unroll
    for (int k = 0; k < 4; ++k) prod[4 * j + k] = __ldg(line + zi[k]);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      double t = prod[4 * j + k];
      t = __dmul_rn(t, wx);
      t = __dmul_rn(t, wy[j]);
      t = __dmul_rn(t, wz[k]);
      prod[4 * j + k] = t;
    }
  }
  double acc = 0.0;
#pragma unroll
  for (int s4 = 0; s4 < 4; ++s4) {
    if (sub == s4) {
#pragma unroll
      for (int t = 0; t < 16; ++t) acc = __dadd_rn(acc, prod[t]);
    }
    acc = shfl_d(quad_mask, acc, quad_base + s4);
  }
  return acc;
}

// utils.py:145-173 on the last three points (fp32, no clipping: NaN compares False).
__device__ __forceinline__ bool too_curvy(const float* p3, float theta_rad) {
  const float ux = __fsub_rn(p3[6], p3[3]), uy = __fsub_rn(p3[7], p3[4]), uz = __fsub_rn(p3[8], p3[5]);
  const float vx = __fsub_rn(p3[3], p3[0]), vy = __fsub_rn(p3[4], p3[1]), vz = __fsub_rn(p3[5], p3[2]);
  const float nu = __fsqrt_rn(dot3f(ux, uy, uz, ux, uy, uz));
  const float nv = __fsqrt_rn(dot3f(vx, vy, vz, vx, vy, vz));
  const float d = dot3f(__fdiv_rn(ux, nu), __fdiv_rn(uy, nu), __fdiv_rn(uz, nu),
                        __fdiv_rn(vx, nv), __fdiv_rn(vy, nv), __fdiv_rn(vz, nv));
  return acosf(d) > theta_rad;
}

// env.py:567-603 in the dict order LENGTH, CURVATURE, MASK (env.py:233-260).
// P = first point of the row, L = number of points.
__device__ int stopping_flags(const ttl_volume& v, const ttl_params& prm, const float* P, int L,
                              double* mask_value_out) {
  int f = 0;
  if (L >= prm.max_nb_steps) f |= TTL_STOPPING_LENGTH;
  if (L >= 3 && too_curvy(P + (size_t)(L - 3) * 3, prm.theta_rad)) f |= TTL_STOPPING_CURVATURE;
  const float* tip = P + (size_t)(L - 1) * 3;
  const double mv = mask_spline_value(v, tip[0], tip[1], tip[2]);
  if (mask_value_out) *mask_value_out = mv;
  if (mv < prm.mask_threshold) f |= TTL_STOPPING_MASK;
  return f;
}

// quad-cooperative version of stopping_flags (same result in all 4 lanes)
__device__ int stopping_flags_quad(const ttl_volume& v, const ttl_params& prm, const float* P, int L, int sub,
                                   unsigned quad_mask, int lane) {
  int f = 0;
  if (L >= prm.max_nb_steps) f |= TTL_STOPPING_LENGTH;
  if (L >= 3 && too_curvy(P + (size_t)(L - 3) * 3, prm.theta_rad)) f |= TTL_STOPPING_CURVATURE;
  const float* tip = P + (size_t)(L - 1) * 3;
  const double mv = mask_spline_value_quad(v, tip[0], tip[1], tip[2], sub, quad_mask, lane);
  if (mv < prm.mask_threshold) f |= TTL_STOPPING_MASK;
  return f;
}

__device__ __forceinline__ float nan_to_num(float x) {
  if (isnan(x)) return 0.f;
  if (isinf(x)) return x > 0 ? 3.4028234663852886e+38f : -3.4028234663852886e+38f;
  return x;
}

// local_reward.py:29-107.  P = row start, L >= 2.
__device__ float alignment_reward(const ttl_volume& v, const float* P, int L) {
  const float* p2 = P + (size_t)(L - 2) * 3;  // streamlines[:, -2]
  const float* p1 = P + (size_t)(L - 1) * 3;
  // .astype(int32) truncates toward zero; interpolation.py:20-23 rounds (no-op) and clips
  int ix = min(max(__float2int_rz(p2[0]), 0), v.PX - 1);
  int iy = min(max(__float2int_rz(p2[1]), 0), v.PY - 1);
  int iz = min(max(__float2int_rz(p2[2]), 0), v.PZ - 1);
  const float* pk = v.peaks + (((size_t)ix * v.PY + iy) * v.PZ + iz) * 15;
  float ux = __fsub_rn(p1[0], p2[0]), uy = __fsub_rn(p1[1], p2[1]), uz = __fsub_rn(p1[2], p2[2]);
  {
    const float n = __fsqrt_rn(dot3f(ux, uy, uz, ux, uy, uz));
    ux = nan_to_num(__fdiv_rn(ux, n));
    uy = nan_to_num(__fdiv_rn(uy, n));
    uz = nan_to_num(__fdiv_rn(uz, n));
  }
  float best = 0.f;
  bool best_nan = false;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    float a = __ldg(pk + 3 * k), b = __ldg(pk + 3 * k + 1), c = __ldg(pk + 3 * k + 2);
    const float n = __fsqrt_rn(dot3f(a, b, c, a, b, c));
    a = nan_to_num(__fdiv_rn(a, n));
    b = nan_to_num(__fdiv_rn(b, n));
    c = nan_to_num(__fdiv_rn(c, n));
    const float d = fabsf(dot3f(a, b, c, ux, uy, uz));
    if (isnan(d)) best_nan = true;   // np.amax propagates NaN
    best = fmaxf(best, d);
  }
  float r = best_nan ? __int_as_float(0x7fc00000) : best;
  if (L >= 3) {
    const float* p3 = P + (size_t)(L - 3) * 3;
    float wx = __fsub_rn(p2[0], p3[0]), wy = __fsub_rn(p2[1], p3[1]), wz = __fsub_rn(p2[2], p3[2]);
    const float n = __fsqrt_rn(dot3f(wx, wy, wz, wx, wy, wz));
    wx = nan_to_num(__fdiv_rn(wx, n));
    wy = nan_to_num(__fdiv_rn(wy, n));
    wz = nan_to_num(__fdiv_rn(wz, n));
    // np.einsum(..., out=float64 factors): the dot product is taken in double
    const double f = dot3d((double)ux, (double)uy, (double)uz, (double)wx, (double)wy, (double)wz);
    r = (float)__dmul_rn((double)r, f);  // rewards(f32) *= factors(f64)
  }
  return r;
}

// Per-rank record of an alive list (ttl_batch.rank_rec): {row, points so far, tip, point before the
// tip (zeros when there is none)}.  One aligned 32-byte load gives a step kernel everything it would
// otherwise chase through alive[] -> npts[] -> points[] (three dependent random loads).
struct RankRec {
  int row, L;
  float tx, ty, tz, px, py, pz;
};
__device__ __forceinline__ void write_rank_rec(float* base, int rank, int row, int L, float tx, float ty,
                                               float tz, float px, float py, float pz) {
  float4* d = reinterpret_cast<float4*>(base) + 2 * (size_t)rank;
  d[0] = make_float4(__int_as_float(row), __int_as_float(L), tx, ty);
  d[1] = make_float4(tz, px, py, pz);
}
__device__ __forceinline__ RankRec read_rank_rec(const float* base, int rank) {
  const float4* d = reinterpret_cast<const float4*>(base) + 2 * (size_t)rank;
  const float4 a = __ldg(d), c = __ldg(d + 1);
  RankRec r;
  r.row = __float_as_int(a.x); r.L = __float_as_int(a.y);
  r.tx = a.z; r.ty = a.w; r.tz = c.x; r.px = c.y; r.py = c.z; r.pz = c.w;
  return r;
}

// ------------------------------------------------------------------------------------------
// K0: reset
// ------------------------------------------------------------------------------------------
__global__ void reset_kernel(ttl_batch b, const double* __restrict__ seeds) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n0 = min(b.n, b.n_slots);
  if (i == 0) {
    b.ctrl[0] = n0;
    b.ctrl[1] = 0;
    b.ctrl[2] = 0;
    b.ctrl[3] = 0;
    b.ctrl[4] = 0;
    b.ctrl[5] = 0;
    b.ctrl[6] = n0;  // next unseeded row
    b.ctrl[7] = 0;
    b.ctrl[8] = 0;
    b.ctrl[9] = 0;
    b.ctrl[10] = 0;
    b.ctrl[12] = n0;  // ping-pong copies of the cursor that the step kernels read / write
    b.ctrl[13] = n0;
    b.ctrl[14] = 0;
  }
  for (int j = i; j < 2 * super_count(b.max_groups); j += gridDim.x * blockDim.x) b.sg_stops[j] = 0;
  if (i < b.n_slots) {
    b.dest[i] = i;
    b.stop[i] = 0;
    b.step_flags[i] = 0;
    b.reward[i] = 0.f;
    if (i < n0) {   // rank i of the first alive list
      const int row = b.order ? b.order[i] : i;
      b.alive[0][i] = row;
      write_rank_rec(b.rank_rec[0], i, row, 1, (float)seeds[3 * row + 0], (float)seeds[3 * row + 1],
                     (float)seeds[3 * row + 2], 0.f, 0.f, 0.f);
    }
  }
  if (i >= b.n) return;
  float* P = b.points + (size_t)i * b.max_pts * 3;
  P[0] = (float)seeds[3 * i + 0];
  P[1] = (float)seeds[3 * i + 1];
  P[2] = (float)seeds[3 * i + 2];
  b.flags[i] = 0;
  b.lengths[i] = 1;
  b.npts[i] = 1;
  b.dones[i] = 0;
}

// Ordered-compaction bookkeeping shared by propagate_stop_kernel and oracle_apply_kernel: every CTA
// (kGroup ranks, kK1Threads threads) publishes how many of its ranks stopped -- per group, and added
// into the counter of its super-group (kSuper groups).  Nothing waits: the state kernel that follows
// turns the counts into positions (survivors_before) and advances the control block, with the kernel
// boundary as the only synchronisation.  `stopped` must be non-zero in exactly one thread per stopped
// rank.  sg_stops holds two sets of counters; set `cur` is used by the step that reads alive[cur] and
// is cleared again by the state kernel of the following step.
__device__ __forceinline__ void publish_stops(const ttl_batch& b, int cur, int stopped) {
  const int grp_stops = __syncthreads_count(stopped);
  if (threadIdx.x == 0) {
    b.grp_stops[blockIdx.x] = grp_stops;
    if (grp_stops) atomicAdd(b.sg_stops + cur * super_count(b.max_groups) + (blockIdx.x / kSuper), grp_stops);
  }
}

// ------------------------------------------------------------------------------------------
// K1: propagate + stopping criteria + reward, one thread per alive streamline
// ------------------------------------------------------------------------------------------
// Where the actions come from.  partial != NULL: straight from the actor's fused head
// (ttl_actor_head_partial): action = tanh(sum_t partial[r][t][0..2] + bias[0..2]), the deterministic
// policy (prob = 0) -- the same additions in the same order as the actor's own head_finish kernel,
// so both routes give the same bits; this one saves a launch and a round trip through HBM.
struct ActionSrc {
  const float* actions;   // [n_alive][lda] fp32
  int lda;
  const float* partial;   // [n_alive][n_tiles][8] fp32 per-n-tile partial sums of the 6-wide head
  int n_tiles;
  int tiles_per_256;      // 256 / (tile width of the launch that wrote the partials)
  const float* bias;      // head bias
  int n_rows;             // rows the launch covers (>= the alive count): bound for speculative loads
};

// Where the noise comes from.  RNG = false: the optional host-drawn array `noise` [n_alive][3] per rank.
// RNG = true (dir_f64 only): drawn here from the counter-based generator (ttl_rng.cuh) at
// (nz.seed, nz.row_base + row, L); lanes 0-2 of the quad draw one component each and share them.
template <bool RNG>
__global__ void __launch_bounds__(kK1Threads, 6) propagate_stop_kernel(
    ttl_volume v, ttl_params prm, ttl_batch b, int cur, ActionSrc src,
    const double* __restrict__ noise, int defer, ttl_noise nz) {
  // 4 lanes per streamline: they redo the cheap scalar work together and split the spline taps
  const int lane = threadIdx.x & 31, sub = threadIdx.x & (kLanesPerRow - 1);
  const unsigned quad_mask = 0xFu << (lane & ~(kLanesPerRow - 1));
  const int r = blockIdx.x * kGroup + (threadIdx.x / kLanesPerRow);
  ttl_grid_dep_wait();     // the actor's last layer (head partials) / the previous step's state kernel
  // Everything this rank needs arrives with independent loads issued together -- alive count, rank
  // record, action (or head partials) -- at a rank clamped into the launch so that the loads need
  // not wait for the count they are checked against.
  const int r_ld = min(r, src.n_rows - 1);
  const RankRec rec = read_rank_rec(b.rank_rec[cur], r_ld);
  float ax = 0.f, ay = 0.f, az = 0.f;
  if (src.partial) {
    ttl_head_tree_sum3(src.partial + (size_t)r_ld * src.n_tiles * 8, src.n_tiles, src.tiles_per_256, ax, ay, az);
  } else {
    ax = src.actions[(size_t)r_ld * src.lda + 0];
    ay = src.actions[(size_t)r_ld * src.lda + 1];
    az = src.actions[(size_t)r_ld * src.lda + 2];
  }
  const int n_alive = b.ctrl[cur];
  int stopped = 0;
  if (r < n_alive) {
  if (src.partial) {
    ax = tanhf(ax + __ldg(src.bias + 0));
    ay = tanhf(ay + __ldg(src.bias + 1));
    az = tanhf(az + __ldg(src.bias + 2));
  }
  const int i = rec.row;
  const int L = rec.L;  // points so far in this row
  float* P = b.points + (size_t)i * b.max_pts * 3;
  const float px = rec.tx, py = rec.ty, pz = rec.tz;

  float qx, qy, qz;  // the new point
  if (prm.dir_f64) {
    // noisy_tracking_env.py:74-77 then env.py:493-502, all float64
    double dx = (double)ax, dy = (double)ay, dz = (double)az;
    const int quad_base = lane & ~(kLanesPerRow - 1);
    if constexpr (RNG) {
      const double za = __dmul_rn(nz.sigma, ttl_noise_normal(nz.seed, nz.row_base + i, L, min(sub, 2)));
      dx = __dadd_rn(dx, __shfl_sync(quad_mask, za, quad_base + 0));
      dy = __dadd_rn(dy, __shfl_sync(quad_mask, za, quad_base + 1));
      dz = __dadd_rn(dz, __shfl_sync(quad_mask, za, quad_base + 2));
    } else if (noise) {
      dx = __dadd_rn(dx, noise[3 * (size_t)r + 0]);
      dy = __dadd_rn(dy, noise[3 * (size_t)r + 1]);
      dz = __dadd_rn(dz, noise[3 * (size_t)r + 2]);
    }
    const double nrm = __dsqrt_rn(dot3d(dx, dy, dz, dx, dy, dz));
    // lane a of the quad scales and adds component a (one fp64 division per lane instead of three)
    const double da = sub == 0 ? dx : (sub == 1 ? dy : dz);
    const double pa = (double)(sub == 0 ? px : (sub == 1 ? py : pz));
    const double sa = __dmul_rn(__ddiv_rn(da, nrm), prm.step_vox);
    const float qa = (float)__dadd_rn(pa, sa);
    qx = __shfl_sync(quad_mask, qa, quad_base + 0);
    qy = __shfl_sync(quad_mask, qa, quad_base + 1);
    qz = __shfl_sync(quad_mask, qa, quad_base + 2);
    if (L == 1) {  // tracking_env.py:165-178: flip if the first step would stop
      const float two[6] = {px, py, pz, qx, qy, qz};
      if (stopping_flags_quad(v, prm, two, 2, sub, quad_mask, lane) != 0) {
        const float fa = (float)__dadd_rn(pa, -sa);
        qx = __shfl_sync(quad_mask, fa, quad_base + 0);
        qy = __shfl_sync(quad_mask, fa, quad_base + 1);
        qz = __shfl_sync(quad_mask, fa, quad_base + 2);
      }
    }
  } else {
    const float stepf = (float)prm.step_vox;
    const float nrm = __fsqrt_rn(dot3f(ax, ay, az, ax, ay, az));
    const float dx = __fmul_rn(__fdiv_rn(ax, nrm), stepf);
    const float dy = __fmul_rn(__fdiv_rn(ay, nrm), stepf);
    const float dz = __fmul_rn(__fdiv_rn(az, nrm), stepf);
    qx = __fadd_rn(px, dx); qy = __fadd_rn(py, dy); qz = __fadd_rn(pz, dz);
    if (L == 1) {
      const float two[6] = {px, py, pz, qx, qy, qz};
      if (stopping_flags_quad(v, prm, two, 2, sub, quad_mask, lane) != 0) {
        qx = __fadd_rn(px, -dx); qy = __fadd_rn(py, -dy); qz = __fadd_rn(pz, -dz);
      }
    }
  }
  // the last three points as this step leaves them (the new one is not in memory yet)
  const int Ln = L + 1;
  float last3[9];
  last3[6] = qx; last3[7] = qy; last3[8] = qz;
  last3[3] = px; last3[4] = py; last3[5] = pz;
  last3[0] = rec.px; last3[1] = rec.py; last3[2] = rec.pz;   // zeros while L < 2
  int f = 0;
  if (Ln >= prm.max_nb_steps) f |= TTL_STOPPING_LENGTH;
  if (Ln >= 3 && too_curvy(last3, prm.theta_rad)) f |= TTL_STOPPING_CURVATURE;
  if (mask_spline_value_quad(v, qx, qy, qz, sub, quad_mask, lane) < prm.mask_threshold) f |= TTL_STOPPING_MASK;
  float rew = 0.f;
  if (prm.compute_reward && v.peaks) {
    // reward.py:63-67: w * f(...) stays float32 (weak python scalar); Ln >= 2 always holds here
    rew = __fmul_rn((float)prm.alignment_weighting,
                    alignment_reward(v, last3 + (Ln >= 3 ? 0 : 3), Ln >= 3 ? 3 : 2));
  }
  if (sub == 0) {
    P[L * 3 + 0] = qx; P[L * 3 + 1] = qy; P[L * 3 + 2] = qz;
    reinterpret_cast<float4*>(b.step_tip)[r] = make_float4(qx, qy, qz, 0.f);
    b.npts[i] = Ln;
    b.step_flags[r] = f;
    b.stop[r] = f != 0;
    stopped = f != 0;
    if (f) {
      b.flags[i] = f;
      b.dones[i] = 1;
      b.lengths[i] = Ln;  // the reference records it in harvest(); nothing reads it in between
    }
    if (prm.compute_reward) b.reward[r] = rew;
  }
  }  // r < n_alive

  if (!(defer & 1)) publish_stops(b, cur, stopped);
}

// ttl_noise_normals: one thread per (row, component)
__global__ void noise_normals_kernel(unsigned long long seed, const long long* __restrict__ g,
                                     const int32_t* __restrict__ L, int n, double* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 3LL * n) return;
  const int k = (int)(t / 3), c = (int)(t % 3);
  out[t] = ttl_noise_normal(seed, g[k], L[k], c);
}

// OracleStoppingCriterion (stopping_criteria.py:113-154) and OracleReward (oracle_reward.py:45-93)
// on top of what propagate_stop_kernel decided: scores [n_alive] are TractOracle-Net's predictions
// for the alive streamlines (including the point just added).  Runs with the K1 geometry (4 threads
// per rank, only thread 0 of each quad works) so it can share the compaction bookkeeping.
__global__ void __launch_bounds__(kK1Threads) oracle_apply_kernel(ttl_params prm, ttl_batch b, int cur,
                                                                 const float* __restrict__ scores,
                                                                 int use_stop, int min_pts_stop,
                                                                 int min_pts_reward, float bonus) {
  const int sub = threadIdx.x & (kLanesPerRow - 1);
  const int r = blockIdx.x * kGroup + (threadIdx.x / kLanesPerRow);
  const int n_alive = b.ctrl[cur];
  int stopped = 0;
  if (r < n_alive && sub == 0) {
    const int i = b.alive[cur][r];
    const int L = b.npts[i];
    int f = b.step_flags[r];
    const float sc = scores[r];
    if (use_stop && L > min_pts_stop && sc < 0.5f) f |= TTL_STOPPING_ORACLE;
    if (f != b.step_flags[r]) {
      b.step_flags[r] = f;
      b.stop[r] = 1;
      b.flags[i] = f;
      b.dones[i] = 1;
      b.lengths[i] = L;
    }
    stopped = f != 0;
    // sparse bonus for streamlines that are done after this step and that the oracle likes
    if (prm.compute_reward && bonus > 0.f && stopped && L > min_pts_reward && sc > 0.5f)
      b.reward[r] = (float)((double)b.reward[r] + (double)bonus);
  }
  publish_stops(b, cur, stopped);
}

// ------------------------------------------------------------------------------------------
// K3: state rows.  One warp per rank of the OLD alive list.
// ------------------------------------------------------------------------------------------
constexpr int kStateWarps = 8;
constexpr int kMaxStateLd = 640;   // floats per state row (>= ld_state)
constexpr int kMaxDirPts = 104;    // n_dirs + 1 points staged (n_dirs <= 103)
constexpr int kMaxCP = 128;        // padded channels per voxel
// per-warp shared memory: 56 weights, 56 voxel ids, staged points, the output row
constexpr int kWarpSmemFloats = 64 + 64 + kMaxDirPts * 3 + kMaxStateLd;
constexpr int kWarpSmemBytes = ((kWarpSmemFloats * 4 + 127) / 128) * 128;
constexpr int kWarpSmemSmall = 512;   // weights + voxel ids only (bf16-only path)

struct TriAxis {  // one axis of one neighbourhood point
  int i0, i1;     // clamped lower / upper lattice index
  float d;        // unclamped fractional part
};

__device__ __forceinline__ TriAxis tri_axis(float c, int n) {
  TriAxis t;
  const float fl = floorf(c);
  t.d = __fsub_rn(c, fl);
  // clamp in float first: NaN -> -1 -> index 0, +-inf and huge values saturate safely
  const float lo = fminf(fmaxf(fl, -1.f), (float)n);
  const int i = (int)lo;
  t.i0 = min(max(i, 0), n - 1);
  t.i1 = min(max(i + 1, 0), n - 1);
  return t;
}

// dwi_ml torch_trilinear_interpolation weights: W = B1^T . Q1 in float32 (polynomial form).
__device__ __forceinline__ void tri_weights(float dx, float dy, float dz, float w[8]) {
  const float xy = dx * dy, yz = dy * dz, xz = dx * dz, xyz = xy * dz;
  w[0] = 1.f - dx - dy - dz + xy + yz + xz - xyz;   // 000
  w[1] = dz - yz - xz + xyz;                        // 001
  w[2] = dy - xy - yz + xyz;                        // 010
  w[3] = yz - xyz;                                  // 011
  w[4] = dx - xy - xz + xyz;                        // 100
  w[5] = xz - xyz;                                  // 101
  w[6] = xy - xyz;                                  // 110
  w[7] = xyz;                                       // 111
}

// volatile: keeps the compiler from sinking the gathers next to their uses (it otherwise
// serialises them to save registers and the kernel loses its memory-level parallelism)
__device__ __forceinline__ float4 ldg_nc_v4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

// phase 0 shared by both paths: lane i (and i+32) owns corner i = 8*p + c of the 7-point
// neighbourhood (order env.py:210-213: 0, +x, +y, +z, -x, -y, -z): voxel index and weight.
__device__ __forceinline__ void corner_table(const ttl_volume& v, const ttl_params& prm, float3 tip,
                                             float* s_w, int* s_vox, int lane) {
  const float tx = tip.x, ty = tip.y, tz = tip.z;
  const float rad = (float)prm.step_vox;  // env.py:207-213, float32 neighbourhood vectors
#pragma unroll
  for (int rep = 0; rep < 2; ++rep) {
    const int i = lane + 32 * rep;
    if (i < 56) {
      const int p = i >> 3, c = i & 7;
      float cx = tx, cy = ty, cz = tz;
      if (p == 1) cx = __fadd_rn(tx, rad);
      if (p == 2) cy = __fadd_rn(ty, rad);
      if (p == 3) cz = __fadd_rn(tz, rad);
      if (p == 4) cx = __fadd_rn(tx, -rad);
      if (p == 5) cy = __fadd_rn(ty, -rad);
      if (p == 6) cz = __fadd_rn(tz, -rad);
      const TriAxis X = tri_axis(cx, v.X), Y = tri_axis(cy, v.Y), Z = tri_axis(cz, v.Z);
      float w[8];
      tri_weights(X.d, Y.d, Z.d, w);
      float wc = w[0];
#pragma unroll
      for (int k = 1; k < 8; ++k) wc = (c == k) ? w[k] : wc;
      const int xi = (c & 4) ? X.i1 : X.i0, yi = (c & 2) ? Y.i1 : Y.i0, zi = (c & 1) ? Z.i1 : Z.i0;
      s_w[i] = wc;
      s_vox[i] = (xi * v.Y + yi) * v.Z + zi;
    }
  }
}

// Builds one state row for the streamline whose points start at P (L points) and writes
//   out_f32 [0, n_f32)   fp32: 7*C SH values | 3*n_dirs previous directions | zero padding
//   out_bf16 [0, n_bf16) the same values rounded to bf16 (actor operand), zero padded
// smem_f: this warp's private staging area (kWarpSmemBytes).  All 32 lanes participate.
// Generic channel count: lane l produces elements l, l+32, ... with scalar gathers.
__device__ void build_state_row_generic(const ttl_volume& v, const ttl_params& prm, const float* P, int L, float3 tip,
                                        float* __restrict__ out_f32, int n_f32,
                                        uint16_t* __restrict__ out_bf16, int n_bf16, float* smem_f,
                                        int lane, int fmt) {
  float* s_w = smem_f;
  int* s_vox = reinterpret_cast<int*>(smem_f + 64);
  float* s_pts = smem_f + 128;
  const int C = v.C, CP = v.CP;
  corner_table(v, prm, tip, s_w, s_vox, lane);
  const int nd = prm.n_dirs;
  const int npts = min(L, nd + 1);
  const float* src = P + (size_t)(L - npts) * 3;
  for (int j = lane; j < npts * 3; j += 32) s_pts[j] = src[j];
  __syncwarp();
  const int S = 7 * C;
  const int n_out = max(n_f32, n_bf16);
  for (int o0 = 0; o0 < n_out; o0 += 32) {
    const int o = o0 + lane;
    float val = 0.f;
    if (o < S) {
      const int p = o / C, ch = o - p * C;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        val = fmaf(s_w[p * 8 + k], __ldg(v.sh + (size_t)s_vox[p * 8 + k] * CP + ch), val);
    } else if (o < S + nd * 3) {
      const int j = o - S;
      const int k = j / 3, c = j - 3 * k;
      if (k < npts - 1) val = __fsub_rn(s_pts[(npts - 1 - k) * 3 + c], s_pts[(npts - 2 - k) * 3 + c]);
    }
    if (out_f32 && o < n_f32) out_f32[o] = val;
    if (out_bf16) {
      const float nxt = __shfl_down_sync(0xffffffffu, val, 1);
      if (!(lane & 1) && o < n_bf16) *reinterpret_cast<uint32_t*>(out_bf16 + o) = ttl_pack16(val, nxt, fmt);
    }
  }
  __syncwarp();
}

// Fast path for the order-8 volume (C = 45 coefficients padded to CP = 48 floats = 12 float4).
// Work item = (neighbourhood point p, float4 chunk ck): 84 items per row, three per lane; each
// item gathers its 8 trilinear corners with LDG.128 straight into registers (8 independent
// 16-byte loads in flight per lane; corners shared between the 7 points hit L1), so a row needs
// only 4.3 KB of shared memory (weights, voxel ids, previous points, the output row) and ~32
// warps fit on an SM.  The finished row leaves through shared memory as 16-byte stores.
// (A cp.async-staged variant that parked all 56 corner voxels in shared memory first was
// measured at 172 us/step at 50 000 rows: 12.5 KB/warp capped the SM at 16 warps.)
__device__ void build_state_row_c45(const ttl_volume& v, const ttl_params& prm, const float* P, int L, float3 tip,
                                    float* __restrict__ out_f32, int n_f32,
                                    uint16_t* __restrict__ out_bf16, int n_bf16, float* smem_f, int lane, int fmt) {
  constexpr int C = 45, CP4 = 12, S = 7 * C;
  float* s_w = smem_f;                                  // [56] trilinear weights
  int* s_vox = reinterpret_cast<int*>(smem_f + 64);     // [56] voxel index
  float* s_pts = smem_f + 128;                          // [(n_dirs+1)*3]
  float* s_row = smem_f + 128 + kMaxDirPts * 3;         // [640] output row
  corner_table(v, prm, tip, s_w, s_vox, lane);
  const int nd = prm.n_dirs;
  const int npts = min(L, nd + 1);
  const float* src = P + (size_t)(L - npts) * 3;
  for (int j = lane; j < npts * 3; j += 32) s_pts[j] = src[j];
  __syncwarp();

  const float4* vol4 = reinterpret_cast<const float4*>(v.sh);
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const int item = lane + 32 * t;
    if (item < 7 * CP4) {
      const int p = item / CP4, ck = item - p * CP4;
      const int4 v0 = *reinterpret_cast<const int4*>(s_vox + p * 8);
      const int4 v1 = *reinterpret_cast<const int4*>(s_vox + p * 8 + 4);
      const int vx[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
      float4 a[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] = __ldg(vol4 + (size_t)vx[k] * CP4 + ck);
      const float4 w0 = *reinterpret_cast<const float4*>(s_w + p * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(s_w + p * 8 + 4);
      const float wk[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        acc.x = fmaf(wk[k], a[k].x, acc.x);
        acc.y = fmaf(wk[k], a[k].y, acc.y);
        acc.z = fmaf(wk[k], a[k].z, acc.z);
        acc.w = fmaf(wk[k], a[k].w, acc.w);
      }
      float* o = s_row + p * C + ck * 4;
      o[0] = acc.x;                          // channel 44 is the only valid one of chunk 11
      if (ck < CP4 - 1) { o[1] = acc.y; o[2] = acc.z; o[3] = acc.w; }
    }
  }
  // previous directions, newest first, zero padded (env.py:549-563), then the row padding
  for (int j = lane; j < nd * 3; j += 32) {
    const int k = j / 3, c = j - 3 * k;
    float val = 0.f;
    if (k < npts - 1) val = __fsub_rn(s_pts[(npts - 1 - k) * 3 + c], s_pts[(npts - 2 - k) * 3 + c]);
    s_row[S + j] = val;
  }
  const int n_pad = max(n_f32, n_bf16);
  for (int j = S + nd * 3 + lane; j < n_pad; j += 32) s_row[j] = 0.f;
  __syncwarp();

  // copy-out
  if (out_f32) {
    if (((n_f32 & 3) == 0) && ((reinterpret_cast<uintptr_t>(out_f32) & 15) == 0)) {
      const float4* s4 = reinterpret_cast<const float4*>(s_row);
      float4* d4 = reinterpret_cast<float4*>(out_f32);
      for (int q = lane; q < (n_f32 >> 2); q += 32) d4[q] = s4[q];
    } else {
      for (int q = lane; q < n_f32; q += 32) out_f32[q] = s_row[q];
    }
  }
  if (out_bf16) {
    uint4* d8 = reinterpret_cast<uint4*>(out_bf16);     // rows are 128-byte aligned (ld multiple of 64)
    for (int q = lane; q < (n_bf16 >> 3); q += 32) {
      const float4 a = *reinterpret_cast<const float4*>(s_row + 8 * q);
      const float4 c = *reinterpret_cast<const float4*>(s_row + 8 * q + 4);
      d8[q] = make_uint4(ttl_pack16(a.x, a.y, fmt), ttl_pack16(a.z, a.w, fmt), ttl_pack16(c.x, c.y, fmt),
                         ttl_pack16(c.z, c.w, fmt));
    }
  }
  __syncwarp();
}

// Direction block of a device-mode row (columns 336..639 of the operand row): the previous row's
// block moved back by one direction with the newest one in front -- for the 16-bit formats a 6-byte
// shift of 600 bytes instead of re-reading 101 fp32 points and redoing 300 subtractions (each value
// was rounded when it was the newest; copying it is the same as recomputing it).  A fresh streamline
// (L == 1) has no directions.  n_dirs == 100, 304 columns.  FMT: TTL_OPERAND_*.
template <int FMT>
__device__ __forceinline__ void write_dirs_shifted(const uint8_t* __restrict__ old_dirs, uint8_t* __restrict__ out_dirs,
                                                   int L, float3 tip, float3 prev_tip, int lane) {
  const uint4* o4 = reinterpret_cast<const uint4*>(old_dirs);
  uint4* d4 = reinterpret_cast<uint4*>(out_dirs);
  const float dxf = __fsub_rn(tip.x, prev_tip.x), dyf = __fsub_rn(tip.y, prev_tip.y),
              dzf = __fsub_rn(tip.z, prev_tip.z);
  if (FMT == TTL_OPERAND_TF32) {
    // 304 fp32 words = 76 quads; out[j] = old[j - 3]
#pragma unroll
    for (int it = 0; it < 3; ++it) {
      const int q = lane + 32 * it;
      if (q < 76) {
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (L > 1 && q < 75) {
          const uint4 cur4 = __ldg(o4 + q);
          if (q > 0) {
            const uint4 prv4 = __ldg(o4 + q - 1);
            o.x = prv4.y; o.y = prv4.z; o.z = prv4.w;
          } else {
            o.x = ttl_round_tf32(dxf); o.y = ttl_round_tf32(dyf); o.z = ttl_round_tf32(dzf);
          }
          o.w = cur4.x;
        }
        d4[q] = o;
      }
    }
    return;
  }
  const uint32_t w_xy = ttl_pack16(dxf, dyf, FMT), w_z = ttl_pack16(dzf, 0.f, FMT);
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int q = lane + 32 * it;
    if (q < 38) {
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (L > 1) {
        const uint4 cur4 = __ldg(o4 + q);
        const uint4 prv4 = q > 0 ? __ldg(o4 + q - 1) : make_uint4(0u, 0u, 0u, 0u);
        o.x = __byte_perm(prv4.z, prv4.w, 0x5432);
        o.y = __byte_perm(prv4.w, cur4.x, 0x5432);
        o.z = __byte_perm(cur4.x, cur4.y, 0x5432);
        o.w = __byte_perm(cur4.y, cur4.z, 0x5432);
        if (q == 0) { o.x = w_xy; o.y = (w_z & 0xffffu) | (cur4.x << 16); }
        if (q == 37) { o.z = 0u; o.w = 0u; }     // columns 300..303: row padding
      }
      d4[q] = o;
    }
  }
}

// Operand-only fast path (ttl_batch.bf16_layout == 1, no fp32 row): the state is produced straight
// as the actor's first-layer operand in the element type FMT (bf16 / fp16: 2 bytes; tf32: fp32 words
// rounded to tf32).  Point p owns columns [48p, 48p+48) so every (point, chunk) work item converts its
// float4 and stores 8 (16) aligned bytes from registers; previous directions follow at column 336.
// No row staging: 512 B of shared memory per warp.  fp16 range: a trilinear value is a convex combination
// of coefficients and a direction is at most a step long, so the host checks max |coefficient| <= 65504
// once per volume instead of every kernel checking every value (tracking_env.py, _start).
template <int FMT>
__device__ void build_state_row_c45_op(const ttl_volume& v, const ttl_params& prm, const float* P, int L, float3 tip,
                                       void* __restrict__ out_v, int n_op, float* smem_f, int lane,
                                       const uint8_t* __restrict__ old_dirs = nullptr,
                                       float3 prev_tip = make_float3(0.f, 0.f, 0.f)) {
  constexpr int CP = 48, CP4 = 12, S = 7 * CP;
  constexpr int ES = FMT == TTL_OPERAND_TF32 ? 4 : 2;
  uint8_t* out = static_cast<uint8_t*>(out_v);
  float* s_w = smem_f;
  int* s_vox = reinterpret_cast<int*>(smem_f + 64);
  corner_table(v, prm, tip, s_w, s_vox, lane);
  __syncwarp();
  const float4* vol4 = reinterpret_cast<const float4*>(v.sh);
  // all 24 gathers of this lane's three work items are issued before the first is consumed
  float4 a[3][8];
  int pp[3], cc[3];
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const int item = min(lane + 32 * t, 7 * CP4 - 1);
    const int p = item / CP4, ck = item - p * CP4;
    pp[t] = p;
    cc[t] = ck;
    const int4 v0 = *reinterpret_cast<const int4*>(s_vox + p * 8);
    const int4 v1 = *reinterpret_cast<const int4*>(s_vox + p * 8 + 4);
    const int vx[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) a[t][k] = ldg_nc_v4(vol4 + (size_t)vx[k] * CP4 + ck);
  }
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const int p = pp[t], ck = cc[t];
    const float4 w0 = *reinterpret_cast<const float4*>(s_w + p * 8);
    const float4 w1 = *reinterpret_cast<const float4*>(s_w + p * 8 + 4);
    const float wk[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      acc.x = fmaf(wk[k], a[t][k].x, acc.x);
      acc.y = fmaf(wk[k], a[t][k].y, acc.y);
      acc.z = fmaf(wk[k], a[t][k].z, acc.z);
      acc.w = fmaf(wk[k], a[t][k].w, acc.w);
    }
    // the volume's padding channels are zero, so columns 45..47 of every point come out zero
    // (NaN weights excepted, and those columns meet zero weights in the actor anyway)
    if (lane + 32 * t < 7 * CP4) {
      uint8_t* d = out + (size_t)(p * CP + ck * 4) * ES;
      if (FMT == TTL_OPERAND_TF32) {
        *reinterpret_cast<uint4*>(d) = make_uint4(ttl_round_tf32(acc.x), ttl_round_tf32(acc.y),
                                                  ttl_round_tf32(acc.z), ttl_round_tf32(acc.w));
      } else {
        *reinterpret_cast<uint2*>(d) = make_uint2(ttl_pack16(acc.x, acc.y, FMT), ttl_pack16(acc.z, acc.w, FMT));
      }
    }
  }
  // previous directions, newest first, zero padded (env.py:549-563)
  const int nd3 = prm.n_dirs * 3;
  if (old_dirs != nullptr && nd3 == 300 && n_op - S == 304) {
    write_dirs_shifted<FMT>(old_dirs, out + (size_t)S * ES, L, tip, prev_tip, lane);
    return;
  }
  const float* last = P + (size_t)(L - 1) * 3;   // element j = last[c - 3k] - last[c - 3k - 3]
  for (int j = 2 * lane; j < n_op - S; j += 64) {
    float val[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int jj = j + e;
      const int k = jj / 3, c = jj - 3 * k;
      val[e] = 0.f;
      if (jj < nd3 && k < L - 1) val[e] = __fsub_rn(__ldg(last + c - 3 * k), __ldg(last + c - 3 * k - 3));
    }
    if (FMT == TTL_OPERAND_TF32)
      *reinterpret_cast<uint2*>(out + (size_t)(S + j) * 4) = make_uint2(ttl_round_tf32(val[0]), ttl_round_tf32(val[1]));
    else
      *reinterpret_cast<uint32_t*>(out + (size_t)(S + j) * 2) = ttl_pack16(val[0], val[1], FMT);
  }
}

// tip = P[L-1] (passed by value so a caller that already holds it skips the dependent load)
__device__ __forceinline__ void build_state_row(const ttl_volume& v, const ttl_params& prm, const float* P,
                                                int L, float3 tip, float* __restrict__ out_f32, int n_f32,
                                                void* __restrict__ out_op, int n_op,
                                                float* smem_f, int lane, int layout = 0, int fmt = 0) {
  if (layout == 1) {   // host guarantees C == 45, CP == 48, no fp32 row
    if (fmt == TTL_OPERAND_TF32) build_state_row_c45_op<TTL_OPERAND_TF32>(v, prm, P, L, tip, out_op, n_op, smem_f, lane);
    else if (fmt == TTL_OPERAND_FP16) build_state_row_c45_op<TTL_OPERAND_FP16>(v, prm, P, L, tip, out_op, n_op, smem_f, lane);
    else build_state_row_c45_op<TTL_OPERAND_BF16>(v, prm, P, L, tip, out_op, n_op, smem_f, lane);
    return;
  }
  uint16_t* o16 = static_cast<uint16_t*>(out_op);   // layout 0 carries a 16-bit copy only (check_layout)
  if (v.C == 45 && v.CP == 48 && max(n_f32, n_op) <= kMaxStateLd)
    build_state_row_c45(v, prm, P, L, tip, out_f32, n_f32, o16, n_op, smem_f, lane, fmt);
  else
    build_state_row_generic(v, prm, P, L, tip, out_f32, n_f32, o16, n_op, smem_f, lane, fmt);
}

// Position bookkeeping of the state kernel, per warp, from what the stop kernels published:
//   stops before rank r = sum of the super-group counters before r's super-group
//                       + sum of the group counts of r's super-group before r's group
//                       + stopped ranks of r's own group before r (ballot over the stop flags);
//   total stops         = sum of all super-group counters.
// Every address depends on r alone (counters beyond the alive range are zero, buffers are padded past
// n_slots), so the loads are issued at kernel entry together with the alive count they are later masked
// with -- one memory round trip, not two -- and reduced with two REDUX instructions.
struct CompactionLoads {
  int sg[2];        // this lane's super-group counters (lane, lane + 32)
  int grp[kSuper / 32];
  int stop_lane;    // stop flag of rank base + lane
};
struct Compaction {
  int keep_before;   // survivors among the ranks before r
  int total_keep;    // survivors of the whole list
};
__device__ __forceinline__ CompactionLoads compaction_loads(const ttl_batch& b, int cur, int r, int lane) {
  const int g = r / kGroup, base = g * kGroup, sgr = g / kSuper;
  const int n_super_max = super_count(b.max_groups);
  const int* sg = b.sg_stops + cur * n_super_max;
  CompactionLoads L;
#pragma unroll
  for (int j = 0; j < 2; ++j) L.sg[j] = lane + 32 * j < n_super_max ? __ldcg(sg + lane + 32 * j) : 0;
#pragma unroll
  for (int j = 0; j < kSuper / 32; ++j) {
    const int gg = sgr * kSuper + lane + 32 * j;
    L.grp[j] = gg < g ? __ldcg(b.grp_stops + gg) : 0;
  }
  L.stop_lane = b.stop[base + lane];
  return L;
}
__device__ __forceinline__ Compaction survivors_before(const ttl_batch& b, const CompactionLoads& L, int cur, int r,
                                                       int n_old, int lane) {
  const int g = r / kGroup, base = g * kGroup, pos = r - base, sgr = g / kSuper;
  const int n_super_max = super_count(b.max_groups);
  int total = L.sg[0] + L.sg[1];
  int before = (lane < sgr ? L.sg[0] : 0) + (lane + 32 < sgr ? L.sg[1] : 0);
  if (n_super_max > 64) {               // more than 131 072 slots: the remaining counters, the slow way
    const int* sg = b.sg_stops + cur * n_super_max;
    for (int j = lane + 64; j < n_super_max; j += 32) {
      const int v = __ldcg(sg + j);
      total += v;
      before += j < sgr ? v : 0;
    }
  }
#pragma unroll
  for (int j = 0; j < kSuper / 32; ++j) before += L.grp[j];
  before += (lane < pos && base + lane < n_old && L.stop_lane != 0) ? 1 : 0;
  Compaction c;
  c.keep_before = r - (int)__reduce_add_sync(0xffffffffu, (unsigned)before);      // REDUX: one instruction each
  c.total_keep = n_old - (int)__reduce_add_sync(0xffffffffu, (unsigned)total);
  return c;
}

// FAST = 1: the operand-only device mode (ttl_batch.bf16_layout == 1) compiled on its own for 6 CTAs per
// SM, which caps it at 40 registers: ptxas spills a few dozen bytes per thread to fit (`-Xptxas -v`), and
// launch_state_fmt records why 6 is still the fastest.  FAST = 0: every other layout, without a register
// cap.  FMT: element type of the operand rows in the operand-only mode.  early_release: release the
// dependent launch before this kernel's work (PDL on), see below.
template <int FAST, int FMT>
__global__ void __launch_bounds__(kStateWarps * 32, FAST ? 6 : 1) build_state_kernel(ttl_volume v, ttl_params prm,
                                                                                     ttl_batch b, int cur, int warp_smem,
                                                                                     int early_release) {
  extern __shared__ __align__(128) uint8_t smem_dyn[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* smem_f = reinterpret_cast<float*>(smem_dyn + (size_t)warp * warp_smem);
  const int r = blockIdx.x * kStateWarps + warp;
  ttl_grid_dep_wait();     // propagate_stop / oracle_apply: flags, new points, stop counts
  // Release the dependent (the actor's first layer) now: once the last wave of this grid is running,
  // its CTAs take over SMs as they drain and set up barriers / tensor memory / descriptors there.
  // Measured on B200 (50 000 rows): 316 -> 312 us per step.  The same early release in the dense
  // kernels and in propagate_stop was measured slower (up to +38 us with all of them on), so those
  // release at exit.
  if (early_release) ttl_grid_dep_launch();
  // independent loads first, all of them addressed by r alone (buffers are padded past n_slots): alive count
  // and cursor, stop counts / flags, this rank's record and new point
  const int n_old = b.ctrl[cur];
  const int cursor = b.ctrl[12 + cur];
  const CompactionLoads cl = compaction_loads(b, cur, r, lane);
  const RankRec rec = read_rank_rec(b.rank_rec[cur], r);
  const float4 q = __ldg(reinterpret_cast<const float4*>(b.step_tip) + r);
  const int stop_r = b.stop[r];
  const Compaction cp = survivors_before(b, cl, cur, r, n_old, lane);
  const int total_keep = cp.total_keep;
  const int n_new = prm.refill ? max(0, min(b.n_slots - total_keep, b.n - cursor)) : 0;
  if (r == 0 && lane == 0) {
    // one thread of the grid advances the control block (what the reference's harvest() does on the
    // host, tracking_env.py:223-245).  Every value it overwrites is either unused by this kernel or
    // read by it from the other ping-pong slot.
    b.ctrl[cur ^ 1] = total_keep + n_new;   // alive count of the next list
    b.ctrl[2] = b.ctrl[2] + 1;
    b.ctrl[3] = n_old;
    b.ctrl[6] = cursor + n_new;
    b.ctrl[12 + (cur ^ 1)] = cursor + n_new;
    b.ctrl[8] = total_keep;
    b.ctrl[9] = n_new;
    b.ctrl[10] = cursor;
    long long* total = reinterpret_cast<long long*>(b.ctrl + 4);
    *total += n_old;
    int* sg_next = b.sg_stops + (cur ^ 1) * super_count(b.max_groups);
    for (int j = 0; j < super_count(b.max_groups); ++j) sg_next[j] = 0;
  }
  if (r >= n_old) return;
  const int keep_before = cp.keep_before;
  const bool stopped = stop_r != 0;
  int row, dst, L;
  float3 tip = make_float3(q.x, q.y, q.z);
  if (!stopped) {
    row = rec.row;
    dst = keep_before;
    L = rec.L + 1;
    if (lane == 0) {
      b.alive[cur ^ 1][dst] = row;
      b.dest[r] = dst;
      write_rank_rec(b.rank_rec[cur ^ 1], dst, row, L, q.x, q.y, q.z, rec.tx, rec.ty, rec.tz);
    }
  } else {
    const int j = r - keep_before;        // how many stopped before this rank
    dst = total_keep + j;
    if (lane == 0) b.dest[r] = dst;
    if (j < n_new) {                      // streaming refill: this freed slot takes a fresh seed
      row = b.order ? b.order[cursor + j] : cursor + j;
      L = 1;
      const float* S = b.points + (size_t)row * b.max_pts * 3;
      tip = make_float3(S[0], S[1], S[2]);
      if (lane == 0) {
        b.alive[cur ^ 1][dst] = row;
        write_rank_rec(b.rank_rec[cur ^ 1], dst, row, 1, tip.x, tip.y, tip.z, 0.f, 0.f, 0.f);
      }
    } else if (prm.state_stopped) {       // parity mode: state of the streamline that just stopped
      row = rec.row;
      L = rec.L + 1;
    } else {
      return;
    }
  }
  const float* P = b.points + (size_t)row * b.max_pts * 3;
  uint8_t* op_next = static_cast<uint8_t*>(b.state_bf16[cur ^ 1]);
  const int op_es = b.operand_fmt == TTL_OPERAND_TF32 ? 4 : 2;
  void* o16 = op_next ? op_next + (size_t)dst * b.ld_bf16 * op_es : nullptr;
  float* o32 = b.state[cur ^ 1] ? b.state[cur ^ 1] + (size_t)dst * b.ld_state : nullptr;
  if (FAST) {
    // survivors (and, in parity mode, rows that just stopped) extend the direction block of the row
    // the actor has just read; a refilled slot starts from zeros (L == 1)
    const uint8_t* old_dirs = static_cast<const uint8_t*>(b.state_bf16[cur]) +
                              ((size_t)r * b.ld_bf16 + 7 * 48) * (FMT == TTL_OPERAND_TF32 ? 4 : 2);
    const float3 prev_tip = make_float3(rec.tx, rec.ty, rec.tz);
    build_state_row_c45_op<FMT>(v, prm, P, L, tip, o16, b.ld_bf16, smem_f, lane, old_dirs, prev_tip);
  }
  else
    build_state_row(v, prm, P, L, tip, o32, b.ld_state, o16, b.ld_bf16, smem_f, lane, b.bf16_layout, b.operand_fmt);
}

// reset: alive[0] = identity, state goes to state[0]
__global__ void __launch_bounds__(kStateWarps * 32) reset_state_kernel(ttl_volume v, ttl_params prm,
                                                                       ttl_batch b, int warp_smem) {
  extern __shared__ __align__(128) uint8_t smem_dyn[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* smem_f = reinterpret_cast<float*>(smem_dyn + (size_t)warp * warp_smem);
  const int r = blockIdx.x * kStateWarps + warp;
  if (r >= min(b.n, b.n_slots)) return;
  const int row = b.order ? b.order[r] : r;
  const float* P = b.points + (size_t)row * b.max_pts * 3;
  const int op_es = b.operand_fmt == TTL_OPERAND_TF32 ? 4 : 2;
  void* o16 = b.state_bf16[0] ? static_cast<uint8_t*>(b.state_bf16[0]) + (size_t)r * b.ld_bf16 * op_es : nullptr;
  float* o32 = b.state[0] ? b.state[0] + (size_t)r * b.ld_state : nullptr;
  build_state_row(v, prm, P, 1, make_float3(P[0], P[1], P[2]), o32, b.ld_state, o16, b.ld_bf16, smem_f, lane,
                  b.bf16_layout, b.operand_fmt);
}

// stand-alone _format_state for arbitrary streamlines [n][L][3]
__global__ void __launch_bounds__(kStateWarps * 32) format_state_kernel(ttl_volume v, ttl_params prm,
                                                                        const float* points, int n,
                                                                        int L, float* out, int ld_out) {
  extern __shared__ __align__(128) uint8_t smem_dyn[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* smem_f = reinterpret_cast<float*>(smem_dyn + (size_t)warp * kWarpSmemBytes);
  const int r = blockIdx.x * kStateWarps + warp;
  if (r >= n) return;
  const int S = 7 * v.C + 3 * prm.n_dirs;
  const float* P = points + (size_t)r * L * 3;
  const float* T = P + (size_t)(L - 1) * 3;
  build_state_row(v, prm, P, L, make_float3(T[0], T[1], T[2]), out + (size_t)r * ld_out, S, nullptr, 0, smem_f, lane);
}

__global__ void stopping_flags_kernel(ttl_volume v, ttl_params prm, const float* points, int n, int L,
                                      int* out_flags, double* out_mask, float* out_reward) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float* P = points + (size_t)r * L * 3;
  double mv;
  out_flags[r] = stopping_flags(v, prm, P, L, &mv);
  if (out_mask) out_mask[r] = mv;
  if (out_reward) {
    float rew = 1.f;  // local_reward.py:46-48: fewer than 2 points -> ones
    if (L >= 2 && v.peaks) rew = alignment_reward(v, P, L);
    out_reward[r] = rew;
  }
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ src,
                                                          const int* __restrict__ dest, int n,
                                                          int ld_src, float* __restrict__ out,
                                                          int ld_out, int width) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const float* s = src + (size_t)dest[warp] * ld_src;
  float* o = out + (size_t)warp * ld_out;
  for (int j = lane; j < width; j += 32) o[j] = s[j];
}

__global__ void pad_channels_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                    long long n_voxels, int C, int CP) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = n_voxels * CP;
  if (t >= total) return;
  const long long vx = t / CP;
  const int c = (int)(t - vx * CP);
  dst[t] = c < C ? src[vx * C + c] : 0.f;
}

// ------------------------------------------------------------------------------------------
// get_streamlines: effective lengths -> exclusive scan -> ragged copy
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) offsets_kernel(ttl_batch b, long long* offsets) {
  __shared__ long long s_sum[1024];
  const int n = b.n, tid = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int beg = min(n, tid * per), end = min(n, beg + per);
  long long acc = 0;
  for (int i = beg; i < end; ++i) {
    const int cut = (b.flags[i] & (TTL_STOPPING_CURVATURE | TTL_STOPPING_MASK)) ? 1 : 0;
    acc += b.lengths[i] - cut;
  }
  s_sum[tid] = acc;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    long long a = 0;
    if (tid >= off) a = s_sum[tid - off];
    __syncthreads();
    s_sum[tid] += a;
    __syncthreads();
  }
  long long pos = s_sum[tid] - acc;
  for (int i = beg; i < end; ++i) {
    offsets[i] = pos;
    const int cut = (b.flags[i] & (TTL_STOPPING_CURVATURE | TTL_STOPPING_MASK)) ? 1 : 0;
    pos += b.lengths[i] - cut;
  }
  if (tid == 1023) offsets[n] = s_sum[1023];
}

__global__ void __launch_bounds__(256) pack_kernel(ttl_batch b, const long long* __restrict__ offsets,
                                                   float* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= b.n) return;
  const long long o = offsets[warp];
  const int len = (int)(offsets[warp + 1] - o);
  const float* s = b.points + (size_t)warp * b.max_pts * 3;
  float* d = out + o * 3;
  for (int j = lane; j < len * 3; j += 32) d[j] = s[j];
}

constexpr int kStateSmem = kStateWarps * kWarpSmemBytes;

// Operand-only state kernel at 6 CTAs per SM (40 registers).  4 (64 registers, more of a lane's 24 gathers in
// flight) and 8 (32 registers) were measured at 70.0 and 74.7 us against 68.8 us for 50 000 rows.
template <int FMT>
cudaError_t launch_state_fmt(int grid, int smem, cudaStream_t s, const ttl_volume& vol, const ttl_params& prm,
                             const ttl_batch& b, int cur, int warp_smem, int early_release) {
  static bool ready = false;
  if (!ready) {
    cudaError_t e = cudaFuncSetAttribute(build_state_kernel<1, FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         kStateSmem);
    if (e != cudaSuccess) return e;
    ready = true;
  }
  return ttl_launch_chain(build_state_kernel<1, FMT>, grid, kStateWarps * 32, smem, s, vol, prm, b, cur, warp_smem,
                          early_release);
}

int state_kernels_ready() {
  static bool done = false;
  if (done) return 0;
  cudaError_t e = cudaFuncSetAttribute(build_state_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kStateSmem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(reset_state_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStateSmem);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(format_state_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStateSmem);
  if (e != cudaSuccess) return (int)e;
  done = true;
  return 0;
}

int check_common(const ttl_volume* vol, const ttl_params* prm) {
  if (!vol || !prm) return TTL_ERR_BAD_ARG;
  if ((vol->CP & 3) || vol->CP < vol->C || vol->CP > kMaxCP) return TTL_ERR_UNSUPPORTED;
  if (prm->n_dirs + 1 > kMaxDirPts) return TTL_ERR_UNSUPPORTED;
  if (7 * vol->C + 3 * prm->n_dirs > kMaxStateLd) return TTL_ERR_UNSUPPORTED;
  return 0;
}

// bf16_layout 1 needs the order-8 volume and room for 7*48 + 3*n_dirs columns; without fp32 rows
// the operand rows must exist.  Layout 0 (fp32 rows + a 16-bit copy) has no tf32 operand: a tf32 actor
// packs from the fp32 rows itself.
int check_layout(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b) {
  if (!b->rank_rec[0] || !b->rank_rec[1] || !b->step_tip || !b->sg_stops || !b->grp_stops) return TTL_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(b->rank_rec[0]) | reinterpret_cast<uintptr_t>(b->rank_rec[1]) |
       reinterpret_cast<uintptr_t>(b->step_tip)) & 15)
    return TTL_ERR_BAD_ARG;
  if (b->operand_fmt != TTL_OPERAND_BF16 && b->operand_fmt != TTL_OPERAND_FP16 && b->operand_fmt != TTL_OPERAND_TF32)
    return TTL_ERR_BAD_ARG;
  if (b->bf16_layout == 0) {
    if (b->operand_fmt == TTL_OPERAND_TF32) return TTL_ERR_UNSUPPORTED;
    return (b->state[0] && b->state[1]) ? 0 : TTL_ERR_BAD_ARG;
  }
  if (b->bf16_layout != 1) return TTL_ERR_BAD_ARG;
  if (vol->C != 45 || vol->CP != 48) return TTL_ERR_UNSUPPORTED;
  if (!b->state_bf16[0] || !b->state_bf16[1] || (b->ld_bf16 & 7)) return TTL_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(b->state_bf16[0]) | reinterpret_cast<uintptr_t>(b->state_bf16[1])) & 15)
    return TTL_ERR_BAD_ARG;
  if (7 * 48 + 3 * prm->n_dirs > b->ld_bf16) return TTL_ERR_UNSUPPORTED;
  if (b->state[0] || b->state[1]) return TTL_ERR_BAD_ARG;   // layout 1 is the operand-only mode
  return 0;
}

}  // namespace

extern "C" {

int ttl_abi_version(void) { return TTL_ABI_VERSION; }
int64_t ttl_launch_count(void) { return (int64_t)g_ttl_launches.load(); }

int ttl_pad_channels(const float* src, float* dst, int64_t n_voxels, int32_t C, int32_t CP,
                     void* stream) {
  if (!src || !dst || CP < C) return TTL_ERR_BAD_ARG;
  const long long total = (long long)n_voxels * CP;
  TTL_LAUNCH("pad_channels_kernel", (cudaStream_t)stream, pad_channels_kernel<<<ttl_div_up(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, n_voxels, C, CP));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_env_reset(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b,
                  const double* seeds, void* stream) {
  int rc = check_common(vol, prm);
  if (rc) return rc;
  if (!b || (!seeds && b->n > 0) || b->n < 0 || b->n > b->capacity || b->ld_state > kMaxStateLd ||
      (b->ld_state & 3) || b->ld_state < 7 * vol->C + 3 * prm->n_dirs || b->n_slots <= 0)
    return TTL_ERR_BAD_ARG;
  rc = check_layout(vol, prm, b);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (b->n == 0) {   // an empty batch (reset(k, k)) still has to clear the control block
    TTL_LAUNCH("reset_kernel", s, reset_kernel<<<1, 32, 0, s>>>(*b, seeds));
    TTL_CHECK_LAST();
    return 0;
  }
  const int n_init = b->n > b->n_slots ? b->n : b->n_slots;
  TTL_LAUNCH("reset_kernel", s, reset_kernel<<<ttl_div_up(n_init, 256), 256, 0, s>>>(*b, seeds));
  const int n0 = b->n < b->n_slots ? b->n : b->n_slots;
  rc = state_kernels_ready();
  if (rc) return rc;
  // the bf16-only path keeps just the corner table in shared memory: a small allocation leaves
  // the SM's 228 KB to L1, which is what dedupes the overlapping trilinear corners
  const int warp_smem = b->bf16_layout == 1 ? kWarpSmemSmall : kWarpSmemBytes;
  TTL_LAUNCH("reset_state_kernel", s,
             reset_state_kernel<<<ttl_div_up(n0, kStateWarps), kStateWarps * 32, kStateWarps * warp_smem, s>>>(
                 *vol, *prm, *b, warp_smem));
  TTL_CHECK_LAST();
  return 0;
}

// propagate_stop_kernel is latency-bound (a short dependent chain per streamline and ~90 registers
// of fp64 spline state): how many 128-thread CTAs share an SM decides how many waves 50 000 rows
// take.  It is built for 6 CTAs per SM (80 registers); 5 (94 registers, what ptxas picks
// unconstrained) and 8 (64, a few spilled doubles) were measured and not adopted.
extern "C++" {   // (inside the extern "C" block)
template <bool RNG>
static void launch_propagate_as(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int cur,
                                const ActionSrc& src, const double* noise, int defer, const ttl_noise& nz,
                                int grid, cudaStream_t s) {
  TTL_LAUNCH("propagate_stop_kernel", s, ttl_launch_chain(propagate_stop_kernel<RNG>, grid, kK1Threads, 0, s, *vol, *prm, *b, cur, src, noise, defer, nz));
}
}  // extern "C++"

// nz != NULL: the noise is drawn in the kernel (ttl_noise) and `noise` must be NULL
static void launch_propagate(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int cur,
                             const ActionSrc& src, const double* noise, int defer, int n_upper, cudaStream_t s,
                             const ttl_noise* nz = nullptr) {
  const int grid = ttl_div_up(n_upper, kGroup);
  if (nz)
    launch_propagate_as<true>(vol, prm, b, cur, src, nullptr, defer, *nz, grid, s);
  else
    launch_propagate_as<false>(vol, prm, b, cur, src, noise, defer, ttl_noise{0.0, 0, 0}, grid, s);
}

// the device-noise entry points need the float64 direction arithmetic the noise is defined in
static int check_noise(const ttl_params* prm, const ttl_noise* nz) {
  if (!prm || !nz || !(nz->sigma >= 0.0) || isinf(nz->sigma)) return TTL_ERR_BAD_ARG;
  if (!prm->dir_f64) return TTL_ERR_UNSUPPORTED;
  return 0;
}

static int launch_build_state(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int cur,
                              int n_upper, cudaStream_t s) {
  int rc = state_kernels_ready();
  if (rc) return rc;
  // the operand-only path keeps just the corner table in shared memory: a small allocation leaves
  // the SM's 228 KB to L1, which is what dedupes the overlapping trilinear corners
  const int warp_smem = b->bf16_layout == 1 ? kWarpSmemSmall : kWarpSmemBytes;
  const int grid = ttl_div_up(n_upper, kStateWarps), smem = kStateWarps * warp_smem;
  const int early_release = g_ttl_pdl.load() ? 1 : 0;
  if (b->bf16_layout == 1 && b->operand_fmt == TTL_OPERAND_TF32)
    TTL_LAUNCH("build_state_kernel", s,
               launch_state_fmt<TTL_OPERAND_TF32>(grid, smem, s, *vol, *prm, *b, cur, warp_smem, early_release));
  else if (b->bf16_layout == 1 && b->operand_fmt == TTL_OPERAND_FP16)
    TTL_LAUNCH("build_state_kernel", s,
               launch_state_fmt<TTL_OPERAND_FP16>(grid, smem, s, *vol, *prm, *b, cur, warp_smem, early_release));
  else if (b->bf16_layout == 1)
    TTL_LAUNCH("build_state_kernel", s,
               launch_state_fmt<TTL_OPERAND_BF16>(grid, smem, s, *vol, *prm, *b, cur, warp_smem, early_release));
  else
    TTL_LAUNCH("build_state_kernel", s,
               ttl_launch_chain(build_state_kernel<0, 0>, grid, kStateWarps * 32, smem, s, *vol, *prm, *b, cur,
                                warp_smem, early_release));
  return 0;
}

static int check_step_args(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                           int32_t* n_upper) {
  int rc = check_common(vol, prm);
  if (rc) return rc;
  if (!b || (cur != 0 && cur != 1)) return TTL_ERR_BAD_ARG;
  if (prm->compute_reward && !vol->peaks && prm->alignment_weighting > 0) return TTL_ERR_BAD_ARG;
  if (prm->refill && prm->state_stopped) return TTL_ERR_BAD_ARG;
  rc = check_layout(vol, prm, b);
  if (rc) return rc;
  if (*n_upper > b->n_slots) *n_upper = b->n_slots;
  if (*n_upper > 0 && (ttl_div_up(*n_upper, kGroup) > b->max_groups || !b->grp_stops || !b->sg_stops ||
                       !b->rank_rec[0] || !b->rank_rec[1] || !b->step_tip))
    return TTL_ERR_BAD_ARG;
  return 0;
}

static int env_step(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                    const float* actions, int32_t lda, const double* noise, const ttl_noise* nz, int defer,
                    int32_t n_upper, cudaStream_t s) {
  if (n_upper <= 0) return 0;   // nothing alive: no launch (and no action buffer to look at)
  if (!actions || lda < 3) return TTL_ERR_BAD_ARG;
  int rc = check_step_args(vol, prm, b, cur, &n_upper);
  if (rc) return rc;
  const ActionSrc src = {actions, lda, nullptr, 0, 1, nullptr, n_upper};
  launch_propagate(vol, prm, b, cur, src, noise, defer, n_upper, s, nz);
  if (!defer) {
    rc = launch_build_state(vol, prm, b, cur, n_upper, s);
    if (rc) return rc;
  }
  TTL_CHECK_LAST();
  return 0;
}

static int env_step_head(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                         const float* head_partial, int32_t n_tiles, int32_t tiles_per_256, const float* head_bias,
                         const ttl_noise* nz, int32_t n_upper, cudaStream_t s) {
  if (n_upper <= 0) return 0;
  if (!head_partial || !head_bias || n_tiles < 1 || (reinterpret_cast<uintptr_t>(head_partial) & 15) ||
      (tiles_per_256 != 1 && tiles_per_256 != 2 && tiles_per_256 != 4))
    return TTL_ERR_BAD_ARG;
  int rc = check_step_args(vol, prm, b, cur, &n_upper);
  if (rc) return rc;
  const ActionSrc src = {nullptr, 0, head_partial, n_tiles, tiles_per_256, head_bias, n_upper};
  launch_propagate(vol, prm, b, cur, src, nullptr, 0, n_upper, s, nz);
  rc = launch_build_state(vol, prm, b, cur, n_upper, s);
  if (rc) return rc;
  TTL_CHECK_LAST();
  return 0;
}

int ttl_env_step(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                 const float* actions, int32_t lda, const double* noise, int32_t n_upper,
                 void* stream) {
  return env_step(vol, prm, b, cur, actions, lda, noise, nullptr, 0, n_upper, (cudaStream_t)stream);
}

int ttl_env_step_head(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                      const float* head_partial, int32_t n_tiles, int32_t tiles_per_256, const float* head_bias,
                      int32_t n_upper, void* stream) {
  return env_step_head(vol, prm, b, cur, head_partial, n_tiles, tiles_per_256, head_bias, nullptr, n_upper,
                       (cudaStream_t)stream);
}

int ttl_env_step_begin(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                       const float* actions, int32_t lda, const double* noise, int32_t n_upper,
                       void* stream) {
  return env_step(vol, prm, b, cur, actions, lda, noise, nullptr, 1, n_upper, (cudaStream_t)stream);
}

int ttl_env_step_rng(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                     const float* actions, int32_t lda, const ttl_noise* nz, int32_t n_upper, void* stream) {
  int rc = check_noise(prm, nz);
  if (rc) return rc;
  return env_step(vol, prm, b, cur, actions, lda, nullptr, nz, 0, n_upper, (cudaStream_t)stream);
}

int ttl_env_step_head_rng(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                          const float* head_partial, int32_t n_tiles, int32_t tiles_per_256,
                          const float* head_bias, const ttl_noise* nz, int32_t n_upper, void* stream) {
  int rc = check_noise(prm, nz);
  if (rc) return rc;
  return env_step_head(vol, prm, b, cur, head_partial, n_tiles, tiles_per_256, head_bias, nz, n_upper,
                       (cudaStream_t)stream);
}

int ttl_env_step_begin_rng(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                           const float* actions, int32_t lda, const ttl_noise* nz, int32_t n_upper,
                           void* stream) {
  int rc = check_noise(prm, nz);
  if (rc) return rc;
  return env_step(vol, prm, b, cur, actions, lda, nullptr, nz, 1, n_upper, (cudaStream_t)stream);
}

int ttl_noise_normals(const ttl_noise* nz, const int64_t* g, const int32_t* L, int32_t n, double* out,
                      void* stream) {
  if (n <= 0) return 0;
  if (!nz || !g || !L || !out) return TTL_ERR_BAD_ARG;
  TTL_LAUNCH("noise_normals_kernel", (cudaStream_t)stream,
             noise_normals_kernel<<<ttl_div_up((long long)n * 3, 256), 256, 0, (cudaStream_t)stream>>>(
                 nz->seed, (const long long*)g, L, n, out));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_env_step_finish(const ttl_volume* vol, const ttl_params* prm, const ttl_batch* b, int32_t cur,
                        const float* scores, int32_t use_stop, int32_t min_pts_stop, int32_t min_pts_reward,
                        float bonus, int32_t n_upper, void* stream) {
  int rc = check_common(vol, prm);
  if (rc) return rc;
  if (n_upper <= 0) return 0;
  if (!b || !scores || (cur != 0 && cur != 1)) return TTL_ERR_BAD_ARG;
  if (n_upper > b->n_slots) n_upper = b->n_slots;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("oracle_apply_kernel", s,
             oracle_apply_kernel<<<ttl_div_up(n_upper, kGroup), kK1Threads, 0, s>>>(
                 *prm, *b, cur, scores, use_stop, min_pts_stop, min_pts_reward, bonus));
  rc = launch_build_state(vol, prm, b, cur, n_upper, s);
  if (rc) return rc;
  TTL_CHECK_LAST();
  return 0;
}

int ttl_env_gather_step_state(const ttl_batch* b, int32_t cur, int32_t n_rows, float* out,
                              int32_t ld_out, void* stream) {
  if (n_rows <= 0) return 0;
  if (!b || !out) return TTL_ERR_BAD_ARG;
  TTL_LAUNCH("gather_rows_kernel", (cudaStream_t)stream, gather_rows_kernel<<<ttl_div_up((long long)n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      b->state[cur ^ 1], b->dest, n_rows, b->ld_state, out, ld_out, b->state_size));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_format_state(const ttl_volume* vol, const ttl_params* prm, const float* points, int32_t n,
                     int32_t L, float* out, int32_t ld_out, void* stream) {
  int rc = check_common(vol, prm);
  if (rc) return rc;
  if (n <= 0) return 0;
  if (!points || !out || L < 1) return TTL_ERR_BAD_ARG;
  rc = state_kernels_ready();
  if (rc) return rc;
  TTL_LAUNCH("format_state_kernel", (cudaStream_t)stream,
             format_state_kernel<<<ttl_div_up(n, kStateWarps), kStateWarps * 32, kStateSmem, (cudaStream_t)stream>>>(
                 *vol, *prm, points, n, L, out, ld_out));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_stopping_flags(const ttl_volume* vol, const ttl_params* prm, const float* points, int32_t n,
                       int32_t L, int32_t* out_flags, double* out_mask_value, float* out_reward,
                       void* stream) {
  int rc = check_common(vol, prm);
  if (rc) return rc;
  if (n <= 0) return 0;
  if (!points || !out_flags || L < 1) return TTL_ERR_BAD_ARG;
  TTL_LAUNCH("stopping_flags_kernel", (cudaStream_t)stream, stopping_flags_kernel<<<ttl_div_up(n, 128), 128, 0, (cudaStream_t)stream>>>(
      *vol, *prm, points, n, L, out_flags, out_mask_value, out_reward));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_streamline_offsets(const ttl_batch* b, int64_t* offsets, void* stream) {
  if (!b || !offsets) return TTL_ERR_BAD_ARG;
  TTL_LAUNCH("offsets_kernel", (cudaStream_t)stream, offsets_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(*b, (long long*)offsets));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_pack_streamlines(const ttl_batch* b, const int64_t* offsets, float* out_points, void* stream) {
  if (b && b->n == 0) return 0;
  if (!b || !offsets || !out_points) return TTL_ERR_BAD_ARG;
  TTL_LAUNCH("pack_kernel", (cudaStream_t)stream, pack_kernel<<<ttl_div_up((long long)b->n * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      *b, (const long long*)offsets, out_points));
  TTL_CHECK_LAST();
  return 0;
}

}  // extern "C"
