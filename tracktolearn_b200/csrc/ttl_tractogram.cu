// Tractogram output path on the device (SURVEY.md section 8(f) rows 1 and 4): what the reference does
// per streamline in Python after tracking (tracking/tracker.py:118-125) -- dipy `length` for the
// min/max length filter and dipy `compress_streamlines` for --compress -- on packed ragged arrays
// [total][3] fp32 + int64 offsets [n+1], one warp per streamline -- and the ordered selection that
// keeps the streamlines passing the length filter and, optionally, the TractOracle-Net score threshold --
// the streamline density and endpoint maps of the streamlines kept -- their connectivity matrix over a
// label volume -- and their tractometry: per-streamline means of scalar maps and metric-weighted matrices.
#include <math.h>

#include <cub/device/device_scan.cuh>

#include "ttl_common.cuh"

namespace {

constexpr int kWarpsPerBlock = 8;

// x*x + y*y + z*z left to right without fused multiply-adds (numpy's order and rounding)
__device__ __forceinline__ double sumsq3(double x, double y, double z) {
  return __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
}

// dipy.tracking.streamline.length: sum of the segment norms, in double (tracker.py:120).
// Lanes take segments round-robin; the 32 partial sums are combined by a shuffle tree, so the value
// can differ from a sequential sum in the last bits (tests allow 1e-12 relative).
__global__ void __launch_bounds__(kWarpsPerBlock * 32) streamline_length_kernel(
    const float* __restrict__ points, const long long* __restrict__ offsets, int n, double* __restrict__ out) {
  const int i = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  const long long beg = offsets[i], end = offsets[i + 1];
  const float* P = points + beg * 3;
  const int N = (int)(end - beg);
  double acc = 0.0;
  for (int j = lane; j + 1 < N; j += 32) {
    const double dx = (double)P[3 * j + 3] - (double)P[3 * j + 0];
    const double dy = (double)P[3 * j + 4] - (double)P[3 * j + 1];
    const double dz = (double)P[3 * j + 5] - (double)P[3 * j + 2];
    acc += sqrt(dx * dx + dy * dy + dz * dz);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) out[i] = acc;
}

// dipy compress_streamlines (streamlinespeed.pyx c_compress_streamline), restated in
// oracle/ttl_oracle.py::compress_streamline -- same arithmetic: coordinate differences and their
// products in float (no contraction), sums and square roots in double.  The walk over `nxt` is
// sequential (prev depends on the previous decision); the test of the points between prev and nxt
// is spread over the lanes (any point off the chord by more than tol, or a NaN distance, keeps
// point nxt-1).  Output: keep[total] (1 = point survives) and count[n].
__global__ void __launch_bounds__(kWarpsPerBlock * 32) compress_mask_kernel(
    const float* __restrict__ points, const long long* __restrict__ offsets, int n, double tol_error,
    double max_segment_length, uint8_t* __restrict__ keep, int* __restrict__ count) {
  const int i = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  const long long beg = offsets[i], end = offsets[i + 1];
  const float* P = points + beg * 3;
  uint8_t* K = keep + beg;
  const int N = (int)(end - beg);
  if (N <= 2) {   // copied as is
    if (lane < N) K[lane] = 1;
    if (lane == 0) count[i] = N;
    return;
  }
  for (int j = lane; j < N; j += 32) K[j] = (j == 0 || j == N - 1) ? 1 : 0;
  __syncwarp();   // lane 0 overwrites entries other lanes have just cleared
  int prev = 0, nb = 2;
  float px = P[0], py = P[1], pz = P[2];
  for (int nxt = 2; nxt < N; ++nxt) {
    const float nx = P[3 * nxt + 0], ny = P[3 * nxt + 1], nz = P[3 * nxt + 2];
    const float ax = __fsub_rn(nx, px), ay = __fsub_rn(ny, py), az = __fsub_rn(nz, pz);
    const double seg = sqrt(sumsq3((double)ax, (double)ay, (double)az));
    bool replace = false;
    if (seg < max_segment_length) {
      const double norm2 = sqrt(__dadd_rn(__dadd_rn((double)__fmul_rn(ax, ax), (double)__fmul_rn(ay, ay)),
                                          (double)__fmul_rn(az, az)));
      bool fail = false;
      for (int base = prev + 1; base < nxt; base += 32) {
        const int curr = base + lane;
        if (curr < nxt) {
          const float bx = __fsub_rn(P[3 * curr + 0], nx), by = __fsub_rn(P[3 * curr + 1], ny),
                      bz = __fsub_rn(P[3 * curr + 2], nz);
          const double cx = (double)__fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by));
          const double cy = (double)__fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz));
          const double cz = (double)__fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx));
          const double dist = sqrt(sumsq3(cx, cy, cz)) / norm2;
          fail |= isnan(dist) || dist > tol_error;
        }
      }
      replace = !__any_sync(0xffffffffu, fail);
    }
    if (!replace) {
      prev = nxt - 1;
      px = P[3 * prev + 0]; py = P[3 * prev + 1]; pz = P[3 * prev + 2];
      if (lane == 0) K[prev] = 1;
      ++nb;
    }
  }
  if (lane == 0) count[i] = nb;
}

// Ordered selection of packed streamlines.  Row i contributes (1, its point count) when it is kept and
// (0, 0) otherwise; an exclusive scan of these pairs gives every kept row its output position and its
// first output point.  A NaN score fails `>=` and is never kept.
struct PairSum {
  __device__ __forceinline__ longlong2 operator()(const longlong2& a, const longlong2& b) const {
    return make_longlong2(a.x + b.x, a.y + b.y);
  }
};

constexpr int kSelectThreads = 256;

__global__ void __launch_bounds__(kSelectThreads) select_flag_kernel(
    const long long* __restrict__ offsets, int n, const uint8_t* __restrict__ keep_in,
    const float* __restrict__ scores, float threshold, longlong2* __restrict__ vals) {
  const int i = blockIdx.x * kSelectThreads + threadIdx.x;
  if (i >= n) return;
  const bool keep = (keep_in == nullptr || keep_in[i] != 0) && (scores == nullptr || scores[i] >= threshold);
  vals[i] = keep ? make_longlong2(1, offsets[i + 1] - offsets[i]) : make_longlong2(0, 0);
}

__global__ void __launch_bounds__(kSelectThreads) select_scatter_kernel(
    const longlong2* __restrict__ vals, const longlong2* __restrict__ pre, int n, long long* __restrict__ out_offsets,
    long long* __restrict__ out_index, long long* __restrict__ result) {
  const int i = blockIdx.x * kSelectThreads + threadIdx.x;
  if (i >= n) return;
  const longlong2 v = vals[i], p = pre[i];
  if (v.x) {
    out_index[p.x] = i;
    out_offsets[p.x + 1] = p.y + v.y;
  }
  if (i == n - 1) {
    out_offsets[0] = 0;
    result[0] = p.x + v.x;
    result[1] = p.y + v.y;
  }
}

// out_points[out_offsets[k]..] = points[offsets[index[k]]..], one warp per kept streamline.
__global__ void __launch_bounds__(kWarpsPerBlock * 32) gather_streamlines_kernel(
    const float* __restrict__ points, const long long* __restrict__ offsets, const long long* __restrict__ index,
    const long long* __restrict__ out_offsets, int m, float* __restrict__ out_points) {
  const int k = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (k >= m) return;
  const float* src = points + offsets[index[k]] * 3;
  float* dst = out_points + out_offsets[k] * 3;
  const long long cnt = (out_offsets[k + 1] - out_offsets[k]) * 3;
  for (long long j = lane; j < cnt; j += 32) dst[j] = src[j];
}

// Streamline maps (DESIGN.md section 2, "Streamline maps").  The voxel of a point p is c_k = floor(p_k + 0.5)
// per axis, computed in double where the addition is exact (dipy density_map's int(p + 0.5) without the
// rounding a float sum would add); the point is in the grid when 0 <= c_k < dim_k on every axis, a test NaN
// and +-inf fail.  Returns the linear index (x * ny + y) * nz + z, or -1 outside the grid.
__device__ __forceinline__ int map_voxel(const float* p, int nx, int ny, int nz) {
  const double cx = floor(__dadd_rn((double)p[0], 0.5));
  const double cy = floor(__dadd_rn((double)p[1], 0.5));
  const double cz = floor(__dadd_rn((double)p[2], 0.5));
  if (!(cx >= 0.0 && cx < (double)nx && cy >= 0.0 && cy < (double)ny && cz >= 0.0 && cz < (double)nz)) return -1;
  return ((int)cx * ny + (int)cy) * nz + (int)cz;
}

// Distinct voxels of one streamline kept in shared memory, per warp: 16 KB a block.  A streamline that
// touches more distinct voxels stays exact through the rescan below, only slower.
constexpr int kMapSeen = 512;

// One warp per streamline, its points in chunks of 32.  density[v] += 1 once for every distinct in-grid voxel
// of the streamline: in a chunk the lowest lane of each voxel (__match_any_sync) is a candidate, and a
// candidate counts unless the voxel is already in the warp's set of the streamline's earlier voxels.  Once that
// set has overflowed it no longer holds every earlier voxel, and a candidate it misses is compared with every
// earlier point instead.  endpoints[v] += 1 for the first and for the last point.  Out-of-grid points are
// summed per warp into *skipped.  Counts are integer atomics: the maps do not depend on launch order.
__global__ void __launch_bounds__(kWarpsPerBlock * 32) tract_maps_kernel(
    const float* __restrict__ points, const long long* __restrict__ offsets, int n, int nx, int ny, int nz,
    int* __restrict__ density, int* __restrict__ endpoints, unsigned long long* __restrict__ skipped) {
  __shared__ int seen_block[kWarpsPerBlock][kMapSeen];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * kWarpsPerBlock + warp;
  if (i >= n) return;
  int* seen = seen_block[warp];
  const long long beg = offsets[i];
  const int N = (int)(offsets[i + 1] - beg);
  const float* P = points + beg * 3;
  if (endpoints != nullptr && lane < 2 && N > 0) {
    const int v = map_voxel(P + 3 * (lane == 0 ? 0 : N - 1), nx, ny, nz);
    if (v >= 0) atomicAdd(endpoints + v, 1);
  }
  unsigned outside = 0;
  int n_seen = 0;
  bool complete = true;      // seen[] holds every in-grid voxel of the points before `base`
  for (int base = 0; base < N; base += 32) {
    const int j = base + lane;
    const int v = j < N ? map_voxel(P + 3 * j, nx, ny, nz) : -1;
    outside += (j < N && v < 0) ? 1u : 0u;
    if (density == nullptr) continue;
    const unsigned same = __match_any_sync(0xffffffffu, v);
    bool cand = v >= 0 && __ffs(same) - 1 == lane;
    for (unsigned todo = __ballot_sync(0xffffffffu, cand); todo != 0; todo &= todo - 1) {
      const int src = __ffs(todo) - 1;
      const int w = __shfl_sync(0xffffffffu, v, src);
      bool hit = false;
      for (int k = lane; k < n_seen; k += 32) hit |= seen[k] == w;
      if (__any_sync(0xffffffffu, hit) && lane == src) cand = false;
    }
    if (!complete && __any_sync(0xffffffffu, cand)) {
      bool found = false;
      for (int b = 0; b < base; b += 32) {       // b + lane < base: base is a multiple of 32
        const int e = map_voxel(P + 3 * (b + lane), nx, ny, nz);
#pragma unroll
        for (int k = 0; k < 32; ++k) found |= __shfl_sync(0xffffffffu, e, k) == v;
      }
      cand = cand && !found;
    }
    if (cand) atomicAdd(density + v, 1);
    const unsigned add = __ballot_sync(0xffffffffu, cand);
    const int pos = n_seen + __popc(add & ((1u << lane) - 1u));
    if (cand && pos < kMapSeen) seen[pos] = v;
    if (n_seen + __popc(add) > kMapSeen) complete = false;
    n_seen = min(n_seen + __popc(add), kMapSeen);
    __syncwarp();
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) outside += __shfl_xor_sync(0xffffffffu, outside, off);
  if (lane == 0 && outside != 0) atomicAdd(skipped, (unsigned long long)outside);
}

// Connectivity matrix (DESIGN.md section 2, "Connectivity matrix").  A label value outside [0, K) reads as 0,
// so no value a caller leaves in the volume can index past the matrix.
__device__ __forceinline__ int conn_label(const int* labels, int v, int K) {
  const int l = labels[v];
  return (l > 0 && l < K) ? l : 0;
}

// Label of the endpoint p, computed by the whole warp (every lane returns it).  Its own voxel
// floor((double)p + 0.5) when in the grid and labelled; otherwise the labelled voxel c of the box
// ceil(p - r) <= c <= floor(p + r) (fp64 bounds, clamped to the grid) with the smallest
// d2 = ((dx*dx) + (dy*dy)) + (dz*dz) <= r2, dx = (double)c - (double)p, every operation rounded to nearest with
// no contraction; ties go to the smaller linear index.  0 when there is none or p is not finite.  Lanes take
// the box's voxels round-robin and read a label only inside the sphere; a shuffle tree finds the minimum of
// (d2, index).
__device__ __forceinline__ int conn_end_label(const float* p, const int* __restrict__ labels, int nx, int ny,
                                              int nz, int K, double r, double r2, int lane) {
  const double px = (double)p[0], py = (double)p[1], pz = (double)p[2];
  const int own = map_voxel(p, nx, ny, nz);
  if (own >= 0) {
    const int l = conn_label(labels, own, K);
    if (l > 0) return l;
  }
  if (!(isfinite(px) && isfinite(py) && isfinite(pz))) return 0;
  const double lx = fmax(ceil(__dsub_rn(px, r)), 0.0), hx = fmin(floor(__dadd_rn(px, r)), (double)(nx - 1));
  const double ly = fmax(ceil(__dsub_rn(py, r)), 0.0), hy = fmin(floor(__dadd_rn(py, r)), (double)(ny - 1));
  const double lz = fmax(ceil(__dsub_rn(pz, r)), 0.0), hz = fmin(floor(__dadd_rn(pz, r)), (double)(nz - 1));
  if (!(lx <= hx && ly <= hy && lz <= hz)) return 0;
  const int x0 = (int)lx, y0 = (int)ly, z0 = (int)lz;
  const int by = (int)hy - y0 + 1, bz = (int)hz - z0 + 1;
  const int plane = by * bz, count = ((int)hx - x0 + 1) * plane;
  double best = r2;
  int best_v = 0x7fffffff, best_l = 0;
  for (int t = lane; t < count; t += 32) {
    const int ix = t / plane, rem = t - ix * plane;
    const int iy = rem / bz, iz = rem - iy * bz;
    const int cx = x0 + ix, cy = y0 + iy, cz = z0 + iz;
    const double d2 = sumsq3(__dsub_rn((double)cx, px), __dsub_rn((double)cy, py), __dsub_rn((double)cz, pz));
    if (d2 <= best) {
      const int v = (cx * ny + cy) * nz + cz;
      const int l = conn_label(labels, v, K);
      if (l > 0 && (d2 < best || v < best_v)) {
        best = d2;
        best_v = v;
        best_l = l;
      }
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, best, off);
    const int ov = __shfl_xor_sync(0xffffffffu, best_v, off);
    const int ol = __shfl_xor_sync(0xffffffffu, best_l, off);
    if (ol > 0 && (best_l == 0 || od < best || (od == best && ov < best_v))) {
      best = od;
      best_v = ov;
      best_l = ol;
    }
  }
  return best_l;
}

// One warp per streamline: the labels (a, b) of its first and last points.  matrix[a][a] += 1 when a == b,
// else matrix[a][b] += 1 and matrix[b][a] += 1 (integer atomics: the matrix does not depend on launch order);
// an empty streamline adds nothing and gets the pair (0, 0).
__global__ void __launch_bounds__(kWarpsPerBlock * 32) connectome_kernel(
    const float* __restrict__ points, const long long* __restrict__ offsets, int n, const int* __restrict__ labels,
    int nx, int ny, int nz, int K, double r, int* __restrict__ matrix, int* __restrict__ pairs) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (i >= n) return;
  const long long beg = offsets[i];
  const long long N = offsets[i + 1] - beg;
  int a = 0, b = 0;
  if (N > 0) {
    const double r2 = __dmul_rn(r, r);
    a = conn_end_label(points + beg * 3, labels, nx, ny, nz, K, r, r2, lane);
    b = conn_end_label(points + (beg + N - 1) * 3, labels, nx, ny, nz, K, r, r2, lane);
  }
  if (lane != 0) return;
  if (pairs != nullptr) {
    pairs[2 * (long long)i] = a;
    pairs[2 * (long long)i + 1] = b;
  }
  if (matrix != nullptr && N > 0) {
    atomicAdd(matrix + a * K + b, 1);
    if (a != b) atomicAdd(matrix + b * K + a, 1);
  }
}

// Tractometry (DESIGN.md section 2, "Tractometry").  The C metrics of voxel v are vol[v*C .. v*C+C-1]: one
// read-only vector load per corner where C allows it (float4 for C = 4 / 8, float2 for C = 2).
template <int C>
__device__ __forceinline__ void metric_corner(const float* __restrict__ vol, int v, float (&m)[C]) {
  const float* p = vol + (long long)v * C;
  if constexpr (C % 4 == 0) {
#pragma unroll
    for (int c = 0; c < C; c += 4) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(p + c));
      m[c] = q.x; m[c + 1] = q.y; m[c + 2] = q.z; m[c + 3] = q.w;
    }
  } else if constexpr (C % 2 == 0) {
#pragma unroll
    for (int c = 0; c < C; c += 2) {
      const float2 q = __ldg(reinterpret_cast<const float2*>(p + c));
      m[c] = q.x; m[c + 1] = q.y;
    }
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) m[c] = __ldg(p + c);
  }
}

// Lower corner index, upper corner index and upper weight of one axis: i = floor(c), d = c - i, corners
// clamp(i, 0, n-1) and clamp(i+1, 0, n-1).  Only called for points map_voxel puts in the grid, so
// -1 <= i <= n-1 and the casts are exact.
__device__ __forceinline__ void metric_axis(float p, int n, int& i0, int& i1, double& d) {
  const double c = (double)p;
  const double f = floor(c);
  d = __dsub_rn(c, f);
  const int i = (int)f;
  i0 = max(i, 0);
  i1 = min(i + 1, n - 1);
}

// One warp per streamline.  Lane l takes points l, l+32, ... in order; a point that map_voxel puts in the
// grid adds its trilinear value, sum over the 8 corners (x, y, z lower before upper, z fastest) of
// ((wx * wy) * wz) * value, every operation fp64 round-to-nearest without contraction, to the lane's fp64
// partial sum of each metric.  A fixed xor-shuffle tree then adds the 32 partial sums, so the order of the
// sum depends on the point count alone.  means[i][c] = (float)(sum / count), NaN without a sampled point.
// Out-of-grid points are summed per warp into *skipped.
template <int C>
__global__ void __launch_bounds__(kWarpsPerBlock * 32) sample_metrics_kernel(
    const float* __restrict__ points, const long long* __restrict__ offsets, int n, const float* __restrict__ vol,
    int nx, int ny, int nz, float* __restrict__ means, unsigned long long* __restrict__ skipped) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (i >= n) return;
  const long long beg = offsets[i];
  const int N = (int)(offsets[i + 1] - beg);
  const float* P = points + beg * 3;
  double acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 0.0;
  int count = 0;
  unsigned outside = 0;
  for (int j = lane; j < N; j += 32) {
    const float* p = P + 3 * j;
    if (map_voxel(p, nx, ny, nz) < 0) {
      ++outside;
      continue;
    }
    int x0, x1, y0, y1, z0, z1;
    double dx, dy, dz;
    metric_axis(p[0], nx, x0, x1, dx);
    metric_axis(p[1], ny, y0, y1, dy);
    metric_axis(p[2], nz, z0, z1, dz);
    const double wx[2] = {__dsub_rn(1.0, dx), dx}, wy[2] = {__dsub_rn(1.0, dy), dy}, wz[2] = {__dsub_rn(1.0, dz), dz};
    const int xs[2] = {x0, x1}, ys[2] = {y0, y1}, zs[2] = {z0, z1};
    double val[C];
#pragma unroll
    for (int c = 0; c < C; ++c) val[c] = 0.0;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const double wxy = __dmul_rn(wx[a], wy[b]);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const double w = __dmul_rn(wxy, wz[e]);
          float m[C];
          metric_corner<C>(vol, (xs[a] * ny + ys[b]) * nz + zs[e], m);
#pragma unroll
          for (int c = 0; c < C; ++c) val[c] = __dadd_rn(val[c], __dmul_rn(w, (double)m[c]));
        }
      }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = __dadd_rn(acc[c], val[c]);
    ++count;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = __dadd_rn(acc[c], __shfl_xor_sync(0xffffffffu, acc[c], off));
    count += __shfl_xor_sync(0xffffffffu, count, off);
    outside += __shfl_xor_sync(0xffffffffu, outside, off);
  }
  if (lane != 0) return;
#pragma unroll
  for (int c = 0; c < C; ++c)
    means[(long long)i * C + c] = count > 0 ? __double2float_rn(__ddiv_rn(acc[c], (double)count)) : __int_as_float(0x7fc00000);
  if (outside != 0) atomicAdd(skipped, (unsigned long long)outside);
}

// The fixed-point shift of every column, passed by value: the host checks them before the launch.
struct SumShifts {
  int s[TTL_CONNECTOME_SUMS_MAX_COLUMNS];
};

// One thread per (streamline, column): a finite value v with end labels (a, b) adds
// q = __double2ll_rn(ldexp((double)v, shift)) to sums[c][a][b] and 1 to counts[c][a][b], and the same at [b][a]
// when a != b.  Integer atomics: the planes do not depend on launch order.  A label outside [0, K) reads as 0.
__global__ void __launch_bounds__(256) connectome_sums_kernel(
    const int* __restrict__ pairs, int n, const float* __restrict__ values, int C, int K, const SumShifts shifts,
    long long* __restrict__ sums, int* __restrict__ counts) {
  const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
  if (t >= (long long)n * C) return;
  const int i = (int)(t / C), c = (int)(t - (long long)i * C);
  const float v = values[t];
  if (!isfinite(v)) return;
  int a = pairs[2 * (long long)i], b = pairs[2 * (long long)i + 1];
  a = (a > 0 && a < K) ? a : 0;
  b = (b > 0 && b < K) ? b : 0;
  int shift = 0;      // selected with constant indices: a dynamic index would copy the array to the stack
#pragma unroll
  for (int k = 0; k < TTL_CONNECTOME_SUMS_MAX_COLUMNS; ++k) shift = k == c ? shifts.s[k] : shift;
  const long long q = __double2ll_rn(ldexp((double)v, shift));
  const long long base = (long long)c * K * K;
  atomicAdd((unsigned long long*)(sums + base + (long long)a * K + b), (unsigned long long)q);
  atomicAdd(counts + base + (long long)a * K + b, 1);
  if (a != b) {
    atomicAdd((unsigned long long*)(sums + base + (long long)b * K + a), (unsigned long long)q);
    atomicAdd(counts + base + (long long)b * K + a, 1);
  }
}

template <int C>
void launch_sample_metrics(const float* points, const long long* offsets, int n, const float* vol, int nx, int ny,
                           int nz, float* means, unsigned long long* skipped, cudaStream_t s) {
  sample_metrics_kernel<C><<<ttl_div_up(n, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
      points, offsets, n, vol, nx, ny, nz, means, skipped);
}

typedef void (*sample_metrics_launcher)(const float*, const long long*, int, const float*, int, int, int, float*,
                                        unsigned long long*, cudaStream_t);
const sample_metrics_launcher kSampleMetrics[TTL_SAMPLE_MAX_METRICS] = {
    launch_sample_metrics<1>, launch_sample_metrics<2>, launch_sample_metrics<3>, launch_sample_metrics<4>,
    launch_sample_metrics<5>, launch_sample_metrics<6>, launch_sample_metrics<7>, launch_sample_metrics<8>};

size_t select_pairs_bytes(int n) { return ((size_t)n * sizeof(longlong2) + 255) / 256 * 256; }

size_t select_scan_bytes(int n) {
  size_t tmp = 0;
  cub::DeviceScan::ExclusiveScan(nullptr, tmp, (const longlong2*)nullptr, (longlong2*)nullptr, PairSum(),
                                 make_longlong2(0, 0), n);
  return tmp;
}

}  // namespace

extern "C" {

int ttl_streamline_lengths(const float* points, const int64_t* offsets, int32_t n, double* out_lengths,
                           void* stream) {
  if (n <= 0) return 0;
  if (!points || !offsets || !out_lengths) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("streamline_length_kernel", s,
             streamline_length_kernel<<<ttl_div_up(n, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
                 points, (const long long*)offsets, n, out_lengths));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_compress_mask(const float* points, const int64_t* offsets, int32_t n, double tol_error,
                      double max_segment_length, uint8_t* keep, int32_t* count, void* stream) {
  if (n <= 0) return 0;
  if (!points || !offsets || !keep || !count || !(tol_error >= 0.0)) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("compress_mask_kernel", s,
             compress_mask_kernel<<<ttl_div_up(n, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
                 points, (const long long*)offsets, n, tol_error, max_segment_length, keep, count));
  TTL_CHECK_LAST();
  return 0;
}

int64_t ttl_select_workspace_bytes(int32_t n) {
  if (n < 0) return TTL_ERR_BAD_ARG;
  if (n == 0) return 0;
  return (int64_t)(2 * select_pairs_bytes(n) + select_scan_bytes(n));
}

int ttl_select_streamlines(const int64_t* offsets, int32_t n, const uint8_t* keep_in, const float* scores,
                           float threshold, void* workspace, int64_t workspace_bytes, int64_t* out_offsets,
                           int64_t* out_index, int64_t* result, void* stream) {
  if (n < 0 || !out_offsets || !result) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  if (n == 0) {
    if (cudaMemsetAsync(out_offsets, 0, sizeof(int64_t), s) != cudaSuccess ||
        cudaMemsetAsync(result, 0, 2 * sizeof(int64_t), s) != cudaSuccess)
      return TTL_ERR_DRIVER;
    return 0;
  }
  if (!offsets || !out_index || !workspace || workspace_bytes < ttl_select_workspace_bytes(n)) return TTL_ERR_BAD_ARG;
  longlong2* vals = (longlong2*)workspace;
  longlong2* pre = (longlong2*)((char*)workspace + select_pairs_bytes(n));
  void* tmp = (char*)workspace + 2 * select_pairs_bytes(n);
  size_t tmp_bytes = select_scan_bytes(n);
  const int blocks = ttl_div_up(n, kSelectThreads);
  TTL_LAUNCH("select_flag_kernel", s,
             select_flag_kernel<<<blocks, kSelectThreads, 0, s>>>((const long long*)offsets, n, keep_in, scores,
                                                                   threshold, vals));
  TTL_CHECK_LAST();
  cudaError_t e = cudaSuccess;
  TTL_LAUNCH("select_scan", s,
             e = cub::DeviceScan::ExclusiveScan(tmp, tmp_bytes, (const longlong2*)vals, pre, PairSum(), make_longlong2(0, 0), n, s));
  if (e != cudaSuccess) return (int)e;
  TTL_LAUNCH("select_scatter_kernel", s,
             select_scatter_kernel<<<blocks, kSelectThreads, 0, s>>>(vals, pre, n, (long long*)out_offsets,
                                                                      (long long*)out_index, (long long*)result));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_gather_streamlines(const float* points, const int64_t* offsets, const int64_t* index,
                           const int64_t* out_offsets, int32_t m, float* out_points, void* stream) {
  if (m < 0) return TTL_ERR_BAD_ARG;
  if (m == 0) return 0;
  if (!points || !offsets || !index || !out_offsets || !out_points) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("gather_streamlines_kernel", s,
             gather_streamlines_kernel<<<ttl_div_up(m, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
                 points, (const long long*)offsets, (const long long*)index, (const long long*)out_offsets, m,
                 out_points));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_tract_maps(const float* points, const int64_t* offsets, int32_t n, int32_t nx, int32_t ny, int32_t nz,
                   int32_t* density, int32_t* endpoints, int64_t* skipped, void* stream) {
  if (n < 0 || nx <= 0 || ny <= 0 || nz <= 0 || (int64_t)nx * ny * nz >= ((int64_t)1 << 31) ||
      (!density && !endpoints) || !skipped)
    return TTL_ERR_BAD_ARG;
  if (n == 0) return 0;
  if (!points || !offsets) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("tract_maps_kernel", s,
             tract_maps_kernel<<<ttl_div_up(n, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
                 points, (const long long*)offsets, n, nx, ny, nz, density, endpoints,
                 (unsigned long long*)skipped));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_connectome(const float* points, const int64_t* offsets, int32_t n, const int32_t* labels, int32_t nx,
                   int32_t ny, int32_t nz, int32_t K, double radius_vox, int32_t* matrix, int32_t* pairs,
                   void* stream) {
  if (n < 0 || nx <= 0 || ny <= 0 || nz <= 0 || (int64_t)nx * ny * nz >= ((int64_t)1 << 31) || K < 1 ||
      K > TTL_CONNECTOME_MAX_LABELS ||
      !(radius_vox >= 0.0 && radius_vox <= TTL_CONNECTOME_MAX_RADIUS) ||
      (!matrix && !pairs) || !labels)
    return TTL_ERR_BAD_ARG;
  if (n == 0) return 0;
  if (!points || !offsets) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("connectome_kernel", s,
             connectome_kernel<<<ttl_div_up(n, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
                 points, (const long long*)offsets, n, labels, nx, ny, nz, K, radius_vox, matrix, pairs));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_sample_metrics(const float* points, const int64_t* offsets, int32_t n, const float* volumes, int32_t C,
                       int32_t nx, int32_t ny, int32_t nz, float* means, int64_t* skipped, void* stream) {
  if (n < 0 || C < 1 || C > TTL_SAMPLE_MAX_METRICS || nx <= 0 || ny <= 0 || nz <= 0 ||
      (int64_t)nx * ny * nz * C >= ((int64_t)1 << 31) || !volumes || !means || !skipped)
    return TTL_ERR_BAD_ARG;
  if (n == 0) return 0;
  if (!points || !offsets) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("sample_metrics_kernel", s,
             kSampleMetrics[C - 1](points, (const long long*)offsets, n, volumes, nx, ny, nz, means,
                                   (unsigned long long*)skipped, s));
  TTL_CHECK_LAST();
  return 0;
}

int ttl_connectome_sums(const int32_t* pairs, int32_t n, const float* values, int32_t C, int32_t K,
                        const int32_t* shifts, int64_t* sums, int32_t* counts, void* stream) {
  if (n < 0 || C < 1 || C > TTL_CONNECTOME_SUMS_MAX_COLUMNS || K < 1 || K > TTL_CONNECTOME_MAX_LABELS || !shifts ||
      !sums || !counts)
    return TTL_ERR_BAD_ARG;
  SumShifts sh;
  for (int c = 0; c < C; ++c) {
    if (shifts[c] < 0 || shifts[c] > TTL_CONNECTOME_SUMS_MAX_SHIFT) return TTL_ERR_BAD_ARG;
    sh.s[c] = shifts[c];
  }
  if (n == 0) return 0;
  if (!pairs || !values) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  TTL_LAUNCH("connectome_sums_kernel", s,
             connectome_sums_kernel<<<ttl_div_up((long long)n * C, 256), 256, 0, s>>>(
                 pairs, n, values, C, K, sh, (long long*)sums, counts));
  TTL_CHECK_LAST();
  return 0;
}

}  // extern "C"
