// Tractogram output path on the device (SURVEY.md section 8(f) rows 1 and 4): what the reference does
// per streamline in Python after tracking (tracking/tracker.py:118-125) -- dipy `length` for the
// min/max length filter and dipy `compress_streamlines` for --compress -- on packed ragged arrays
// [total][3] fp32 + int64 offsets [n+1], one warp per streamline -- and the ordered selection that
// keeps the streamlines passing the length filter and, optionally, the TractOracle-Net score threshold.
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

}  // extern "C"
