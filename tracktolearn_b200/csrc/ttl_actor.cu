// SAC actor forward for B200 (sm_100a): the only dense contraction on the tracking path.
//
// Reference: algorithms/shared/offpolicy.py:94-140 (MaxEntropyActor.forward) over the
// nn.Sequential built by algorithms/shared/utils.py:41-51 (Linear+ReLU x3, Linear), which the
// reference runs as four cuBLAS sgemm calls plus ~15 small elementwise launches.
//
// Here:
//   pack_state   fp32 state rows [n][ld] -> operand rows [n][k_pad] (skipped when the env step already
//                wrote them, ttl_actor_forward_packed)
//   hidden layers  ONE persistent launch of mlp_pair_kernel (ttl_mlp.cuh): TMA-staged operands,
//                tcgen05.mma.cta_group::2 (M = 256), fp32 accumulators in tensor memory, layers chained
//                through dependency flags; operands in bf16, fp16 or tf32 (TTL_PRECISION_*)
//   head         the last (6-wide) layer is contracted in fp32 inside the last hidden layer's epilogue
//                (per-tile partial sums); head_finish_kernel -- or the env step itself
//                (ttl_env_step, ttl_step_action) -- sums them and applies clamp / exp / tanh / log-prob.
// A CUDA-core fp32 tier (TTL_PRECISION_FP32) reproduces the reference's fp32 arithmetic to ~1e-6 for
// parity tests and users who want it.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "ttl_common.cuh"
#include "ttl_mlp.cuh"
#include "ttl_tc.cuh"

namespace {
using namespace ttl_tc;
using namespace ttl_mlp;

// ==========================================================================================
// Packing kernels
// ==========================================================================================
// operand element of KIND from fp32: bf16 / fp16 (saturating) / fp32 rounded to tf32
template <int KIND>
__device__ __forceinline__ void store_operand(void* out, long long idx, float x) {
  if (KIND == KIND_TF32) {
    static_cast<uint32_t*>(out)[idx] = round_tf32(x);
  } else if (KIND == KIND_F16) {
    static_cast<uint16_t*>(out)[idx] = (uint16_t)(pack_pair<KIND_F16>(x, 0.f) & 0xffffu);
  } else {
    static_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(x);
  }
}
template <int KIND>
__global__ void pack_weight_kernel(const float* __restrict__ w, void* __restrict__ out, int n_out, int n_in,
                                   int n_pad, int k_pad) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n_pad * k_pad) return;
  const int r = (int)(t / k_pad), c = (int)(t - (long long)r * k_pad);
  const float x = (r < n_out && c < n_in) ? w[(size_t)r * n_in + c] : 0.f;
  store_operand<KIND>(out, t, x);
}
// first-layer weights for the channel-padded input layout: packed column q reads original column
// p*C + ch for q = p*CP + ch (ch < C), n_points*C + (q - n_points*CP) behind the SH block, else 0
template <int KIND>
__global__ void pack_weight_layout_kernel(const float* __restrict__ w, void* __restrict__ out, int n_out,
                                          int n_in, int n_pad, int k_pad, int C, int CP, int n_pts) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n_pad * k_pad) return;
  const int r = (int)(t / k_pad), q = (int)(t - (long long)r * k_pad);
  int c = -1;
  if (q < n_pts * CP) {
    const int p = q / CP, ch = q - p * CP;
    if (ch < C) c = p * C + ch;
  } else {
    c = n_pts * C + (q - n_pts * CP);
  }
  const float x = (r < n_out && c >= 0 && c < n_in) ? w[(size_t)r * n_in + c] : 0.f;
  store_operand<KIND>(out, t, x);
}
__global__ void pack_bias_kernel(const float* __restrict__ b, float* __restrict__ out, int n_out, int n_pad) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_pad) out[t] = t < n_out ? b[t] : 0.f;
}
// fp32 state rows -> operand rows padded to k_pad (4 consecutive outputs per thread)
template <int KIND>
__global__ void __launch_bounds__(256) pack_state_kernel(const float* __restrict__ state, int ld, int width,
                                                         const int* __restrict__ n_dev, int n_max,
                                                         void* __restrict__ out, int k_pad,
                                                         unsigned* __restrict__ overflow) {
  int n = n_dev ? *n_dev : n_max;
  n = min(n, n_max);
  const int per_row = k_pad >> 2;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * per_row) return;
  const int r = (int)(t / per_row), g = (int)(t - (long long)r * per_row);
  const float* s = state + (size_t)r * ld + g * 4;
  float x[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) x[j] = g * 4 + j < width ? s[j] : 0.f;
  if (KIND == KIND_TF32) {
    *reinterpret_cast<uint4*>(static_cast<uint32_t*>(out) + (size_t)r * k_pad + g * 4) =
        make_uint4(round_tf32(x[0]), round_tf32(x[1]), round_tf32(x[2]), round_tf32(x[3]));
  } else {
    if (KIND == KIND_F16 && overflow &&
        (fabsf(x[0]) > 65504.f || fabsf(x[1]) > 65504.f || fabsf(x[2]) > 65504.f || fabsf(x[3]) > 65504.f))
      atomicOr(overflow, 1u);
    *reinterpret_cast<uint2*>(static_cast<uint16_t*>(out) + (size_t)r * k_pad + g * 4) =
        make_uint2(pack_pair<KIND>(x[0], x[1]), pack_pair<KIND>(x[2], x[3]));
  }
}

// ==========================================================================================
// Head: last linear layer (<= 8 outputs) in fp32 + SAC policy head (offpolicy.py:116-140)
// ==========================================================================================
constexpr int HEAD_MAX_OUT = 8;

template <typename T>
__device__ __forceinline__ float to_f32(T x);
template <>
__device__ __forceinline__ float to_f32<float>(float x) { return x; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <>
__device__ __forceinline__ float to_f32<__half>(__half x) { return __half2float(x); }

__device__ __forceinline__ float softplus_f(float x) {  // F.softplus, threshold 20
  return x > 20.f ? x : log1pf(expf(x));
}

template <typename T>
__global__ void __launch_bounds__(256) head_kernel(const T* __restrict__ h, int ldh, int k,
                                                   const float* __restrict__ w, const float* __restrict__ b,
                                                   int n_out, const int* __restrict__ n_dev, int n_max,
                                                   float prob, const float* __restrict__ eps,
                                                   float* __restrict__ action, float* __restrict__ logp,
                                                   float* __restrict__ pre) {
  extern __shared__ float s_w[];  // [n_out][k]
  for (int t = threadIdx.x; t < n_out * k; t += blockDim.x) s_w[t] = w[t];
  __syncthreads();
  int n = n_dev ? *n_dev : n_max;
  n = min(n, n_max);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warps_total = gridDim.x * (blockDim.x >> 5);
  const int A = n_out >> 1;
  for (int r = blockIdx.x * (blockDim.x >> 5) + warp; r < n; r += warps_total) {
    float acc[HEAD_MAX_OUT];
#pragma unroll
    for (int o = 0; o < HEAD_MAX_OUT; ++o) acc[o] = 0.f;
    const T* row = h + (size_t)r * ldh;
    for (int c = lane; c < k; c += 32) {
      const float x = to_f32<T>(row[c]);
#pragma unroll
      for (int o = 0; o < HEAD_MAX_OUT; ++o)
        if (o < n_out) acc[o] = fmaf(x, s_w[o * k + c], acc[o]);
    }
#pragma unroll
    for (int o = 0; o < HEAD_MAX_OUT; ++o)
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], off);
    if (lane == 0) {
      float lp = 0.f;
#pragma unroll
      for (int o = 0; o < HEAD_MAX_OUT; ++o)
        if (o < n_out) {
          acc[o] += b[o];
          if (pre) pre[(size_t)r * n_out + o] = acc[o];
        }
#pragma unroll
      for (int a = 0; a < HEAD_MAX_OUT / 2; ++a) {
        if (a >= A) break;
        const float mu = acc[a];
        const float log_std = fminf(fmaxf(acc[A + a], -20.f), 2.f);
        const float std = expf(log_std) * prob;
        const float e = eps ? eps[(size_t)r * A + a] : 0.f;
        const float pi = eps ? fmaf(std, e, mu) : mu;
        if (logp) {
          // Normal(mu,std).log_prob(pi) and the tanh correction of offpolicy.py:131-135
          const float z = pi - mu;
          lp += -(z * z) / (2.f * std * std) - logf(std) - 0.9189385332046727f;
          lp -= 2.f * (0.6931471805599453f - pi - softplus_f(-2.f * pi));
        }
        action[(size_t)r * A + a] = tanhf(pi);
      }
      if (logp) logp[r] = lp;
    }
  }
}

// Sums the per-n-tile partials of the fused head (ttl_head_tree_sum: the same additions in the same order
// whatever tile width the launch used), adds the bias and applies the policy head.  One thread per row.
__global__ void __launch_bounds__(256) head_finish_kernel(const float* __restrict__ partial, int n_tiles,
                                                          int tiles_per_256,
                                                          const float* __restrict__ b, int n_out,
                                                          const int* __restrict__ n_dev, int n_max,
                                                          float prob, const float* __restrict__ eps,
                                                          float* __restrict__ action,
                                                          float* __restrict__ logp, float* __restrict__ pre) {
  int n = n_dev ? *n_dev : n_max;
  n = min(n, n_max);
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  float acc[8];
  const float* prow = partial + (size_t)r * n_tiles * 8;
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = o < n_out ? ttl_head_tree_sum(prow, n_tiles, tiles_per_256, o) : 0.f;
  const int A = n_out >> 1;
  float lp = 0.f;
#pragma unroll
  for (int o = 0; o < 8; ++o)
    if (o < n_out) {
      acc[o] += b[o];
      if (pre) pre[(size_t)r * n_out + o] = acc[o];
    }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    if (a >= A) break;
    const float mu = acc[a];
    float ls = 0.f;
#pragma unroll
    for (int o = 0; o < 8; ++o)
      if (o == A + a) ls = acc[o];
    const float log_std = fminf(fmaxf(ls, -20.f), 2.f);
    const float std = expf(log_std) * prob;
    const float e = eps ? eps[(size_t)r * A + a] : 0.f;
    const float pi = eps ? fmaf(std, e, mu) : mu;
    if (logp) {
      const float z = pi - mu;
      lp += -(z * z) / (2.f * std * std) - logf(std) - 0.9189385332046727f;
      lp -= 2.f * (0.6931471805599453f - pi - softplus_f(-2.f * pi));
    }
    action[(size_t)r * A + a] = tanhf(pi);
  }
  if (logp) logp[r] = lp;
}

// ==========================================================================================
// fp32 tier: plain tiled SGEMM on CUDA cores (reference precision)
// ==========================================================================================
constexpr int SG_T = 64, SG_K = 16;
__global__ void __launch_bounds__(256) dense_f32_kernel(const float* __restrict__ A, int lda,
                                                        const float* __restrict__ W,
                                                        const float* __restrict__ bias,
                                                        float* __restrict__ C, int ldc, int m, int n,
                                                        int k, int relu) {
  __shared__ float sA[SG_K][SG_T + 1];
  __shared__ float sB[SG_K][SG_T + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * SG_T, n0 = blockIdx.x * SG_T;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < k; k0 += SG_K) {
    for (int t = threadIdx.x; t < SG_T * SG_K; t += 256) {
      const int r = t / SG_K, c = t - r * SG_K;
      sA[c][r] = (m0 + r < m && k0 + c < k) ? A[(size_t)(m0 + r) * lda + k0 + c] : 0.f;
      sB[c][r] = (n0 + r < n && k0 + c < k) ? W[(size_t)(n0 + r) * k + k0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SG_K; ++kk) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sA[kk][ty * 4 + i]; bb[i] = sB[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = m0 + ty * 4 + i, c = n0 + tx * 4 + j;
      if (r < m && c < n) {
        float x = acc[i][j] + bias[c];
        if (relu) x = fmaxf(x, 0.f);
        C[(size_t)r * ldc + c] = x;
      }
    }
}

// ==========================================================================================
// Host side: TMA descriptors, plan
// ==========================================================================================
// row-major [rows][cols] tensor of KIND elements, box = [box_rows][128 bytes], 128-byte swizzle.
// pitch: elements between consecutive rows (0 = cols).
int make_tmap(CUtensorMap* map, int kind, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows,
              uint64_t pitch = 0) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return TTL_ERR_DRIVER;
  const int es = kind_esize(kind);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {(pitch ? pitch : cols) * (uint64_t)es};
  cuuint32_t box[2] = {(cuuint32_t)kind_bk(kind), box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = kind == KIND_TF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : (kind == KIND_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                     : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  CUresult r = fn(map, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : TTL_ERR_DRIVER;
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

int g_num_sms = 0;
int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

// A/B switches (ttl_actor_options or the environment): bit 0 = one launch per layer instead of one
// for the whole network (TTL_ACTOR_FUSED=0); bits 8.. = pin the N tile to 256 / 128 / 64
// (TTL_ACTOR_BN; default: chosen from the row count).
std::atomic<int> g_actor_opts{-1};
int actor_opts() {
  int v = g_actor_opts.load(std::memory_order_relaxed);
  if (v < 0) {
    v = 0;
    const char* e = getenv("TTL_ACTOR_FUSED");
    if (e && e[0] == '0') v |= 1;
    e = getenv("TTL_ACTOR_BN");
    const int bn = e ? atoi(e) : 0;
    if (bn == 256 || bn == 128 || bn == 64) v |= bn << 8;
    g_actor_opts.store(v);
  }
  return v;
}
bool fused_layers() { return !(actor_opts() & 1); }
int forced_bn() { return actor_opts() >> 8; }

constexpr int kMaxSmem = 232448;   // 227 KB opt-in limit per CTA on sm_100

int kind_of_precision(int precision) {
  switch (precision) {
    case TTL_PRECISION_BF16: return KIND_BF16;
    case TTL_PRECISION_FP16: return KIND_F16;
    case TTL_PRECISION_TF32: return KIND_TF32;
    default: return -1;
  }
}
int bn_index(int bn) { return bn == 256 ? 0 : (bn == 128 ? 1 : 2); }

// N tile for a launch over up to m_max rows: the widest tile that still gives every cluster work
int choose_bn(int m_max, int n_pad_max) {
  if (forced_bn()) return forced_bn();
  const int n_m = ttl_div_up(m_max, 2 * MLP_BM), nc = num_sms() / 2;
  for (int bn = 256; bn > 64; bn >>= 1)
    if (n_m * ttl_div_up(n_pad_max, bn) * 2 > nc) return bn;   // at least half the clusters busy
  return 64;
}

template <int KIND>
int launch_mlp_kind(const MlpMaps& maps, const MlpArgs& a, int grid, int smem, bool head, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(mlp_pair_kernel<KIND, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(mlp_pair_kernel<KIND, MLP_HEAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const char* name = a.n_layers > 1 ? (head ? "mlp_fused_head_kernel" : "mlp_fused_kernel")
                                    : (head ? "dense_head_kernel" : "dense_kernel");
  if (head)
    TTL_LAUNCH(name, s, ttl_launch_chain(mlp_pair_kernel<KIND, MLP_HEAD>, grid, MLP_THREADS, smem, s, maps, a));
  else
    TTL_LAUNCH(name, s, ttl_launch_chain(mlp_pair_kernel<KIND, 0>, grid, MLP_THREADS, smem, s, maps, a));
  TTL_CHECK_LAST();
  return 0;
}

// Fills the launch geometry (stages, groups, grid) and launches.  `a` comes with everything else set.
int launch_mlp(int kind, const MlpMaps& maps, MlpArgs a, cudaStream_t s) {
  const int nc = num_sms() / 2;
  const int n_m = ttl_div_up(a.m_max, 2 * MLP_BM);
  int n_n_max = 1, total = 0, max_np = 0;
  for (int l = 0; l < a.n_layers; ++l) {
    const int n_n = ttl_div_up(a.n_pad[l], a.bn);
    n_n_max = n_n > n_n_max ? n_n : n_n_max;
    total += n_m * n_n;
    max_np = a.n_pad[l] > max_np ? a.n_pad[l] : max_np;
  }
  if (total <= 0) return 0;
  a.bias_stride = max_np;
  const bool head = a.head_w != nullptr;
  const int extra = 4 * (a.n_layers * a.bias_stride + (head ? a.head_n * a.n_pad[a.n_layers - 1] : 0));
  a.n_stages = 6;
  while (a.n_stages > 2 && a.n_stages * MLP_STAGE_BYTES + 1024 + MLP_BAR_BYTES + extra > kMaxSmem) --a.n_stages;
  const int smem = a.n_stages * MLP_STAGE_BYTES + 1024 + MLP_BAR_BYTES + extra;
  if (smem > kMaxSmem) return TTL_ERR_UNSUPPORTED;
  // groups of m-tiles worth about two tile waves, balanced
  const int g0 = ttl_div_up(2 * nc, n_n_max) > 0 ? ttl_div_up(2 * nc, n_n_max) : 1;
  const int n_groups = ttl_div_up(n_m, g0);
  a.group_m = ttl_div_up(n_m, n_groups);
  const int clusters = total < nc ? total : nc;
  const int grid = 2 * clusters;
  switch (kind) {
    case KIND_BF16: return launch_mlp_kind<KIND_BF16>(maps, a, grid, smem, head, s);
    case KIND_F16: return launch_mlp_kind<KIND_F16>(maps, a, grid, smem, head, s);
    case KIND_TF32: return launch_mlp_kind<KIND_TF32>(maps, a, grid, smem, head, s);
  }
  return TTL_ERR_BAD_ARG;
}

}  // namespace

struct ttl_actor_plan {
  ttl_actor_weights w;
  int max_rows;
  int precision;                     // TTL_PRECISION_*
  int kind;                          // KIND_* of the tensor-core tiers, -1 for fp32
  int k_pad[TTL_ACTOR_MAX_LAYERS];   // padded fan-in of layer i  (whole 128-byte rows)
  int n_pad[TTL_ACTOR_MAX_LAYERS];   // padded fan-out of layer i (= k_pad[i+1], multiple of 64)
  void* wq[TTL_ACTOR_MAX_LAYERS];
  float* bq[TTL_ACTOR_MAX_LAYERS];
  void* act_in;                      // packed first-layer operand rows [max_rows][k_pad[0]] (ttl_actor_forward)
  void* act[2];                      // ping-pong activations [max_rows][act_pitch]: ONE pitch for every layer, so
                                     // that a row occupies the same bytes whichever layer wrote it -- in the
                                     // fused launch layers run concurrently on different rows of these buffers
  int act_pitch;
  float* f32[2];                     // fp32-tier scratch [F32_CHUNK][max_width]
  float* head_partial;               // fused head partials [max_rows][16][8]
  unsigned* flags;                   // inter-layer dependency counts + ticket (mlp_pair_kernel)
  int flag_stride;
  unsigned* overflow;                // fp16 saturation flag
  bool fuse_head;
  int last_tiles, last_tiles_per_256;   // geometry of the partials the last forward left
  int max_kpad, max_width;
  CUtensorMap map_w[TTL_ACTOR_MAX_LAYERS][3];   // W boxes for bn = 256 / 128 / 64
  void* w0_alt;                                 // first-layer weights for bf16_layout 1
  CUtensorMap map_w0_alt[3];
  bool has_alt;
  CUtensorMap map_a[TTL_ACTOR_MAX_LAYERS];  // A operand of layer i
  // first-layer operand maps for caller-owned state buffers (ttl_actor_forward_packed)
  struct ExtMap { const void* ptr; int rows; CUtensorMap map; };
  std::vector<ExtMap> ext_maps;
};

namespace {
constexpr int F32_CHUNK = 8192;
constexpr int kHeadTilesMax = 16;

struct Layout {
  int64_t total;
  int64_t off_w[TTL_ACTOR_MAX_LAYERS], off_b[TTL_ACTOR_MAX_LAYERS], off_act_in, off_act[2], off_f32[2], off_hp,
      off_w0_alt, off_flags;
  int act_pitch;
  int k_pad[TTL_ACTOR_MAX_LAYERS], n_pad[TTL_ACTOR_MAX_LAYERS];
  int max_kpad, max_width, flag_stride;
};

int plan_layout(const ttl_actor_weights* w, int max_rows, int precision, Layout* L) {
  if (!w || w->n_layers < 2 || w->n_layers > TTL_ACTOR_MAX_LAYERS || max_rows <= 0) return TTL_ERR_BAD_ARG;
  if (w->out_dim[w->n_layers - 1] > HEAD_MAX_OUT || (w->out_dim[w->n_layers - 1] & 1)) return TTL_ERR_UNSUPPORTED;
  const int kind = kind_of_precision(precision);
  if (kind < 0 && precision != TTL_PRECISION_FP32) return TTL_ERR_BAD_ARG;
  const int es = kind < 0 ? 4 : kind_esize(kind);
  int64_t off = 0;
  auto take = [&](int64_t bytes) { int64_t o = off; off += (bytes + 1023) / 1024 * 1024; return o; };
  L->max_kpad = 0;
  L->max_width = 0;
  for (int i = 0; i < w->n_layers; ++i) {
    if (i > 0 && w->in_dim[i] != w->out_dim[i - 1]) return TTL_ERR_BAD_ARG;
    // fan-in padded to 64 for every kind so that k_pad[i+1] == n_pad[i] (the 64-column head groups)
    L->k_pad[i] = round_up(w->in_dim[i], 64);
    L->n_pad[i] = round_up(w->out_dim[i], 64);
    if (L->k_pad[i] > L->max_kpad) L->max_kpad = L->k_pad[i];
    if (w->in_dim[i] > L->max_width) L->max_width = w->in_dim[i];
    if (w->out_dim[i] > L->max_width) L->max_width = w->out_dim[i];
  }
  L->flag_stride = ttl_div_up(max_rows, 2 * MLP_BM) + 1;
  for (int i = 0; i < w->n_layers - 1; ++i) {
    L->off_w[i] = kind < 0 ? 0 : take((int64_t)L->n_pad[i] * L->k_pad[i] * es);
    L->off_b[i] = kind < 0 ? 0 : take((int64_t)round_up(L->n_pad[i], 256) * 4);
  }
  L->act_pitch = 0;
  for (int i = 0; i < w->n_layers - 1; ++i) L->act_pitch = L->n_pad[i] > L->act_pitch ? L->n_pad[i] : L->act_pitch;
  L->off_act_in = kind < 0 ? 0 : take((int64_t)max_rows * L->k_pad[0] * es);
  for (int j = 0; j < 2; ++j) L->off_act[j] = kind < 0 ? 0 : take((int64_t)max_rows * L->act_pitch * es);
  for (int j = 0; j < 2; ++j) L->off_f32[j] = kind < 0 ? take((int64_t)F32_CHUNK * L->max_width * 4) : 0;
  L->off_hp = kind < 0 ? 0 : take((int64_t)max_rows * kHeadTilesMax * 8 * 4);
  L->off_w0_alt = kind < 0 ? 0 : take((int64_t)L->n_pad[0] * L->k_pad[0] * es);
  L->off_flags = take((int64_t)(TTL_ACTOR_MAX_LAYERS * L->flag_stride + 8) * 4);
  L->total = off;
  return 0;
}

template <int KIND>
void pack_weights_kind(ttl_actor_plan* p, int i, cudaStream_t s) {
  const ttl_actor_weights& w = p->w;
  const long long tot = (long long)p->n_pad[i] * p->k_pad[i];
  TTL_LAUNCH("pack_weight_kernel", s,
             pack_weight_kernel<KIND><<<ttl_div_up(tot, 256), 256, 0, s>>>(w.w[i], p->wq[i], w.out_dim[i], w.in_dim[i],
                                                                         p->n_pad[i], p->k_pad[i]));
}
void pack_weights(ttl_actor_plan* p, cudaStream_t s) {
  const ttl_actor_weights& w = p->w;
  for (int i = 0; i < w.n_layers - 1; ++i) {
    if (p->kind == KIND_BF16) pack_weights_kind<KIND_BF16>(p, i, s);
    else if (p->kind == KIND_F16) pack_weights_kind<KIND_F16>(p, i, s);
    else pack_weights_kind<KIND_TF32>(p, i, s);
    const int bp = round_up(p->n_pad[i], 256);
    TTL_LAUNCH("pack_bias_kernel", s, pack_bias_kernel<<<ttl_div_up(bp, 256), 256, 0, s>>>(w.b[i], p->bq[i], w.out_dim[i], bp));
  }
}

// Hidden layers on tensor cores (the last one carries the fused head when possible) + head.
// map_a0: TMA map of the first layer's operand rows [rows][k_pad[0]].
int run_tc_layers(ttl_actor_plan* p, const CUtensorMap& map_a0, const int32_t* n_rows_dev, int32_t n_rows_max,
                  float probabilistic, const float* eps, float* action, float* logp, float* pre, cudaStream_t s,
                  bool alt_w0 = false) {
  const ttl_actor_weights& w = p->w;
  const int nl = w.n_layers, nh = nl - 1;     // nh tensor-core layers
  const int n_out = w.out_dim[nl - 1], k_last = w.in_dim[nl - 1];
  int max_np = 0;
  for (int i = 0; i < nh; ++i) max_np = p->n_pad[i] > max_np ? p->n_pad[i] : max_np;
  const int bn = choose_bn(n_rows_max, max_np);
  const int bi = bn_index(bn);
  // only mu is needed when nothing reads log_std: deterministic policy, no log-prob, no raw output (with
  // action == NULL, probabilistic != 0 leaves the log_std partials for the policy the env step samples)
  const int head_n = (p->fuse_head && probabilistic == 0.f && !logp && !pre) ? n_out / 2 : n_out;

  auto fill_layer = [&](MlpMaps& maps, MlpArgs& a, int slot, int i) {
    maps.a[slot] = i == 0 ? map_a0 : p->map_a[i];
    maps.w[slot] = (alt_w0 && i == 0) ? p->map_w0_alt[bi] : p->map_w[i][bi];
    a.kblocks[slot] = p->k_pad[i] / kind_bk(p->kind);
    a.n_pad[slot] = p->n_pad[i];
    a.ldc[slot] = p->act_pitch;
    a.C[slot] = p->act[(i + 1) & 1];
    a.bias[slot] = p->bq[i];
  };
  auto base_args = [&]() {
    MlpArgs a;
    memset(&a, 0, sizeof(a));
    a.bn = bn;
    a.m_dev = n_rows_dev;
    a.m_max = n_rows_max;
    a.flags = p->flags;
    a.flag_stride = p->flag_stride;
    a.overflow = p->overflow;
    return a;
  };
  auto add_head = [&](MlpArgs& a) {
    a.head_w = w.w[nl - 1];
    a.head_k = k_last;
    a.head_n = head_n;
    a.head_partial = p->head_partial;
    p->last_tiles = ttl_div_up(p->n_pad[nh - 1], bn);
    p->last_tiles_per_256 = 256 / bn;
  };
  if (fused_layers() && nh <= MLP_MAX_LAYERS) {
    MlpMaps maps;
    MlpArgs a = base_args();
    a.n_layers = nh;
    for (int i = 0; i < nh; ++i) fill_layer(maps, a, i, i);
    a.relu_mask = (1 << nh) - 1;
    if (p->fuse_head) add_head(a);
    int rc = launch_mlp(p->kind, maps, a, s);
    if (rc) return rc;
  } else {
    for (int i = 0; i < nh; ++i) {
      MlpMaps maps;
      MlpArgs a = base_args();
      a.n_layers = 1;
      fill_layer(maps, a, 0, i);
      a.relu_mask = 1;
      if (p->fuse_head && i == nh - 1) add_head(a);
      int rc = launch_mlp(p->kind, maps, a, s);
      if (rc) return rc;
    }
  }
  if (p->fuse_head && !action) return 0;   // the caller reads the partial sums (ttl_actor_head_partial)
  if (p->fuse_head) {
    TTL_LAUNCH("head_finish_kernel", s,
               head_finish_kernel<<<ttl_div_up(n_rows_max, 256), 256, 0, s>>>(
                   p->head_partial, p->last_tiles, p->last_tiles_per_256, w.b[nl - 1], n_out, n_rows_dev,
                   n_rows_max, probabilistic, eps, action, logp, pre));
  } else {
    const size_t head_smem = (size_t)n_out * k_last * sizeof(float);
    const int head_grid = num_sms() * 2;
    static bool head_attr = false;
    if (!head_attr) {
      cudaFuncSetAttribute(head_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      cudaFuncSetAttribute(head_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      cudaFuncSetAttribute(head_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      head_attr = true;
    }
    const void* h = p->act[nh & 1];
    if (p->kind == KIND_BF16)
      TTL_LAUNCH("head_kernel", s, head_kernel<__nv_bfloat16><<<head_grid, 256, head_smem, s>>>(
          static_cast<const __nv_bfloat16*>(h), p->act_pitch, k_last, w.w[nl - 1], w.b[nl - 1], n_out, n_rows_dev,
          n_rows_max, probabilistic, eps, action, logp, pre));
    else if (p->kind == KIND_F16)
      TTL_LAUNCH("head_kernel", s, head_kernel<__half><<<head_grid, 256, head_smem, s>>>(
          static_cast<const __half*>(h), p->act_pitch, k_last, w.w[nl - 1], w.b[nl - 1], n_out, n_rows_dev,
          n_rows_max, probabilistic, eps, action, logp, pre));
    else
      TTL_LAUNCH("head_kernel", s, head_kernel<float><<<head_grid, 256, head_smem, s>>>(
          static_cast<const float*>(h), p->act_pitch, k_last, w.w[nl - 1], w.b[nl - 1], n_out, n_rows_dev,
          n_rows_max, probabilistic, eps, action, logp, pre));
  }
  TTL_CHECK_LAST();
  return 0;
}

// fp32 state rows -> the plan's first-layer operand rows (ttl_actor_forward on the tensor-core tiers)
void pack_state(ttl_actor_plan* p, const float* state, int ld_state, const int32_t* n_rows_dev, int n_rows_max,
                cudaStream_t s) {
  const long long tot = (long long)n_rows_max * (p->k_pad[0] >> 2);
  const int grid = ttl_div_up(tot, 256);
  const int width = p->w.in_dim[0];
  if (p->kind == KIND_BF16)
    TTL_LAUNCH("pack_state_kernel", s, pack_state_kernel<KIND_BF16><<<grid, 256, 0, s>>>(
        state, ld_state, width, n_rows_dev, n_rows_max, p->act_in, p->k_pad[0], p->overflow));
  else if (p->kind == KIND_F16)
    TTL_LAUNCH("pack_state_kernel", s, pack_state_kernel<KIND_F16><<<grid, 256, 0, s>>>(
        state, ld_state, width, n_rows_dev, n_rows_max, p->act_in, p->k_pad[0], p->overflow));
  else
    TTL_LAUNCH("pack_state_kernel", s, pack_state_kernel<KIND_TF32><<<grid, 256, 0, s>>>(
        state, ld_state, width, n_rows_dev, n_rows_max, p->act_in, p->k_pad[0], p->overflow));
}

// TMA map of caller-owned operand rows (ttl_actor_forward_packed), cached per (pointer, rows)
int ext_map(ttl_actor_plan* p, const void* state_op, int ld, int rows_alloc, const CUtensorMap** out) {
  for (auto& e : p->ext_maps)
    if (e.ptr == state_op && e.rows == rows_alloc) { *out = &e.map; return 0; }
  if (p->ext_maps.size() >= 16) p->ext_maps.clear();
  ttl_actor_plan::ExtMap e;
  e.ptr = state_op;
  e.rows = rows_alloc;
  int rc = make_tmap(&e.map, p->kind, state_op, (uint64_t)rows_alloc, (uint64_t)ld, MLP_BM);
  if (rc) return rc;
  p->ext_maps.push_back(e);
  *out = &p->ext_maps.back().map;
  return 0;
}
}  // namespace

extern "C" {

int64_t ttl_actor_workspace_bytes(const ttl_actor_weights* w, int32_t max_rows, int32_t precision) {
  Layout L;
  if (plan_layout(w, max_rows, precision, &L)) return -1;
  return L.total;
}

int ttl_actor_plan_create(ttl_actor_plan** out, const ttl_actor_weights* w, int32_t max_rows, int32_t precision,
                          void* workspace, int64_t workspace_bytes, void* stream) {
  if (!out || !workspace) return TTL_ERR_BAD_ARG;
  Layout L;
  int rc = plan_layout(w, max_rows, precision, &L);
  if (rc) return rc;
  if (workspace_bytes < L.total || (reinterpret_cast<uintptr_t>(workspace) & 1023)) return TTL_ERR_BAD_ARG;
  ttl_actor_plan* p = new (std::nothrow) ttl_actor_plan();
  if (!p) return TTL_ERR_BAD_ARG;
  p->w = *w;
  p->max_rows = max_rows;
  p->precision = precision;
  p->kind = kind_of_precision(precision);
  p->max_kpad = L.max_kpad;
  p->max_width = L.max_width;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  cudaStream_t s = (cudaStream_t)stream;
  const int nl = w->n_layers;
  for (int i = 0; i < nl; ++i) { p->k_pad[i] = L.k_pad[i]; p->n_pad[i] = L.n_pad[i]; }
  p->flags = reinterpret_cast<unsigned*>(ws + L.off_flags);
  p->flag_stride = L.flag_stride;
  p->overflow = p->flags + (size_t)TTL_ACTOR_MAX_LAYERS * L.flag_stride + 4;
  p->has_alt = false;
  p->fuse_head = false;
  p->last_tiles = 0;
  p->last_tiles_per_256 = 1;
  cudaError_t e = cudaMemsetAsync(p->flags, 0, (size_t)(TTL_ACTOR_MAX_LAYERS * L.flag_stride + 8) * 4, s);
  if (e != cudaSuccess) { delete p; return (int)e; }
  if (p->kind < 0) {   // fp32 tier: CUDA-core layers reading the caller's weights in place
    for (int j = 0; j < 2; ++j) p->f32[j] = reinterpret_cast<float*>(ws + L.off_f32[j]);
    *out = p;
    return 0;
  }
  for (int j = 0; j < 2; ++j) p->act[j] = ws + L.off_act[j];
  p->act_in = ws + L.off_act_in;
  p->act_pitch = L.act_pitch;
  p->head_partial = reinterpret_cast<float*>(ws + L.off_hp);
  p->w0_alt = ws + L.off_w0_alt;
  // the last hidden layer can carry the head when it is 6 wide and the layer fits 16 tiles of 64
  p->fuse_head = w->out_dim[nl - 1] == MLP_HEAD && L.n_pad[nl - 2] <= 1024;
  for (int i = 0; i < nl - 1; ++i) {  // hidden layers run on tensor cores
    p->wq[i] = ws + L.off_w[i];
    p->bq[i] = reinterpret_cast<float*>(ws + L.off_b[i]);
    for (int b = 0; b < 3 && !rc; ++b)
      rc = make_tmap(&p->map_w[i][b], p->kind, p->wq[i], (uint64_t)L.n_pad[i], (uint64_t)L.k_pad[i], 128u >> b);
    // A operand of layer i: the packed state rows (i == 0) or act[i & 1] with the common pitch
    if (!rc)
      rc = i == 0 ? make_tmap(&p->map_a[0], p->kind, p->act_in, (uint64_t)max_rows, (uint64_t)L.k_pad[0], MLP_BM)
                  : make_tmap(&p->map_a[i], p->kind, p->act[i & 1], (uint64_t)max_rows, (uint64_t)L.k_pad[i], MLP_BM,
                              (uint64_t)L.act_pitch);
    if (rc) { delete p; return rc; }
  }
  pack_weights(p, s);
  e = cudaGetLastError();
  if (e != cudaSuccess) { delete p; return (int)e; }
  *out = p;
  return 0;
}

void ttl_actor_plan_destroy(ttl_actor_plan* plan) { delete plan; }

int ttl_actor_forward(ttl_actor_plan* p, const float* state, int32_t ld_state, const int32_t* n_rows_dev,
                      int32_t n_rows_max, float probabilistic, const float* eps, float* action,
                      float* logp, float* pre, void* stream) {
  if (!p || !state || n_rows_max > p->max_rows) return TTL_ERR_BAD_ARG;
  if (!action && (logp || pre || eps || !p->fuse_head || p->kind < 0)) return TTL_ERR_BAD_ARG;
  if (probabilistic != 0.f && !eps && action) return TTL_ERR_BAD_ARG;
  if (n_rows_max <= 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const ttl_actor_weights& w = p->w;
  const int nl = w.n_layers;
  const int n_out = w.out_dim[nl - 1], k_last = w.in_dim[nl - 1];

  if (p->kind >= 0) {
    pack_state(p, state, ld_state, n_rows_dev, n_rows_max, s);
    return run_tc_layers(p, p->map_a[0], n_rows_dev, n_rows_max, probabilistic, eps, action, logp, pre, s);
  }
  // Reference-precision tier; needs the row count on the host.
  const size_t head_smem = (size_t)n_out * k_last * sizeof(float);
  const int head_grid = num_sms() * 2;
  int n = n_rows_max;
  if (n_rows_dev) {
    cudaError_t e = cudaMemcpyAsync(&n, n_rows_dev, sizeof(int), cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) return (int)e;
    e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return (int)e;
    if (n > n_rows_max) n = n_rows_max;
  }
  static bool head_attr32 = false;
  if (!head_attr32 && head_smem > 48 * 1024) {
    cudaFuncSetAttribute(head_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    head_attr32 = true;
  }
  const int A = n_out / 2;
  for (int r0 = 0; r0 < n; r0 += F32_CHUNK) {
    const int m = (n - r0) < F32_CHUNK ? (n - r0) : F32_CHUNK;
    const float* in = state + (size_t)r0 * ld_state;
    int ld_in = ld_state;
    for (int i = 0; i < nl - 1; ++i) {
      float* o = p->f32[i & 1];
      dim3 grid(ttl_div_up(w.out_dim[i], SG_T), ttl_div_up(m, SG_T));
      TTL_LAUNCH("dense_f32_kernel", s, dense_f32_kernel<<<grid, 256, 0, s>>>(in, ld_in, w.w[i], w.b[i], o, p->max_width, m, w.out_dim[i],
                                            w.in_dim[i], 1));
      in = o;
      ld_in = p->max_width;
    }
    TTL_LAUNCH("head_kernel_f32", s, head_kernel<float><<<head_grid, 256, head_smem, s>>>(
        in, ld_in, k_last, w.w[nl - 1], w.b[nl - 1], n_out, nullptr, m, probabilistic,
        eps ? eps + (size_t)r0 * A : nullptr, action + (size_t)r0 * A, logp ? logp + r0 : nullptr,
        pre ? pre + (size_t)r0 * n_out : nullptr));
  }
  TTL_CHECK_LAST();
  return 0;
}

int ttl_actor_forward_packed(ttl_actor_plan* p, const void* state_op, int32_t ld, int32_t rows_alloc,
                             const int32_t* n_rows_dev, int32_t n_rows_max, float probabilistic,
                             const float* eps, float* action, float* logp, float* pre, int32_t layout,
                             void* stream) {
  if (!p || !state_op || p->kind < 0 || n_rows_max > p->max_rows || n_rows_max > rows_alloc) return TTL_ERR_BAD_ARG;
  if (!action && (logp || pre || eps || !p->fuse_head)) return TTL_ERR_BAD_ARG;
  if (layout != 0 && !(layout == 1 && p->has_alt)) return TTL_ERR_BAD_ARG;
  if (ld != p->k_pad[0] || (reinterpret_cast<uintptr_t>(state_op) & 15)) return TTL_ERR_BAD_ARG;
  if (probabilistic != 0.f && !eps && action) return TTL_ERR_BAD_ARG;
  if (n_rows_max <= 0) return 0;
  const CUtensorMap* map = nullptr;
  int rc = ext_map(p, state_op, ld, rows_alloc, &map);
  if (rc) return rc;
  return run_tc_layers(p, *map, n_rows_dev, n_rows_max, probabilistic, eps, action, logp, pre,
                       (cudaStream_t)stream, layout == 1);
}

int ttl_actor_head_partial(const ttl_actor_plan* p, const float** partial, int32_t* n_tiles,
                           int32_t* tiles_per_256, const float** bias) {
  if (!p || !partial || !n_tiles || !tiles_per_256 || !bias) return TTL_ERR_BAD_ARG;
  if (!p->fuse_head) return TTL_ERR_UNSUPPORTED;
  const int nl = p->w.n_layers;
  *partial = p->head_partial;
  *n_tiles = p->last_tiles;
  *tiles_per_256 = p->last_tiles_per_256;
  *bias = p->w.b[nl - 1];
  return 0;
}

int ttl_actor_precision(const ttl_actor_plan* p) { return p ? p->precision : TTL_ERR_BAD_ARG; }

void ttl_actor_options(int32_t bits) {
  const int bn = bits >> 8;
  g_actor_opts.store((bits & 1) | ((bn == 256 || bn == 128 || bn == 64) ? bn << 8 : 0));
}

int ttl_actor_overflow(ttl_actor_plan* p, int32_t* out_host, int32_t clear, void* stream) {
  if (!p || !out_host) return TTL_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned v = 0;
  cudaError_t e = cudaMemcpyAsync(&v, p->overflow, sizeof(v), cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && clear) e = cudaMemsetAsync(p->overflow, 0, sizeof(unsigned), s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return (int)e;
  *out_host = (int32_t)v;
  return 0;
}

int ttl_actor_plan_set_layout(ttl_actor_plan* p, int32_t C, int32_t CP, int32_t n_points, void* stream) {
  if (!p || p->kind < 0 || C <= 0 || CP < C || n_points <= 0) return TTL_ERR_BAD_ARG;
  const int n_in = p->w.in_dim[0];
  if (n_points * C > n_in || n_points * CP + (n_in - n_points * C) > p->k_pad[0]) return TTL_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  const long long tot = (long long)p->n_pad[0] * p->k_pad[0];
  const int grid = ttl_div_up(tot, 256);
  if (p->kind == KIND_BF16)
    TTL_LAUNCH("pack_weight_layout_kernel", s, pack_weight_layout_kernel<KIND_BF16><<<grid, 256, 0, s>>>(
        p->w.w[0], p->w0_alt, p->w.out_dim[0], n_in, p->n_pad[0], p->k_pad[0], C, CP, n_points));
  else if (p->kind == KIND_F16)
    TTL_LAUNCH("pack_weight_layout_kernel", s, pack_weight_layout_kernel<KIND_F16><<<grid, 256, 0, s>>>(
        p->w.w[0], p->w0_alt, p->w.out_dim[0], n_in, p->n_pad[0], p->k_pad[0], C, CP, n_points));
  else
    TTL_LAUNCH("pack_weight_layout_kernel", s, pack_weight_layout_kernel<KIND_TF32><<<grid, 256, 0, s>>>(
        p->w.w[0], p->w0_alt, p->w.out_dim[0], n_in, p->n_pad[0], p->k_pad[0], C, CP, n_points));
  for (int b = 0; b < 3; ++b) {
    int rc = make_tmap(&p->map_w0_alt[b], p->kind, p->w0_alt, (uint64_t)p->n_pad[0], (uint64_t)p->k_pad[0], 128u >> b);
    if (rc) return rc;
  }
  p->has_alt = true;
  TTL_CHECK_LAST();
  return 0;
}

int ttl_actor_plan_refresh(ttl_actor_plan* p, void* stream) {
  // the fp32 weights changed in place (an optimiser step): repack the operand copies
  if (!p) return TTL_ERR_BAD_ARG;
  if (p->kind < 0) return 0;
  pack_weights(p, (cudaStream_t)stream);
  p->has_alt = false;   // ttl_actor_plan_set_layout repacks the permuted first layer on demand
  TTL_CHECK_LAST();
  return 0;
}

int ttl_gemm_tc(const void* A, const void* W, const float* bias, void* C, int32_t m, int32_t n, int32_t k,
                int32_t ldc, int32_t relu, const int32_t* m_dev, int32_t precision, int32_t bn, void* stream) {
  const int kind = kind_of_precision(precision);
  if (kind < 0 || !A || !W || !bias || !C || (k % 64) || (n % 64) || ldc < n || (ldc % 16)) return TTL_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(C) & 31) || (reinterpret_cast<uintptr_t>(bias) & 15) ||
      (bn != 0 && bn != 256 && bn != 128 && bn != 64))
    return TTL_ERR_BAD_ARG;
  if (m <= 0) return 0;
  if (bn == 0) bn = choose_bn(m, n);
  MlpMaps maps;
  int rc = make_tmap(&maps.a[0], kind, A, (uint64_t)m, (uint64_t)k, MLP_BM);
  if (rc) return rc;
  rc = make_tmap(&maps.w[0], kind, W, (uint64_t)n, (uint64_t)k, (uint32_t)(bn / 2));
  if (rc) return rc;
  MlpArgs a;
  memset(&a, 0, sizeof(a));
  a.n_layers = 1;
  a.bn = bn;
  a.kblocks[0] = k / kind_bk(kind);
  a.n_pad[0] = n;
  a.ldc[0] = ldc;
  a.C[0] = C;
  a.bias[0] = bias;      // readable for n floats
  a.m_dev = m_dev;
  a.m_max = m;
  a.relu_mask = relu ? 1 : 0;
  return launch_mlp(kind, maps, a, (cudaStream_t)stream);
}

int ttl_gemm_bf16(const void* A, const void* W, const float* bias, void* C, int32_t m, int32_t n,
                  int32_t k, int32_t ldc, int32_t relu, const int32_t* m_dev, void* stream) {
  return ttl_gemm_tc(A, W, bias, C, m, n, k, ldc, relu, m_dev, TTL_PRECISION_BF16, 0, stream);
}

}  // extern "C"
