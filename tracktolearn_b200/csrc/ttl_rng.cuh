// Counter-based Gaussian draws for the device-side tracking noise (ttl_noise, include/ttl_b200.h).
//
// One standard normal per (seed, global seed index g, point count L, component c):
//   (w0, w1, w2, w3) = Philox4x32-10(counter = (lo32(g), hi32(g), L, c), key = (lo32(seed), hi32(seed)))
//   u1 = (((w1 << 32 | w0) >> 12) + 0.5) * 2^-52      exact in fp64, in (0, 1)
//   u2 = (((w3 << 32 | w2) >> 12) + 0.5) * 2^-52
//   z  = sqrt(-2 ln u1) * cos(2 pi u2)                 |z| <= sqrt(106 ln 2) = 8.58
// A pure function of its arguments: a streamline's noise does not depend on where it sits in the alive
// list, on how many streamlines are tracked at once or on which GPU tracks it.  tests/noise_oracle.py
// restates it in numpy (philox4x32_10, philox_normals).
#pragma once
#include <stdint.h>

// Philox4x32-10 (Salmon et al., SC'11) with the Random123 constants.
__device__ __forceinline__ uint4 ttl_philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t kM0 = 0xD2511F53u, kM1 = 0xCD9E8D57u, kW0 = 0x9E3779B9u, kW1 = 0xBB67AE85u;
#pragma unroll
  for (int round = 0; round < 10; ++round) {
    const uint32_t hi0 = __umulhi(kM0, ctr.x), lo0 = kM0 * ctr.x;
    const uint32_t hi1 = __umulhi(kM1, ctr.z), lo1 = kM1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += kW0;
    key.y += kW1;
  }
  return ctr;
}

// (hi:lo >> 12) + 0.5 scaled by 2^-52: 52 random bits, never 0 or 1
__device__ __forceinline__ double ttl_open_unit(uint32_t lo, uint32_t hi) {
  const unsigned long long v = ((unsigned long long)hi << 32 | lo) >> 12;
  return __dmul_rn(__dadd_rn((double)v, 0.5), 0x1p-52);
}

// z_c(seed, g, L) of the definition above (Box-Muller, cosine branch), fp64
__device__ __forceinline__ double ttl_noise_normal(unsigned long long seed, long long g, int L, int c) {
  const unsigned long long ug = (unsigned long long)g;
  const uint4 w = ttl_philox4x32_10(make_uint4((uint32_t)ug, (uint32_t)(ug >> 32), (uint32_t)L, (uint32_t)c),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const double u1 = ttl_open_unit(w.x, w.y), u2 = ttl_open_unit(w.z, w.w);
  return __dmul_rn(__dsqrt_rn(__dmul_rn(-2.0, log(u1))), cospi(__dmul_rn(2.0, u2)));
}

// eps_c of the stochastic policy (ttl_policy, include/ttl_b200.h): counter words 3..5, so that it is
// independent of the tracking noise (words 0..2) under the same seed; rounded once to fp32
__device__ __forceinline__ float ttl_policy_eps(unsigned long long seed, long long g, int L, int c) {
  return (float)ttl_noise_normal(seed, g, L, 3 + c);
}
