// philox.cuh — Philox4x32-10 counter-based streams (this repo's RNG spec; the reference's
// Julia MersenneTwister streams cannot be reproduced).  Restated bit-exactly in
// oracle/shems_oracle.c (oracle_philox).  key = seed, counter = (id_lo, id_hi, ctr, stream).
#pragma once
#include <stdint.h>

enum : uint32_t { STREAM_RESET = 0x5245u, STREAM_ACTION = 0x4143u, STREAM_NOISE = 0x4e4fu, STREAM_SAMPLE = 0x534du, STREAM_INIT = 0x494eu,
                  STREAM_PBT = 0x5042u, STREAM_PER = 0x5052u };

// the 64-bit product of two words.  On the device one mul.wide.u32 (a single IMAD.WIDE.U32): the compiler's lowering of the
// C expression adds a zero high word to every product, one wasted instruction each.
__host__ __device__ __forceinline__ uint64_t mul_wide_u32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  uint64_t p;
  asm("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(a), "r"(b));
  return p;
#else
  return (uint64_t)a * b;
#endif
}

__host__ __device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
  const uint64_t p0 = mul_wide_u32(0xD2511F53u, c0);
  const uint64_t p1 = mul_wide_u32(0xCD9E8D57u, c2);
  const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
  const uint32_t n1 = (uint32_t)p1;
  const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
  const uint32_t n3 = (uint32_t)p0;
  c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__host__ __device__ __forceinline__ void philox4x32_10(uint64_t seed, uint64_t id, uint32_t ctr, uint32_t stream, uint32_t out[4]) {
  uint32_t c0 = (uint32_t)id, c1 = (uint32_t)(id >> 32), c2 = ctr, c3 = stream;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c0, c1, c2, c3, k0, k1);
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// The 10 round keys of a seed, for a kernel that draws many blocks under one seed: passed as a kernel argument, the rounds read
// them as constant-bank operands instead of adding the Weyl increments per thread and call.
struct PhiloxKeys { uint32_t k0[10], k1[10]; };
inline PhiloxKeys philox_keys(uint64_t seed) {
  PhiloxKeys K;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r, k0 += 0x9E3779B9u, k1 += 0xBB67AE85u) { K.k0[r] = k0; K.k1[r] = k1; }
  return K;
}
// philox4x32_10(seed, id, ctr, stream, out) with K = philox_keys(seed)
__device__ __forceinline__ void philox4x32_10(const PhiloxKeys& K, uint64_t id, uint32_t ctr, uint32_t stream, uint32_t out[4]) {
  uint32_t c0 = (uint32_t)id, c1 = (uint32_t)(id >> 32), c2 = ctr, c3 = stream;
#pragma unroll
  for (int r = 0; r < 10; ++r) philox_round(c0, c1, c2, c3, K.k0[r], K.k1[r]);
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// 53-bit uniform in [0,1) from two words (stands in for Julia's Float64 rand())
__host__ __device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return (double)((((uint64_t)(a >> 5)) << 26) | (uint64_t)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// a random action component from one word w: Float32(2u - 1) with u = w * 2^-32 (memory_plotting_saving.jl:14-19), without Float64.
// 2u - 1 = (w - 2^31) * 2^-31; w ^ 2^31 read as a signed word is w - 2^31, its conversion rounds it once to Float32 (round to
// nearest even), and the scaling by 2^-31 is exact (|w - 2^31| is 0 or >= 1).  So this equals RN32(2u - 1), what the Float64
// expression Float32(fma(1 + u, 2, -3)) gives; tests/test_action_decode.py checks all 2^32 words against it.
__host__ __device__ __forceinline__ float action_from_word(uint32_t w) { return (float)(int32_t)(w ^ 0x80000000u) * 0x1p-31f; }
