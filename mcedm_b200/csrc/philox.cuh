// Counter-based Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123
// constants and round function) and the dropout mask of the training forward built on it.
//
// Mask of one UNetBlock's conv1 operand (DESIGN.md §3): element (b, y, x, c) of the block at H x W has the LOGICAL NHWC
// index n = ((b*H + y)*W + x)*64 + c, whatever layout (dense or padded-flat) stores it; with
//   ctr = (uint32(n >> 2), uint32(n >> 34), layer, step),  key = (seed_lo, seed_hi)
// it is kept iff output word (n & 3) of philox(ctr, key) is >= the threshold T = min(2^32 - 1, floor(p * 2^32)).
// One call covers 4 consecutive channels.  `rng` points at three device words {seed_lo, seed_hi, step}, so a replayed
// CUDA graph sees the values the host wrote before the replay.
#pragma once
#include <cstdint>

namespace mcedm {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// the four mask words of logical elements 4q .. 4q+3 (q = n >> 2) of layer `layer`
__device__ __forceinline__ uint4 dropout_words(unsigned long long q, int layer, const uint32_t* __restrict__ rng) {
  return philox4x32_10(make_uint4((uint32_t)q, (uint32_t)(q >> 32), (uint32_t)layer, __ldg(rng + 2)), __ldg(rng),
                       __ldg(rng + 1));
}

// v * s where the word is >= thr, else 0 (one fp32 multiply; the caller rounds once to 16 bits)
__device__ __forceinline__ float4 dropout_apply4(float4 v, uint4 w, uint32_t thr, float s) {
  v.x = w.x >= thr ? v.x * s : 0.f;
  v.y = w.y >= thr ? v.y * s : 0.f;
  v.z = w.z >= thr ? v.z * s : 0.f;
  v.w = w.w >= thr ? v.w * s : 0.f;
  return v;
}

}  // namespace mcedm
