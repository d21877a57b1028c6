// The keyed noise stream of the sampler kernels (include/diffpose_b200.h, "Keyed noise"): Philox4x32-10 (Salmon et al.,
// SC'11; the round function and constants of Random123 / cuRAND Philox4_32_10) with a Box-Muller transform.
//
//   key     (seed & 0xffffffff, seed >> 32)
//   counter (e >> 2, s, b, h): element e = joint * c + coord, step s, global pose b, hypothesis h
//   z       with x = Philox(counter, key), l = e & 3, m = l >> 1:
//           u1 = ((x[2m] >> 8) + 1) 2^-24 in (0, 1],  u2 = (x[2m+1] >> 8) 2^-24 in [0, 1)
//           z  = sqrtf(-2 logf(u1)) * (l even ? cospif(2 u2) : sinpif(2 u2))
//
// Every operation is IEEE-rounded (logf, sqrtf, sincospif, __fmul_rn; no fast-math intrinsics), so the value of an element
// does not depend on which kernel computes it: a keyed sampler call equals the same call fed dp_noise_fill's output.
#pragma once
#include <cstdint>

namespace dp {

// The key of one call as the kernels receive it (by value, so a keyed launch stays graph capturable).
struct NoiseKey {
  uint32_t k0, k1;         // seed & 0xffffffff, seed >> 32
  uint32_t pose_offset;    // b = pose_offset + local pose
  uint32_t step_offset;    // s = step_offset + execution index of the step
  int on;                  // 0: no keyed noise (the noise pointer, if any, is used)
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
  }
  return c;
}

// The Philox output quad that holds elements 4q .. 4q+3 of row (b, h) at step s.
__device__ __forceinline__ uint4 philox_quad(const NoiseKey& key, uint32_t s, uint32_t b, uint32_t h, uint32_t q) {
  return philox4x32_10(make_uint4(q, s, b, h), key.k0, key.k1);
}

// Box-Muller of lane l = e & 3 of a quad.
__device__ __forceinline__ float philox_box_muller(uint4 x, uint32_t l) {
  const uint32_t wa = (l & 2u) ? x.z : x.x, wb = (l & 2u) ? x.w : x.y;
  const float u1 = __fmul_rn((float)((wa >> 8) + 1u), 0x1p-24f);   // exact: at most 24 significant bits
  const float u2 = __fmul_rn((float)(wb >> 8), 0x1p-24f);
  const float r = sqrtf(__fmul_rn(-2.0f, logf(u1)));
  float sn, cs;
  sincospif(__fmul_rn(2.0f, u2), &sn, &cs);
  return __fmul_rn(r, (l & 1u) ? sn : cs);
}

// z of element e of row (b, h) at step s; s and b are the global indices (offsets already added).
__device__ __forceinline__ float philox_normal(const NoiseKey& key, uint32_t s, uint32_t b, uint32_t h, uint32_t e) {
  return philox_box_muller(philox_quad(key, s, b, h, e >> 2), e & 3u);
}

}  // namespace dp
