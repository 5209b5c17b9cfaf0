// Action noise of the fused rollouts (rollout_kernels.cuh: planar, tree_kernels.cuh: 3-D): Philox4x32-10 keyed by
// (seed, global env id, policy step), Box-Muller on its uniforms.  Counter-based, so a draw does not depend on the launch
// partition or the GPU count.
#pragma once
#include <cstdint>

namespace cassie {

// ---- Philox4x32-10 (Salmon et al., SC'11), counter-based
__host__ __device__ inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
// block b of (seed, env, step): the counter {env, step, b, 0}
__device__ __forceinline__ void philox_block(uint64_t seed, uint32_t env, uint32_t step, uint32_t b, uint32_t c[4]) {
  c[0] = env; c[1] = step; c[2] = b; c[3] = 0u;
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
}
// two standard normals from two words of a block: Box-Muller on (0,1] x [0,1) uniforms
template <typename T>
__device__ __forceinline__ void box_muller(uint32_t w0, uint32_t w1, T& z0, T& z1) {
  const float u1 = ((float)(w0 >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0, 1]
  const float u2 = (float)(w1 >> 8) * (1.0f / 16777216.0f);            // [0, 1)
  const float rad = sqrtf(-2.0f * logf(u1));
  float sn, cs;
  sincospif(2.0f * u2, &sn, &cs);
  z0 = (T)(rad * cs);
  z1 = (T)(rad * sn);
}
// eight standard normals for (seed, env, step): blocks 0 and 1, two Box-Muller pairs each
template <typename T>
__device__ inline void normal8(uint64_t seed, uint32_t env, uint32_t step, T out[8]) {
#pragma unroll
  for (int b = 0; b < 2; b++) {
    uint32_t c[4];
    philox_block(seed, env, step, (uint32_t)b, c);
#pragma unroll
    for (int p = 0; p < 2; p++) box_muller(c[2 * p], c[2 * p + 1], out[4 * b + 2 * p], out[4 * b + 2 * p + 1]);
  }
}
// the standard normal of action slot a alone: slot a is word pair (a >> 1) & 1 of block a >> 2, so slots 0..7 are
// normal8's and slots 8, 9 the first pair of block 2
template <typename T>
__device__ __forceinline__ T normal_slot(uint64_t seed, uint32_t env, uint32_t step, int a) {
  uint32_t c[4];
  philox_block(seed, env, step, (uint32_t)(a >> 2), c);
  const bool hi = (a >> 1) & 1;
  T z0, z1;
  box_muller(hi ? c[2] : c[0], hi ? c[3] : c[1], z0, z1);
  return (a & 1) ? z1 : z0;
}

}  // namespace cassie
