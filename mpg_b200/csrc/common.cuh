// Shared device helpers for the mpg_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/mpg_b200.h"

namespace mpg {

// The hidden width H (64, 128 or 256) is a template parameter of the FFMA tile engine (mlp_tile.cuh); the tensor-core
// path has its own tc::H = 256 (tc_common.cuh).
constexpr int TILE_R = 64;    // rows (trajectories) per CTA tile
constexpr int RP = 68;        // row pitch of [feature][row] activation tiles in shared memory
constexpr int NT = 256;       // threads per CTA
constexpr int KS = 16;        // weight slab depth (k rows) staged per cp.async stage
constexpr int MAX_IN = 20;    // max MLP input width (obs 16 + act 2, padded)
constexpr int MAX_S = 6;      // max env state dim
constexpr int MAX_A = 2;      // max action dim

// ELU (model.py hidden_activation='elu'): x>0 ? x : exp(x)-1.
__device__ __forceinline__ float elu(float x) { return x > 0.f ? x : expm1f(x); }
// derivative expressed through the OUTPUT y (TF EluGrad): y>0 ? 1 : y+1
__device__ __forceinline__ float elu_grad_from_out(float y) { return y > 0.f ? 1.f : y + 1.f; }

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG: noise keyed by (seed, global tiled row, step) so that any
// sharding of the batch over ranks sees the same numbers (SURVEY.md 8(d)/8(e)).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t out[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// standard normal for (row, step): Box-Muller on the first two Philox words
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t row, uint32_t step) {
  uint32_t o[4];
  philox4x32_10((uint32_t)row, (uint32_t)(row >> 32), step, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), o);
  float u1 = ((float)o[0] + 0.5f) * 2.3283064365386963e-10f;  // (0,1]
  float u2 = ((float)o[1] + 0.5f) * 2.3283064365386963e-10f;
  u1 = fminf(fmaxf(u1, 1e-12f), 1.0f);
  return sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
}

}  // namespace mpg
