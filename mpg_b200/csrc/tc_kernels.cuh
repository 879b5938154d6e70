// Tensor-core (tcgen05) model-rollout kernels.
//
// tc_rollout_kernel<ENV,BWD,ACT>: one persistent CTA per SM owns a tile of 128 trajectories and walks the
// horizon.  All 256x256 (and 16x256 / 256x16) contractions of the policy / Q MLPs run on the 5th-gen
// tensor cores with split-bf16 operands (3 products, fp32 accumulation in TMEM); weights are streamed from
// L2 through a shared-memory ring by the TMA engine; the per-row vehicle / pendulum dynamics, rewards,
// output heads and adjoints stay in registers of the thread that owns the row (TMEM lane = row).
// Backward = BPTT from the 24-byte state checkpoints.  The forward pass of the gradient kernel leaves the second
// hidden activation of every step behind as a ready-made operand image (1 KB per row and step, written straight
// from the epilogue registers); BPTT pulls it back with one bulk copy per step instead of re-running layer 1 + layer 2
// (one third of the contraction work and two of the five epilogues of a backward step).  act'(z1) still comes from
// the cheap K = 16 first-layer recompute.  The dX chain (what the recurrence needs) is fully fused.  The weight-gradient contractions (K = rows) cannot be accumulated in place: the
// fp32 accumulator of dW2 alone is 256 KB = all of TMEM.  Their operand tiles (h1, h2, delta1, delta2 as
// split-bf16 images, written to shared memory anyway as UMMA operands) are bulk-stored once and consumed
// by tc_dw_kernel, a split-K tcgen05 GEMM with MN-major operands.
#pragma once
#include "env_models.cuh"
#include "rollout_kernels.cuh"
#include "tc_gemm.cuh"

#ifndef MPG_EPI_INLINE
#define MPG_EPI_INLINE __forceinline__
#endif

namespace mpg {
namespace tc {

struct TcNet {
  const uint8_t* big_fwd;
  const uint8_t* big_dx;
  const uint8_t* l1;    // [W1; b1] as an fp16 pair: forward passes
  const uint8_t* l1b;   // the same as a bf16 pair: first-layer recompute inside BPTT (meets the bf16 [p|1] image of D1)
  const uint8_t* in;
  const float* W3;   // [H][out_dim] natural
  const float* b2;
  const float* b3;
  int in_dim, out_dim;
};

constexpr int BIAS_K = 15;                    // column of the [p|a|1] image that carries the constant 1
// one (tile, step) record of the dW operand store: the h1 and delta2 images (dW2 = h1^T delta2) and the [p|1] image
// (db2 = delta2^T 1).  dW1, db1 and dW3 are accumulated inside the rollout kernel (TM_D1 / TM_D3).
constexpr size_t SLOT_H1 = 0, SLOT_D2 = 131072, SLOT_P = 262144;
constexpr size_t SLOT_BYTES = 270336;

struct TcArgs {
  RolloutArgs r;            // config, lists, pointers (r.pol / r.q unused here)
  TcNet pol, q;
  float* act_ckpt;          // [n_list][M*rows][A] actions at the list steps, at the first entry of each (Q input gradient)
  float* z_ckpt;            // [horizon+1][M*rows][2A] action and head derivative d act / d z of every step (BPTT re-reads them)
  uint8_t* h2store;         // [tile][horizon+1][2*ACT_SPLIT] h2 images of the forward pass (BPTT loads them instead of
                            //    recomputing layer 2)
  uint8_t* store;           // dW operand store: [tile][step][SLOT_BYTES]
  int store_steps;          // steps recorded per tile: horizon+1 (full BPTT) or 1 (first action only)
  int rec_hi_only;          // 1: the dW2 records keep only the hi plane of h1 / delta2 (large batches, see mpg_policy_grad)
  int tile0, tile1;         // tile range of this launch (tile1 == 0: all tiles); CTA c owns tile0 + c, tile0 + c + grid, ...
  int q_regress;            // 1: Q regression gradient (q_forward_and_backward): horizon 0, given actions,
                            //    upstream (Q - target) / B_global, dW operands of the Q net recorded, no policy part
  const float* q_target;    // (rows) regression targets
  float q_inv_rows;         // 1 / B_global
  long long* prof;          // optional: clock64 timestamps of one backward step of CTA 0 (debug / DESIGN.md timeline)
};

// fp32 scratch in shared memory
struct MiscF {
  float W3p[H * 2];
  float b2p[H];
  float W3q[H * 2];
  float b2q[H];
  float part[4 * 2 * ACT_ROWS];   // [column quarter][j][row]
  float d3s[2 * ACT_ROWS];        // [j][row]
  float wsum[8];                  // per-warp delta3 sums [warp][j]
  float b3[4];                    // b3p[0], b3p[1], b3q[0]
};
static_assert(sizeof(MiscF) <= SmemMap::MISC_BYTES, "MISC region too small");

constexpr int SM_D3IMG = SmemMap::TOTAL;          // delta3 image hi|lo (8 KB) appended after the base map
constexpr int SM_TAB = SM_D3IMG + 8192;           // StepTab of the rollout list
constexpr int SM_TOTAL = SM_TAB + (int)((sizeof(StepTab) + 15) / 16 * 16);
static_assert(SM_TOTAL + 1024 <= 227 * 1024, "the rollout kernel's shared memory (+ 1 KB of alignment slack) exceeds 227 KB");

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory"); }
__device__ __forceinline__ float elu_fast(float x) { return x > 0.f ? x : exp_fast(x) - 1.f; }
// hidden activation of the E1 / E2 epilogues.  tanh: the fp32 library tanhf (a few ulp); tanh.approx (MUFU.TANH, relative
// error ~2^-11) would break the 1e-5 closed-loop bar the fp16-pair forward meets.  tanh values lie in [-1, 1]: the fp16 pair
// of h1 does not saturate.
template <int ACT>
__device__ __forceinline__ float act_fast(float x) {
  if constexpr (ACT == MPG_ACT_RELU) return x > 0.f ? x : 0.f;
  else if constexpr (ACT == MPG_ACT_TANH) return tanhf(x);
  else return elu_fast(x);
}
// g act'(z2) through the output h2 (bf16 pair read back from the h2 image): elu' = 1 + min(h2, 0), relu' = [h2 > 0],
// tanh' = 1 - h2^2
template <int ACT>
__device__ __forceinline__ float times_act_grad_out(float g, float h) {
  if constexpr (ACT == MPG_ACT_RELU) return h > 0.f ? g : 0.f;
  else if constexpr (ACT == MPG_ACT_TANH) return g * fmaf(-h, h, 1.f);
  else return fmaf(g, fminf(h, 0.f), g);
}
// act'(z1) from z = z1 log2(e) (the pre-scaled bf16 first-layer image): elu' = 2^min(z, 0), exactly 1 for z >= 0;
// relu' = [z > 0]; tanh' = 1 - tanh^2(z1) = 4 e / (1 + e)^2 with e = 2^(-2|z|) = exp(-2|z1|) (no cancellation)
template <int ACT>
__device__ __forceinline__ float act_grad_log2e(float z) {
  if constexpr (ACT == MPG_ACT_RELU) {
    return z > 0.f ? 1.f : 0.f;
  } else if constexpr (ACT == MPG_ACT_TANH) {
    const float e = ex2_ftz(-2.f * fabsf(z)), d = 1.f + e;
    return __fdividef(4.f * e, d * d);
  } else {
    return ex2_ftz(fminf(z, 0.f));
  }
}

// load 8 consecutive features of row r back from a split-bf16 image (hi + lo)
__device__ __forceinline__ void act_load8(const uint8_t* act_hi, const uint8_t* act_lo, int r, int cc, float* x) {
  const uint32_t off = act_chunk_off(r, cc);
  const uint4 h = *reinterpret_cast<const uint4*>(act_hi + off);
  const uint4 l = *reinterpret_cast<const uint4*>(act_lo + off);
  const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    x[2 * i] = __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
    x[2 * i + 1] = __uint_as_float(hw[i] & 0xFFFF0000u) + __uint_as_float(lw[i] & 0xFFFF0000u);
  }
}

// whole-image bulk store to the dW operand store (one elected epilogue thread); the matching wait must come
// before the shared-memory source is overwritten
__device__ __forceinline__ void store_image(bool elected, uint8_t* gdst, const uint8_t* ssrc, uint32_t bytes) {
  fence_proxy_async();
  epi_bar();
  if (elected) {
    bulk_s2g(gdst, ssrc, bytes);
    bulk_commit();
  }
}
// Block-ordered variant for the big GEMMs' A images (h1, delta2): each K-block of the GEMM reads one 64-feature
// block of the image exactly once, so block kb can leave as soon as the UMMAs of K-block kb are complete
// (kb_done[kb]).  The elected thread -- idle anyway until the accumulator is ready -- issues the four bulk groups
// (hi and lo 16 KB pieces of block kb) behind the GEMM; the next epilogue overwrites the image block by block and
// waits for group kb only (store_wait_block), so the 128 KB store (~4.8 K cycles at the per-SM store rate) drains
// under the GEMM tail and that epilogue instead of in front of it.
__device__ __forceinline__ void store_image_follow(bool elected, Bars* b, const Sync& s, uint8_t* gdst, const uint8_t* ssrc,
                                                   bool hi_only = false) {
  if (elected) {
    const uint32_t par = (s.k_cnt - 1) & 1;                  // the big GEMM issued last
#pragma unroll
    for (int kb = 0; kb < 4; ++kb) {
      mbar_wait(&b->kb_done[kb], par, 20000 + __LINE__);
      bulk_s2g(gdst + kb * ACT_BLOCK, ssrc + kb * ACT_BLOCK, ACT_BLOCK);
      if (!hi_only) bulk_s2g(gdst + ACT_SPLIT + kb * ACT_BLOCK, ssrc + ACT_SPLIT + kb * ACT_BLOCK, ACT_BLOCK);
      bulk_commit();
    }
  }
}
__device__ __forceinline__ void store_wait_block(bool elected, int kb) {
  if (elected) bulk_wait_read_pending(3 - kb);
  epi_bar();
}
__device__ __forceinline__ void store_wait(bool elected) {
  if (elected) bulk_wait_read_all();
  epi_bar();
}

// Block-ordered epilogues: every warp handles 16 columns of each 64-feature block kb, so that block kb of
// the activation image is complete (and published to the MMA warp) after 1/4 of the epilogue.

// z1 (streamed through the two TMEM chunk buffers, bias folded in) -> h1 image
template <int ACT>
__device__ MPG_EPI_INLINE void epi_hidden1_blocks(Bars* b, uint32_t tm_zc_lane, uint8_t* act, int row, int hc) {
  // (reading the two chunk buffers out in pairs, to release chunk 1 early and get chunk 3 out of the layer-2 GEMM's way, was
  // slower: a first-layer chunk takes ~500 cycles in the tensor pipe, so block 0 started that much later)
  for (int kb = 0; kb < 4; ++kb) {
    const int c0 = kb * 64 + hc * 16;
    float v[16];
    epi_wait_chunk(b, kb);
    tmem_ld16(tm_zc_lane + (kb & 1) * 64 + hc * 16, v);
    epi_release_chunk(b, kb);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = act_fast<ACT>(v[i]);
    act_store8<true>(act, act + ACT_SPLIT, row, c0 >> 3, v);
    act_store8<true>(act, act + ACT_SPLIT, row, (c0 >> 3) + 1, v + 8);
    epi_block_done(b, kb);
  }
}
// z2 (TMEM) + b2 -> h2 -> partial output-layer dot products (forward pass: no image needed)
template <int ACT>
__device__ MPG_EPI_INLINE void epi_hidden2(uint32_t tm_lane, const float* b2, const float* W3, int hc, float& p0, float& p1) {
  p0 = 0.f; p1 = 0.f;
  for (int c0 = hc * COLS_PER_WARP; c0 < (hc + 1) * COLS_PER_WARP; c0 += 32) {
    float v[32];
    tmem_ld32(tm_lane + c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float h = act_fast<ACT>(v[i] + b2[c0 + i]);
      const float2 w = *reinterpret_cast<const float2*>(W3 + 2 * (c0 + i));
      p0 = fmaf(h, w.x, p0);
      p1 = fmaf(h, w.y, p1);
    }
  }
}
// same, and leave h2 behind in global memory as an operand image in the row-interleaved layout
//   [split hi|lo][16-byte chunk cc = 8 features][row][16 B]
// (the canonical no-swizzle UMMA layout: K-major with LBO = 2048, SBO = 128, and MN-major with LBO = 128, SBO = 2048).
// A warp (32 consecutive rows, one chunk) writes 512 contiguous bytes per store instruction.
__device__ __forceinline__ uint32_t lin_chunk_off(int r, int cc) { return (uint32_t)(cc * (ACT_ROWS * 16) + r * 16); }
template <int ACT>
__device__ MPG_EPI_INLINE void epi_hidden2_gstore(uint32_t tm_lane, const float* b2, const float* W3, uint8_t* gimg, int row,
                                                  int hc, float& p0, float& p1) {
  p0 = 0.f; p1 = 0.f;
  for (int c0 = hc * COLS_PER_WARP; c0 < (hc + 1) * COLS_PER_WARP; c0 += 16) {
    float v[16];
    tmem_ld16(tm_lane + c0, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      v[i] = act_fast<ACT>(v[i] + b2[c0 + i]);
      const float2 w = *reinterpret_cast<const float2*>(W3 + 2 * (c0 + i));
      p0 = fmaf(v[i], w.x, p0);
      p1 = fmaf(v[i], w.y, p1);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint4 hi, lo;
      split2(v[8 * h + 0], v[8 * h + 1], hi.x, lo.x);
      split2(v[8 * h + 2], v[8 * h + 3], hi.y, lo.y);
      split2(v[8 * h + 4], v[8 * h + 5], hi.z, lo.z);
      split2(v[8 * h + 6], v[8 * h + 7], hi.w, lo.w);
      const uint32_t off = lin_chunk_off(row, (c0 >> 3) + h);
      *reinterpret_cast<uint4*>(gimg + off) = hi;
      *reinterpret_cast<uint4*>(gimg + ACT_SPLIT + off) = lo;
    }
  }
}
// same, and keep h2 as an image (Q part of the backward pass: delta2 and the dW3 operand are derived from it)
template <int ACT>
__device__ MPG_EPI_INLINE void epi_hidden2_img(uint32_t tm_lane, const float* b2, const float* W3, uint8_t* act, int row,
                                               int hc, float& p0, float& p1, bool draining = false, bool elected = false) {
  p0 = 0.f; p1 = 0.f;
  for (int kb = 0; kb < 4; ++kb) {
    const int c0 = kb * 64 + hc * 16;
    float v[16];
    tmem_ld16(tm_lane + c0, v);
    if (draining) store_wait_block(elected, kb);             // block kb of the old image has been read out
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      v[i] = act_fast<ACT>(v[i] + b2[c0 + i]);
      const float2 w = *reinterpret_cast<const float2*>(W3 + 2 * (c0 + i));
      p0 = fmaf(v[i], w.x, p0);
      p1 = fmaf(v[i], w.y, p1);
    }
    act_store8(act, act + ACT_SPLIT, row, c0 >> 3, v);
    act_store8(act, act + ACT_SPLIT, row, (c0 >> 3) + 1, v + 8);
  }
}
// delta2 = (delta3 W3^T) * act'(h2), h2 read back from its image and overwritten in place by delta2
template <int ACT>
__device__ MPG_EPI_INLINE void epi_delta2_blocks(Bars* b, const float* W3, float d30, float d31, uint8_t* act, int row, int hc,
                                                 Sync* wait_half1 = nullptr) {
  for (int kb = 0; kb < 4; ++kb) {
    const int c0 = kb * 64 + hc * 16;
    if (kb == 2 && wait_half1) epi_wait_half(b, *wait_half1);   // the D3 UMMAs have read blocks 2, 3 of the h2 image
    float v[16];
    act_load8(act, act + ACT_SPLIT, row, c0 >> 3, v);
    act_load8(act, act + ACT_SPLIT, row, (c0 >> 3) + 1, v + 8);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float2 w = *reinterpret_cast<const float2*>(W3 + 2 * (c0 + i));
      const float g = fmaf(d30, w.x, d31 * w.y);
      v[i] = times_act_grad_out<ACT>(g, v[i]);        // g act'(z2), expressed through the output h2
    }
    act_store8(act, act + ACT_SPLIT, row, c0 >> 3, v);
    act_store8(act, act + ACT_SPLIT, row, (c0 >> 3) + 1, v + 8);
    epi_block_done(b, kb);
  }
}
// BPTT variant: h2 arrives from the h2 store in the row-interleaved layout (lin_chunk_off); delta2 is written as the
// SW128 K-major image the dX UMMAs and the dW2 record expect.  Both layouts keep 64-feature block kb inside the same
// 16 KB per split, so the conversion is in place block by block: every thread reads its part of block kb, barrier,
// every thread writes.  wait_d3: the D3 UMMAs (dW3 += h2^T delta3) read the same image; blocks 0, 1 may be overwritten when
// their first half has completed (d_full), blocks 2, 3 after the second (d_half).  Only the WRITES wait for that: the
// reads and the arithmetic of blocks 0 and 2 run underneath those UMMAs (16 per half, ~190 cycles each from the
// no-swizzle image).
template <int ACT>
__device__ MPG_EPI_INLINE void epi_delta2_from_h2(Bars* b, const float* W3, float d30, float d31, uint8_t* act, int row, int hc,
                                                  uint32_t img_parity, Sync* wait_d3 = nullptr) {
  for (int kb = 0; kb < 4; ++kb) {
    const int c0 = kb * 64 + hc * 16;
    if (kb == 2) mbar_wait(&b->img_full[1], img_parity, 20000 + __LINE__);      // second half of the h2 image has landed
    float v[16];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t off = lin_chunk_off(row, (c0 >> 3) + h);
      const uint4 hv = *reinterpret_cast<const uint4*>(act + off);
      const uint4 lv = *reinterpret_cast<const uint4*>(act + ACT_SPLIT + off);
      const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        v[8 * h + 2 * i] = __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
        v[8 * h + 2 * i + 1] = __uint_as_float(hw[i] & 0xFFFF0000u) + __uint_as_float(lw[i] & 0xFFFF0000u);
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float2 w = *reinterpret_cast<const float2*>(W3 + 2 * (c0 + i));
      const float g = fmaf(d30, w.x, d31 * w.y);
      v[i] = times_act_grad_out<ACT>(g, v[i]);        // g act'(z2), expressed through the output h2
    }
    if (wait_d3 && kb == 0) epi_wait_d(b, *wait_d3);         // the D3 UMMAs have read blocks 0, 1 of the h2 image
    if (wait_d3 && kb == 2) epi_wait_half(b, *wait_d3);      // ... and blocks 2, 3
    epi_bar();                                               // block kb has been read by everybody
    act_store8(act, act + ACT_SPLIT, row, c0 >> 3, v);
    act_store8(act, act + ACT_SPLIT, row, (c0 >> 3) + 1, v + 8);
    epi_block_done(b, kb);
  }
}
// delta1 = g_h1 (TMEM work) * act'(z1) (z1 log2(e) recomputed with the pre-scaled bf16 first-layer image, streamed through the
// chunk buffers) -> delta1 image
template <int ACT>
__device__ MPG_EPI_INLINE void epi_delta1_blocks(Bars* b, uint32_t tm_work_lane, uint32_t tm_zc_lane, uint8_t* act, int row,
                                                 int hc, bool draining = false, bool elected = false, bool release_img = false) {
  for (int kb = 0; kb < 4; ++kb) {
    const int c0 = kb * 64 + hc * 16;
    float g[16], z[16];
    tmem_ld16(tm_work_lane + c0, g);
    epi_wait_chunk(b, kb);
    tmem_ld16(tm_zc_lane + (kb & 1) * 64 + hc * 16, z);
    epi_release_chunk(b, kb);
    if (draining) store_wait_block(elected, kb);             // block kb of the old image has been read out
#pragma unroll
    for (int i = 0; i < 16; ++i) g[i] *= act_grad_log2e<ACT>(z[i]);     // z = z1 log2(e) (l1b image)
    act_store8(act, act + ACT_SPLIT, row, c0 >> 3, g);
    act_store8(act, act + ACT_SPLIT, row, (c0 >> 3) + 1, g + 8);
    epi_block_done(b, kb);
    // the record store has read blocks 0..kb of the old image (store_wait_block above): with the mma thread's commit
    // behind the UMMAs that read the new one, half kb / 2 is free for the h2 image of the next step
    if (release_img && elected && (kb & 1)) mbar_arrive(&b->img_empty[kb >> 1]);
  }
}
// delta3 image, one plane: the first 16-byte chunk of row `row` is [d0_hi, d1_hi, d0_lo, d1_lo, 0, 0, 0, 0] (hi and lo
// side by side in N, see tc_gemm.cuh); the second chunk stays zero
__device__ __forceinline__ void write_d3(uint8_t* img, int row, float d0, float d1) {
  uint32_t h, l;
  split2(d0, d1, h, l);
  *reinterpret_cast<uint4*>(img + il_chunk_off(row, 0)) = make_uint4(h, l, 0u, 0u);
}

// g_p = delta1 . W1_hi^T + delta1 . W1_lo^T: columns [0,16) + [16,32) of the accumulator
__device__ __forceinline__ void read_gp(uint32_t taddr, float (&g)[16]) {
  float g2[16];
  tmem_ld16(taddr, g);
  tmem_ld16(taddr + 16, g2);
#pragma unroll
  for (int i = 0; i < 16; ++i) g[i] += g2[i];
}

// named barriers between the epilogue warps (512 threads) and the row warps (128 threads)
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
constexpr int BAR_PART = 2;   // epilogue -> row: partial output-layer dots (MiscF::part) written
constexpr int BAR_D3 = 3;     // row -> epilogue: delta3 (MiscF::d3s) written
constexpr int BAR_ROW = 4;    // row warps among themselves
constexpr int ROW_THREADS = ACT_ROWS;
constexpr int XCHG_THREADS = EPI_THREADS + ROW_THREADS;

// One schedule, four roles.  ROLE_EPI: 16 warps, thread = (row, 64-column quarter), all 128 x 256 element-wise work.
// ROLE_ROW: 4 warps, thread = trajectory: environment step and adjoint, output head, [p|a|1] / delta3 images,
// checkpoints, returns -- the scalar recurrence lives in registers of threads that hold nothing else.
// ROLE_PRODUCER / ROLE_MMA: one thread each.
template <int ENV, bool BWD, int ACT, int ROLE>
__device__ __forceinline__ void run_rollout(const TcArgs& A, uint8_t* smem, Bars* b) {
  using E = Env<ENV>;
  constexpr int S = E::S, NA = E::A;
  const RolloutArgs& a = A.r;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row = (warp & 3) * 32 + lane, hc = (warp >> 2) & 3;   // hc: column quarter of an epilogue warp
  const bool rowthread = (ROLE == ROLE_ROW);
  const bool elected = (ROLE == ROLE_EPI) && tid == 0;
  const int MB = a.rows * a.M;
  const int ntiles = (MB + ACT_ROWS - 1) / ACT_ROWS;
  MiscF* mf = reinterpret_cast<MiscF*>(smem + SmemMap::MISC);
  uint8_t* act_img = smem + SmemMap::ACT;
  uint8_t* p_img = smem + SmemMap::PIMG;
  uint8_t* d3_img = smem + SM_D3IMG;
  const uint32_t tmem = b->tmem_base;
  const uint32_t tm_z1c = tmem + TM_Z1C, tm_work = tmem + TM_WORK, tm_gp = tmem + TM_GP, tm_d1 = tmem + TM_D1, tm_d3 = tmem + TM_D3;
  const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
  const float cscale = -1.f / ((float)a.M * (float)a.global_rows);
  const bool store_dw = BWD && A.store != nullptr;
  Sync sy;
  bool d1_started = false, d3_started = false;   // mma role: the persistent accumulators hold a value
  bool d1_pending = false, any_dw = false;       // D1 UMMAs in flight / accumulators were used
  bool store_pending = false;                    // epilogue role: a record store still reads the activation image
  // The D1 UMMAs of a step read the delta1 and [p|1] images.  The activation image is protected by img_empty (mma commit);
  // the [p|1] image is rewritten by the row warps, which wait for acc_done right before they do.  The epilogue warps only
  // count the phases and wait for the last one before they read the accumulators out.
  uint32_t acc_issued = 0;
  auto acc_wait = [&]() {
    if (ROLE == ROLE_ROW && d1_pending) {
      mbar_wait(&b->acc_done, sy.acc_cnt & 1, 20000 + __LINE__);
      ++sy.acc_cnt;
    }
    d1_pending = false;
  };
  float db3acc[2] = {0.f, 0.f};                  // row warps: sum of this row's delta3 over steps and tiles
  int prof_t = -1;   // step being traced
  auto stamp = [&](int id) {      // clock64 timeline of one step of CTA 0 (tools/tc_timeline.py): debug library only
#ifdef MPG_DEBUG_PROBES
    if (A.prof && blockIdx.x == 0 && prof_t >= 0
        && ((ROLE == ROLE_EPI && tid == 0) || ROLE == ROLE_MMA || (ROLE == ROLE_ROW && tid == EPI_THREADS)))
      A.prof[(ROLE == ROLE_MMA ? 32 : (ROLE == ROLE_ROW ? 64 : 0)) + id] = clock64();
#else
    (void)id; (void)prof_t;
#endif
  };

  const StepTab& tab = *reinterpret_cast<const StepTab*>(smem + SM_TAB);   // what the list means at each step

  const int tile_end = A.tile1 > 0 && A.tile1 < ntiles ? A.tile1 : ntiles;
  for (int tile = A.tile0 + blockIdx.x; tile < tile_end; tile += gridDim.x) {
    const int grow = tile * ACT_ROWS + row;
    const bool valid = rowthread && grow < MB;
    const int m_idx = valid ? grow / a.rows : 0, i_idx = valid ? grow % a.rows : 0;
    const unsigned long long noise_row = (unsigned long long)m_idx * (unsigned long long)a.global_rows
                                         + (unsigned long long)(a.row_offset + i_idx);
    uint8_t* h2tile = (BWD && A.h2store) ? A.h2store + (size_t)tile * (size_t)(a.horizon + 1) * (2 * ACT_SPLIT) : nullptr;
    float s[S];
#pragma unroll
    for (int j = 0; j < S; ++j) s[j] = 0.f;
    if (valid) {
      float o[MPG_MAX_OBS];
#pragma unroll
      for (int i = 0; i < MPG_MAX_OBS; ++i) o[i] = i < a.obs_dim ? a.obs[(size_t)i_idx * a.obs_dim + i] : 0.f;
      E::reset(o, s);
    }
    float rsum = 0.f, gpow = 1.f;

    // [sigma*obs_t | act | 0.. | 1] -> p image (row warps).  Step 0 observes the row of obs as given, re-read from global
    // memory (replay data need not lie on the model's observation map); a later step observes get_obs(s_t).
    // f16: forward computations read the image as an fp16 pair; BPTT (first-layer recompute, D1, the db2 record) as bf16
    auto write_pimg = [&](int t, const float* act_or_null, bool f16, uint8_t* gimg = nullptr) {
      // every index below is a compile-time constant (fixed trip counts + predicates): o[] stays in registers, and the
      // image row is produced one 8-element chunk at a time
      float o[MPG_MAX_OBS];
#pragma unroll
      for (int i = 0; i < MPG_MAX_OBS; ++i) o[i] = 0.f;
      E::get_obs(s, o, a.nfd);
#pragma unroll
      for (int kh = 0; kh < 2; ++kh) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int i = kh * 8 + e;
          float v = i < a.obs_dim ? (t == 0 ? a.obs[(size_t)i_idx * a.obs_dim + i] : o[i]) * a.obs_scale[i] : 0.f;
          if (act_or_null) {
#pragma unroll
            for (int j = 0; j < NA; ++j)
              if (i == a.obs_dim + j) v = act_or_null[j];
          }
          x[e] = i == BIAS_K ? 1.f : v;
        }
        uint4 h, l;
        if (f16) {
          split2h(x[0], x[1], h.x, l.x); split2h(x[2], x[3], h.y, l.y); split2h(x[4], x[5], h.z, l.z); split2h(x[6], x[7], h.w, l.w);
        } else {
          split2(x[0], x[1], h.x, l.x); split2(x[2], x[3], h.y, l.y); split2(x[4], x[5], h.z, l.z); split2(x[6], x[7], h.w, l.w);
        }
        const uint32_t off = p_chunk_off(row, kh);
        *reinterpret_cast<uint4*>(p_img + off) = h;
        *reinterpret_cast<uint4*>(p_img + off + P_LO) = l;
        if (gimg) {
          *reinterpret_cast<uint4*>(gimg + off) = h;
          *reinterpret_cast<uint4*>(gimg + off + P_LO) = l;
        }
      }
    };
    // policy forward on the current p image: the row thread gets the pre-activations of the head.
    // The layer-2 UMMAs are issued K-block by K-block while the epilogue is still producing h1.  In the gradient
    // kernel h2 goes to the h2 store of this (tile, step) and, for the steps whose weight gradient is wanted (slot),
    // the h1 image leaves for the dW operand store behind the K-blocks of the GEMM.
    auto policy_forward = [&](float* zpre, uint8_t* h2slot, uint8_t* slot) {
      if (ROLE == ROLE_MMA) stamp(16);
#ifdef MPG_DEBUG_PROBES
      fwd_pair_issue<ROLE>(b, smem, sy, A.pol.l1, A.pol.big_fwd, tm_z1c, tm_work,
                           (ROLE == ROLE_MMA && A.prof && blockIdx.x == 0 && prof_t >= 0) ? A.prof + 96 : nullptr);
#else
      fwd_pair_issue<ROLE>(b, smem, sy, A.pol.l1, A.pol.big_fwd, tm_z1c, tm_work);
#endif
      if (ROLE == ROLE_MMA) stamp(17);
      if (ROLE == ROLE_EPI) {
        stamp(17);
        if (store_pending) { store_wait(elected); store_pending = false; }   // the previous step's h1 record has left long ago
        epi_hidden1_blocks<ACT>(b, tm_z1c + lane_off, act_img, row, hc);          // follows the z1 chunk stream
        stamp(18);
        if (slot) { store_image_follow(elected, b, sy, slot + SLOT_H1, act_img, A.rec_hi_only != 0); store_pending = true; }
        epi_wait_d(b, sy);                                   // z2 (all layer-2 UMMAs done)
        stamp(19);
        float p0, p1;
        if (BWD) epi_hidden2_gstore<ACT>(tm_work + lane_off, mf->b2p, mf->W3p, h2slot, row, hc, p0, p1);
        else epi_hidden2<ACT>(tm_work + lane_off, mf->b2p, mf->W3p, hc, p0, p1);
        stamp(20);
        mf->part[(hc * 2 + 0) * ACT_ROWS + row] = p0;
        mf->part[(hc * 2 + 1) * ACT_ROWS + row] = p1;
        bar_arrive(BAR_PART, XCHG_THREADS);
      }
      if (rowthread) {
        bar_sync(BAR_PART, XCHG_THREADS);
#pragma unroll
        for (int j = 0; j < NA; ++j)
          zpre[j] = mf->b3[j] + ((mf->part[(0 * 2 + j) * ACT_ROWS + row] + mf->part[(1 * 2 + j) * ACT_ROWS + row])
                                 + (mf->part[(2 * 2 + j) * ACT_ROWS + row] + mf->part[(3 * 2 + j) * ACT_ROWS + row]));
      }
    };
    // Q forward on the current [p|a|1] image: returns Q for the row thread
    auto q_forward = [&](bool with_img, uint8_t* qslot) -> float {
      float qv = 0.f;
      fwd_pair_issue<ROLE>(b, smem, sy, A.q.l1, A.q.big_fwd, tm_z1c, tm_work);
      if (ROLE == ROLE_EPI) {
        if (store_pending) { store_wait(elected); store_pending = false; }
        epi_hidden1_blocks<ACT>(b, tm_z1c + lane_off, act_img, row, hc);
        if (qslot) store_image(elected, qslot + SLOT_H1, act_img, A.rec_hi_only ? ACT_SPLIT : 2 * ACT_SPLIT);
        epi_wait_d(b, sy);
        float p0, p1;
        if (with_img) {
          if (qslot) store_wait(elected);
          epi_hidden2_img<ACT>(tm_work + lane_off, mf->b2q, mf->W3q, act_img, row, hc, p0, p1);
        } else {
          epi_hidden2<ACT>(tm_work + lane_off, mf->b2q, mf->W3q, hc, p0, p1);
        }
        mf->part[(hc * 2 + 0) * ACT_ROWS + row] = p0;
        bar_arrive(BAR_PART, XCHG_THREADS);
      }
      if (rowthread) {
        bar_sync(BAR_PART, XCHG_THREADS);
        qv = mf->b3[2] + ((mf->part[0 * ACT_ROWS + row] + mf->part[2 * ACT_ROWS + row])
                          + (mf->part[4 * ACT_ROWS + row] + mf->part[6 * ACT_ROWS + row]));
      }
      return qv;
    };

    // =========================================== forward ===========================================
    acc_wait();   // previous tile's last D1 UMMAs still read the [p|1] image
    for (int t = 0; t <= a.horizon; ++t) {
      float act[NA];
#pragma unroll
      for (int j = 0; j < NA; ++j) act[j] = 0.f;
      const bool given = (t == 0 && a.use_start_actions);
      // steps whose weight gradient is wanted leave their dW2 operands (h1 now, delta2 during BPTT) in the operand store
      const bool rec_f = store_dw && !A.q_regress && (a.full_bptt || t == 0);
      uint8_t* slot = rec_f ? A.store + ((size_t)tile * A.store_steps + (a.full_bptt ? t : 0)) * SLOT_BYTES : nullptr;
      if (tile == A.tile0 + (int)blockIdx.x && t == 2) {
        prof_t = t;
        if (ROLE != ROLE_MMA) stamp(16);
      } else if (prof_t >= 0) {
        if (ROLE != ROLE_MMA) stamp(22);
        prof_t = -1;
      }
      if (rowthread) {
        if (BWD && valid) {
          float* c = a.ckpt + ((size_t)t * MB + grow) * S;
#pragma unroll
          for (int j = 0; j < S; ++j) c[j] = s[j];
        }
        if (!given) write_pimg(t, nullptr, true);
      }
      if (!given) {
        float zpre[NA];
        policy_forward(zpre, BWD ? h2tile + (size_t)t * (2 * ACT_SPLIT) : nullptr, slot);
        stamp(21);
        if (rowthread) {
          float hg[NA];
#pragma unroll
          for (int j = 0; j < NA; ++j) head_fwd_grad(zpre[j], a.policy_out_tanh, a.action_range, act[j], hg[j]);
          if (BWD && valid)
#pragma unroll
            for (int j = 0; j < NA; ++j) {
              A.z_ckpt[((size_t)t * MB + grow) * (2 * NA) + j] = act[j];
              A.z_ckpt[((size_t)t * MB + grow) * (2 * NA) + NA + j] = hg[j];
            }
        }
      } else if (valid) {
#pragma unroll
        for (int j = 0; j < NA; ++j) act[j] = a.start_actions[(size_t)i_idx * NA + j];
      }
      if (valid && a.traj_act)
#pragma unroll
        for (int j = 0; j < NA; ++j) a.traj_act[((size_t)t * MB + grow) * NA + j] = act[j];
      const int kidx = tab.first(t);   // the first entry at step t keys the action checkpoint of the step
      if (kidx >= 0) {
        float qv = 0.f;
        if (BWD && valid)
#pragma unroll
          for (int j = 0; j < NA; ++j) A.act_ckpt[((size_t)kidx * MB + grow) * NA + j] = act[j];
        if (a.has_q) {
          if (rowthread) write_pimg(t, act, true);
          qv = q_forward(false, nullptr);
        }
        // every entry of step t gets its row, repeated entries included
        if (valid && a.returns_out)
          for (int k = kidx; k >= 0; k = tab.next[k]) a.returns_out[(size_t)k * MB + grow] = rsum + gpow * qv;
      }
      if (t < a.horizon && valid) {
        float eps = 0.f;
        if (E::HAS_NOISE) {
          if (a.noise_mode == 1) eps = a.noise[(size_t)t * MB + grow];
          else if (a.noise_mode == 2) eps = philox_normal(a.seed, noise_row, (uint32_t)t);
        }
        const float rew = E::step(s, act, eps, a.noise_mode != 0);
        const float prew = (rew + a.rew_shift) * a.rew_scale;
        rsum += gpow * prew;
        gpow *= a.gamma;
        if (a.traj_rew) a.traj_rew[(size_t)t * MB + grow] = prew;
        if (a.traj_obs) {
          float o[MPG_MAX_OBS];
          E::get_obs(s, o, a.nfd);
#pragma unroll
          for (int i = 0; i < MPG_MAX_OBS; ++i)
            if (i < a.obs_dim) a.traj_obs[((size_t)t * MB + grow) * a.obs_dim + i] = o[i];
        }
      }
    }
    // =========================================== backward ==========================================
    if (BWD) {
      float lam[S], snext[S], spre[S], zpre_n[2 * NA];   // zpre_n: action and head derivative of the next step to process
#pragma unroll
      for (int j = 0; j < S; ++j) { lam[j] = 0.f; snext[j] = s[j]; spre[j] = s[j]; }   // s == s_horizon here
#pragma unroll
      for (int j = 0; j < 2 * NA; ++j)
        zpre_n[j] = (valid && !A.q_regress) ? A.z_ckpt[((size_t)a.horizon * MB + grow) * (2 * NA) + j] : 0.f;
      for (int t = a.horizon; t >= 0; --t) {
        float gp = 1.f;
        for (int i = 0; i < t; ++i) gp *= a.gamma;
        const bool want_dw = a.full_bptt || t == 0;
        const bool rec = store_dw && want_dw;
        prof_t = (tile == A.tile0 + (int)blockIdx.x && t == a.horizon - 2) ? t : -1;
        stamp(0);
        uint8_t* slot = rec ? A.store + ((size_t)tile * A.store_steps + (a.full_bptt ? t : 0)) * SLOT_BYTES : nullptr;
        float g_a[NA], g_s[S], act[NA], hgrad[NA];
#pragma unroll
        for (int j = 0; j < NA; ++j) { g_a[j] = 0.f; act[j] = zpre_n[j]; hgrad[j] = zpre_n[NA + j]; }
#pragma unroll
        for (int j = 0; j < S; ++j) g_s[j] = 0.f;
        if (valid) {
          // s_t and the head values were prefetched during the previous iteration; issue the loads of step
          // t-1 now so that their global-memory latency hides behind this step
#pragma unroll
          for (int j = 0; j < S; ++j) s[j] = spre[j];
          if (t > 0) {
            const float* c = a.ckpt + ((size_t)(t - 1) * MB + grow) * S;
#pragma unroll
            for (int j = 0; j < S; ++j) spre[j] = c[j];
            if (!A.q_regress)
#pragma unroll
              for (int j = 0; j < 2 * NA; ++j) zpre_n[j] = A.z_ckpt[((size_t)(t - 1) * MB + grow) * (2 * NA) + j];
          }
        }
        if (ROLE == ROLE_ROW) stamp(4);
        const int kidx = tab.first(t);
        if (want_dw) any_dw = true;
        // ---- Q input gradient at the list steps: upstream c w_t gamma^t on Q1(p_t, a_t), w_t = the summed weight of
        // every entry at step t ----
        // does step tt start with a Q part (which uses the activation image before the policy part does)?  Yes when some
        // entry at tt has a non-zero weight: the h2 prefetch schedule below and the gate of the Q part both ask this
        auto q_part_at = [&](int tt) { return tab.q_part(tt) && a.has_q; };
        // early: the h2 image of this step was requested during the previous one; early_next: request the next one
        const bool early = t < a.horizon && !q_part_at(t);
        const bool early_next = t > 0 && !q_part_at(t - 1) && !A.q_regress;
        auto load_h2 = [&](int tt) {      // producer: both halves of the h2 image of step tt, each as soon as it is free
          const uint8_t* src = h2tile + (size_t)tt * (2 * ACT_SPLIT);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            mbar_wait(&b->img_empty[h], sy.i_cnt & 1, 20000 + __LINE__);
            mbar_expect_tx(&b->img_full[h], ACT_SPLIT);
#pragma unroll
            for (int sp = 0; sp < 2; ++sp)
#pragma unroll
              for (int k = 0; k < 2; ++k) {
                const size_t off = (size_t)sp * ACT_SPLIT + (size_t)(2 * h + k) * ACT_BLOCK;
                bulk_g2s(act_img + off, src + off, ACT_BLOCK, &b->img_full[h]);
              }
          }
        };
        if (kidx >= 0 && a.has_q && (q_part_at(t) || A.q_regress)) {
          const bool reg = A.q_regress != 0;      // regression: weight gradients of the Q net, no input gradient
          uint8_t* qslot = (reg && store_dw) ? A.store + (size_t)tile * SLOT_BYTES : nullptr;
          if (rowthread) {
            float ak[NA];
#pragma unroll
            for (int j = 0; j < NA; ++j) ak[j] = valid ? A.act_ckpt[((size_t)kidx * MB + grow) * NA + j] : 0.f;
            acc_wait();
            write_pimg(t, ak, true);
          }
          const float qv = q_forward(true, qslot);         // h2q image in ACT
          if (rowthread) {
            // the forward part is done with the fp16 image (every z1 chunk has been consumed): the same row as a bf16 pair
            // for the first-layer recompute / D1 of this part and the db2 record
            float ak[NA];
#pragma unroll
            for (int j = 0; j < NA; ++j) ak[j] = valid ? A.act_ckpt[((size_t)kidx * MB + grow) * NA + j] : 0.f;
            write_pimg(t, ak, false, qslot ? qslot + SLOT_P : nullptr);
            fence_proxy_async();
            mbar_arrive(&b->p_full);
          }
          if (rowthread) {
            // upstream on Q: policy loss c w_t gamma^t, or the regression residual (Q - target) / B_global
            const float up = !valid ? 0.f : (reg ? (qv - A.q_target[i_idx]) * A.q_inv_rows : cscale * tab.wq(t) * gp);
            mf->d3s[row] = up;
            if (reg) {
              write_d3(d3_img, row, up, 0.f);
              db3acc[0] += up;
            }
            bar_arrive(BAR_D3, XCHG_THREADS);
          }
          if (reg) d3_issue<ROLE>(b, smem, sy, SM_D3IMG, d3_started, tm_d3);   // dW3q += h2q^T delta3
          if (ROLE == ROLE_EPI) {
            if (reg) epi_wait_d(b, sy);                    // blocks 0, 1 of the h2q image read by the D3 UMMAs
            bar_sync(BAR_D3, XCHG_THREADS);
          }
          gemm_issue<ROLE>(0, b, smem, sy, A.q.big_dx, tm_work);  // g_h1q, K-blocks issued as delta2 blocks appear
          if (ROLE == ROLE_EPI) {
            epi_delta2_blocks<ACT>(b, mf->W3q, mf->d3s[row], 0.f, act_img, row, hc, reg ? &sy : nullptr);
            if (qslot) store_image(elected, qslot + SLOT_D2, act_img, A.rec_hi_only ? ACT_SPLIT : 2 * ACT_SPLIT);
            epi_wait_d(b, sy);
          }
          bwd_tail_issue<ROLE>(b, smem, sy, A.q.l1b, A.q.in, !reg, reg, d1_started, tm_z1c, tm_gp, tm_d1, true);
          if (ROLE == ROLE_EPI) {
            if (qslot) store_wait(elected);                // delta2 image read out before it is overwritten
            epi_delta1_blocks<ACT>(b, tm_work + lane_off, tm_z1c + lane_off, act_img, row, hc);
            if (!reg) epi_wait_d(b, sy);
          }
          if (reg) { d1_pending = true; ++acc_issued; }
          if (rowthread && !reg) {
            mbar_wait(&b->gp_full, sy.gp_cnt & 1, 20000 + __LINE__);
            ++sy.gp_cnt;
            tc_fence_after();
            float gin[16];
            read_gp(tm_gp + lane_off, gin);
            if (valid) {
              float go[MPG_MAX_OBS];
#pragma unroll
              for (int i = 0; i < MPG_MAX_OBS; ++i) go[i] = i < a.obs_dim ? gin[i] * a.obs_scale[i] : 0.f;
              E::obs_grad_to_state(s, go, a.nfd, g_s);
#pragma unroll
              for (int j = 0; j < NA; ++j)
#pragma unroll
                for (int i = 0; i < 16; ++i)
                  if (i == a.obs_dim + j) g_a[j] += gin[i];
            }
          }
        }
        if (A.q_regress) continue;   // Q regression: no policy part
        // ---- per-row environment adjoint and delta3: they need only lambda and the checkpoints, so the row warps
        // run them first; the dX chain of the epilogue warps hangs on delta3 ----
        if (rowthread) {
          tc_fence_before();         // the g_p read of the previous step precedes the next g_p UMMAs (ordered through p_full)
          stamp(5);
          if (t < a.horizon && valid) {
            env_step_bwd<ENV, true>(s, act, lam, cscale * tab.wlater(t) * gp * a.rew_scale, g_s, g_a, snext);
          }
          stamp(14);
          float d3[2] = {0.f, 0.f};
#pragma unroll
          for (int j = 0; j < NA; ++j) {
            d3[j] = valid ? g_a[j] * hgrad[j] : 0.f;
            mf->d3s[j * ACT_ROWS + row] = d3[j];
          }
          if (NA == 1) mf->d3s[ACT_ROWS + row] = 0.f;
          if (want_dw) {
            write_d3(d3_img, row, d3[0], d3[1]);
            db3acc[0] += d3[0]; db3acc[1] += d3[1];
          }
          bar_arrive(BAR_D3, XCHG_THREADS);
          stamp(2);
        }
        // ---- h2 image of step t: store of the forward pass -> activation image, in two 128-feature halves.  A half is
        // free once the UMMAs that read it have completed and no record store reads it.  In the steady state both were
        // released during the previous step (bwd_tail_issue / epi_delta1_blocks) and the loads are already in flight;
        // the first step of a tile and steps with a Q part release them here ----
        if (!early) {
          if (ROLE == ROLE_MMA) { umma_commit(&b->img_empty[0]); umma_commit(&b->img_empty[1]); }
          if (elected) {
            bulk_wait_read_all();
            mbar_arrive(&b->img_empty[0]);
            mbar_arrive(&b->img_empty[1]);
          }
          if (ROLE == ROLE_PRODUCER) load_h2(t);
        }
        store_pending = false;
        stamp(1);
        if (ROLE == ROLE_EPI) {
          mbar_wait(&b->img_full[0], sy.i_cnt & 1, 20000 + __LINE__);         // first half of the h2 image landed
          stamp(3);
        }
        ++sy.i_cnt;
        if (ROLE == ROLE_MMA) stamp(5);
        if (want_dw) d3_issue<ROLE>(b, smem, sy, SM_D3IMG, d3_started, tm_d3, true, A.rec_hi_only != 0);   // dW3 += h2^T delta3
        if (ROLE == ROLE_MMA) stamp(6);
        // ---- [p|1] image of step t (first-layer recompute for act'(z1), D1 operand, db2 record); the D1 UMMAs of the
        // previous step still read the old one ----
        if (rowthread) {
          acc_wait();
          stamp(12);
          write_pimg(t, nullptr, false, rec ? slot + SLOT_P : nullptr);
          fence_proxy_async();
          mbar_arrive(&b->p_full);
          stamp(13);
        }
        if (ROLE == ROLE_EPI) {
          bar_sync(BAR_D3, XCHG_THREADS);                   // delta3 of every row is in MiscF::d3s
        }
        // ---- delta2 image (in place over h2) feeding the dX UMMAs block by block ----
        if (ROLE == ROLE_MMA) stamp(3);
        gemm_issue<ROLE>(0, b, smem, sy, A.pol.big_dx, tm_work);   // g_h1
        if (ROLE == ROLE_MMA) stamp(4);
        if (ROLE == ROLE_EPI) {
          stamp(6);
          epi_delta2_from_h2<ACT>(b, mf->W3p, mf->d3s[row], mf->d3s[ACT_ROWS + row], act_img, row, hc, (sy.i_cnt - 1) & 1,
                             want_dw ? &sy : nullptr);
          stamp(7);
          if (rec) store_image_follow(elected, b, sy, slot + SLOT_D2, act_img, A.rec_hi_only != 0);   // delta2 blocks leave behind their K-blocks
          epi_wait_d(b, sy);                                       // g_h1 complete, delta2 image consumed
          stamp(8);
        }
        // z1 recompute stream, g_p following the delta1 blocks, D1 += delta1^T [p|1]
        bwd_tail_issue<ROLE>(b, smem, sy, A.pol.l1b, A.pol.in, t > 0, want_dw, d1_started, tm_z1c, tm_gp, tm_d1, true, early_next);
        if (ROLE == ROLE_PRODUCER && early_next) load_h2(t - 1);
        if (ROLE == ROLE_EPI) {
          epi_delta1_blocks<ACT>(b, tm_work + lane_off, tm_z1c + lane_off, act_img, row, hc, rec, elected, early_next);
          stamp(9);
          if (t > 0) epi_wait_d(b, sy);
          stamp(10);
        }
        if (want_dw) { d1_pending = true; ++acc_issued; }
        if (t > 0 && rowthread) {
          mbar_wait(&b->gp_full, sy.gp_cnt & 1, 20000 + __LINE__);
          ++sy.gp_cnt;
          tc_fence_after();
          stamp(10);
          float gin[16];
          read_gp(tm_gp + lane_off, gin);
          if (valid) {
#pragma unroll
            for (int j = 0; j < S; ++j) { lam[j] = g_s[j]; snext[j] = s[j]; }
            float go[MPG_MAX_OBS];
#pragma unroll
            for (int i = 0; i < MPG_MAX_OBS; ++i) go[i] = i < a.obs_dim ? gin[i] * a.obs_scale[i] : 0.f;
            E::obs_grad_to_state(s, go, a.nfd, lam);
          }
        }
        stamp(11);
      }
    }
  }
  if (rowthread && BWD) {
    // db3: per-row partial sums -> per-warp (shuffle tree) -> fixed-order total
    float s0 = db3acc[0], s1 = db3acc[1];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
    if (lane == 0) { mf->wsum[(warp & 3) * 2] = s0; mf->wsum[(warp & 3) * 2 + 1] = s1; }
    bar_sync(BAR_ROW, ROW_THREADS);
    if (tid == EPI_THREADS) {
      const GradLayout L(A.pol.in_dim, A.pol.out_dim, H, 2);
      float* partial = a.partial + (size_t)blockIdx.x * a.partial_stride;
      partial[L.obout + 0] = (mf->wsum[0] + mf->wsum[2]) + (mf->wsum[4] + mf->wsum[6]);
      if (NA > 1) partial[L.obout + 1] = (mf->wsum[1] + mf->wsum[3]) + (mf->wsum[5] + mf->wsum[7]);
    }
  }
  if (ROLE == ROLE_EPI && acc_issued > 0) mbar_wait(&b->acc_done, (acc_issued - 1) & 1, 20000 + __LINE__);   // last D1 accumulation complete
  if (ROLE == ROLE_EPI) {
    tc_fence_before();
    if (elected) bulk_wait_all();
    if (BWD) {
      const GradLayout L(A.pol.in_dim, A.pol.out_dim, H, 2);
      float* partial = a.partial + (size_t)blockIdx.x * a.partial_stride;
      if (any_dw && hc == 0) {
        // D1 / D3: TMEM lane = feature inside the 128-feature half, columns = input index (BIAS_K: bias) / action
        tc_fence_after();
        const int ncol3 = A.q_regress ? 1 : NA;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int f = half * 128 + row;
          float v[16], v2[16];
          tmem_ld16(tm_d1 + half * 32 + lane_off, v);
          tmem_ld16(tm_d1 + half * 32 + 16 + lane_off, v2);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < A.pol.in_dim) partial[L.oW1 + (size_t)i * H + f] = v[i] + v2[i];
          partial[L.ob1 + f] = v[BIAS_K] + v2[BIAS_K];
          tmem_ld16(tm_d3 + half * 16 + lane_off, v);
#pragma unroll
          for (int j = 0; j < 2; ++j)
            if (j < ncol3) partial[L.oWout + (size_t)f * A.pol.out_dim + j] = v[j] + v[2 + j];
        }
      }
    }
  }
}

// The rollout kernel is launched with SIX warpgroups: four epilogue warpgroups (16 warps), the row warpgroup (4 warps,
// thread = trajectory) and one that holds the producer warp, the mma warp and two idle warps.  setmaxnreg moves registers
// inside the CTA's launch allocation (768 threads x 80 registers) from the last warpgroup to the row warpgroup.  Why it
// matters: with 221 KB of shared memory in use only ~7 KB of L1 is left, so every register spill is an L2 round trip
// (~270 cycles) -- and the scalar recurrence of a row (state, adjoint, checkpoints) used to be spilled around the 16-wide
// epilogue vectors when the same threads did both jobs.
constexpr int ROLLOUT_THREADS = EPI_THREADS + ROW_THREADS + 128;
constexpr int ROW_WARP0 = EPI_WARPS, PRODUCER_WARP = EPI_WARPS + 4, MMA_WARP = EPI_WARPS + 5;
constexpr int LAUNCH_REGS = 80, EPI_REGS = 80, ROW_REGS = 96, AUX_REGS = 64;
static_assert(EPI_THREADS * EPI_REGS + ROW_THREADS * ROW_REGS + 128 * AUX_REGS <= ROLLOUT_THREADS * LAUNCH_REGS,
              "setmaxnreg only redistributes the register pool of the CTA");

template <int ENV, bool BWD, int ACT>
__global__ void __launch_bounds__(ROLLOUT_THREADS, 1) tc_rollout_kernel(const __grid_constant__ TcArgs A) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  MiscF* mf = reinterpret_cast<MiscF*>(smem + SmemMap::MISC);
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    mf->b2p[i] = A.pol.b2[i];
    mf->W3p[2 * i] = A.pol.W3[i * A.pol.out_dim];
    mf->W3p[2 * i + 1] = Env<ENV>::A > 1 ? A.pol.W3[i * A.pol.out_dim + 1] : 0.f;
    if (A.r.has_q) {
      mf->b2q[i] = A.q.b2[i];
      mf->W3q[2 * i] = A.q.W3[i];
      mf->W3q[2 * i + 1] = 0.f;
    }
  }
  for (int i = threadIdx.x; i < 8192 / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem + SM_D3IMG)[i] = make_uint4(0u, 0u, 0u, 0u);
  build_step_tab(*reinterpret_cast<StepTab*>(smem + SM_TAB), A.r.list, A.r.list_w, A.r.n_list, A.r.far_steps, threadIdx.x,
                 blockDim.x);
  if (threadIdx.x == 0) {
    mf->b3[0] = A.pol.b3[0];
    mf->b3[1] = Env<ENV>::A > 1 ? A.pol.b3[1] : 0.f;
    mf->b3[2] = A.r.has_q ? A.q.b3[0] : 0.f;
  }
  Bars* b = cta_setup(smem, XCHG_THREADS, MMA_WARP);   // contains __syncthreads()
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp < EPI_WARPS) {
    run_rollout<ENV, BWD, ACT, ROLE_EPI>(A, smem, b);
  } else if (warp < PRODUCER_WARP) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(ROW_REGS));
    run_rollout<ENV, BWD, ACT, ROLE_ROW>(A, smem, b);
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AUX_REGS));
    if (warp == PRODUCER_WARP) { if (elect_one()) run_rollout<ENV, BWD, ACT, ROLE_PRODUCER>(A, smem, b); }
    else if (warp == MMA_WARP) { if (elect_one()) run_rollout<ENV, BWD, ACT, ROLE_MMA>(A, smem, b); }
  }
  cta_teardown(b, MMA_WARP);
}

}  // namespace tc
}  // namespace mpg
