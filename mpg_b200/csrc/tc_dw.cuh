// tc_dw_kernel: the weight-gradient GEMMs of the tensor-core path, over the dW operand store tc_rollout_kernel writes.  It
// does not depend on the hidden activation, so only api.cu compiles it.
#pragma once
#include "tc_kernels.cuh"

namespace mpg {
namespace tc {

// =================================================================================================
// dW2 / db2 from the operand store: split-K tcgen05 GEMMs with MN-major operands (K = rows).
// CTA c owns feature half mh = c & 1 of the left operand and the records r = c>>1, c>>1 + G/2, ...
//   D2  [128 x 256] += h1[:, mh]^T . delta2            -> dW2[k][n]
//   Db2 [128 x 16]  += delta2[:, mh]^T . [p|1]         -> column BIAS_K = db2[n]
// (dW1, db1, dW3 are accumulated inside the rollout kernel, db3 is a shuffle reduction there.)
// =================================================================================================
struct DwArgs {
  const uint8_t* store;
  int nrecords;            // tiles * store_steps
  int in_dim, out_dim;     // gradient layout of the net
  float* partial;
  long long partial_stride;
  int hi_only;             // records hold only the hi planes: one product per contraction instead of three
};

#ifndef MPG_DW_ROWS
#define MPG_DW_ROWS 32
#endif
#ifndef MPG_DW_NSTAGE
#define MPG_DW_NSTAGE 4
#endif
constexpr int DW_ROWS = MPG_DW_ROWS;                            // rows (K) per stage (multiple of the UMMA k-step)
constexpr int DW_NSTAGE = MPG_DW_NSTAGE;                        // ring depth: bytes in flight per SM set the HBM rate
constexpr int DW_BLK = DW_ROWS * 128;                           // one 64-feature block of one stage
constexpr int DW_R16 = DW_ROWS * 32;                            // one [rows x 16] bf16 image of one stage
constexpr int DW_OFF_H1 = 0, DW_OFF_D2 = 4 * DW_BLK, DW_OFF_P = 12 * DW_BLK;
constexpr int DW_STAGE = DW_OFF_P + 2 * DW_R16;                 // bytes per stage (50 KB)
constexpr int DW_COPIES = 14;                                   // bulk copies per stage, one lane each
constexpr int DW_SMEM = DW_NSTAGE * DW_STAGE + 256 + 1024;      // dynamic shared memory of tc_dw_kernel
constexpr int DW_TM_D2 = 0, DW_TM_DB2 = 256;
static_assert(DW_STAGE % 1024 == 0 && DW_ROWS % 16 == 0, "stages hold whole SW128 atoms and UMMA k-steps");
static_assert(DW_SMEM <= 232448, "tc_dw_kernel shared memory");


struct DwBars {
  uint64_t full[DW_NSTAGE], empty[DW_NSTAGE], conv[DW_NSTAGE], d_full;
  uint32_t tmem_base;
};

constexpr int DW_CONV_WARPS = 8;                                // warps 0..7 convert h1 (0..3 also read the accumulators out)
constexpr int DW_THREADS = (DW_CONV_WARPS + 2) * 32;           // + producer warp + mma warp
__global__ void __launch_bounds__(DW_THREADS, 1) tc_dw_kernel(const __grid_constant__ DwArgs A) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* stage_buf = smem;                                    // DW_NSTAGE x DW_STAGE
  DwBars* b = reinterpret_cast<DwBars*>(smem + DW_NSTAGE * DW_STAGE);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < DW_NSTAGE; ++i) { mbar_init(&b->full[i], 1); mbar_init(&b->empty[i], 1); mbar_init(&b->conv[i], DW_CONV_WARPS * 32); }
    mbar_init(&b->d_full, 1);
    fence_barrier_init();
  }
  if (warp == DW_CONV_WARPS + 1) tmem_alloc(&b->tmem_base, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = b->tmem_base;
  const int mh = blockIdx.x & 1, first = blockIdx.x >> 1, stride = gridDim.x >> 1;
  const int nmine = first < A.nrecords ? (A.nrecords - first + stride - 1) / stride : 0;
  const int nstages = nmine * (ACT_ROWS / DW_ROWS);

  if (warp == DW_CONV_WARPS) {
    // ------------------------------- producer: one lane per bulk copy of a stage -------------------------------
    const int sp = lane / 7, k = lane % 7;
    size_t src = 0; uint32_t dsto = 0, bytes = DW_BLK, qstep = DW_BLK;
    if (k < 2) {            // left operand h1: the two 64-feature blocks of half mh
      src = SLOT_H1 + (size_t)sp * ACT_SPLIT + (size_t)(2 * mh + k) * ACT_BLOCK;
      dsto = DW_OFF_H1 + (sp * 2 + k) * DW_BLK;
    } else if (k < 6) {     // right operand delta2: all four blocks
      src = SLOT_D2 + (size_t)sp * ACT_SPLIT + (size_t)(k - 2) * ACT_BLOCK;
      dsto = DW_OFF_D2 + (sp * 4 + (k - 2)) * DW_BLK;
    } else {                // [p|1] image: hi and lo chunks of an 8-row group are adjacent, one copy takes both
      src = SLOT_P;
      dsto = DW_OFF_P;
      bytes = sp == 0 ? 2 * DW_R16 : 0; qstep = 2 * DW_R16;
    }
    uint32_t slot = 0, par = 0;
    for (int r = first; r < A.nrecords; r += stride) {
      const uint8_t* rec = A.store + (size_t)r * SLOT_BYTES;
      for (int q = 0; q < ACT_ROWS / DW_ROWS; ++q) {
        if (lane == 0) {
          mbar_wait(&b->empty[slot], par ^ 1, 20000 + __LINE__);
          mbar_expect_tx(&b->full[slot], A.hi_only ? 6 * DW_BLK + 2 * DW_R16 : DW_STAGE);
        }
        __syncwarp();
        if (lane < DW_COPIES && bytes && !(A.hi_only && sp == 1 && k < 6)) bulk_g2s(stage_buf + slot * DW_STAGE + dsto, rec + src + (size_t)q * qstep, bytes, &b->full[slot]);
        if (++slot == DW_NSTAGE) { slot = 0; par ^= 1; }
      }
    }
  } else if (warp == DW_CONV_WARPS + 1) {
    // ------------------------------- mma -------------------------------
    if (elect_one()) {
      constexpr uint32_t id256 = make_idesc(128, 256, 1, 1), id16 = make_idesc(128, 16, 1, 1);
      const uint32_t sbase = smem_u32(stage_buf);
      uint32_t slot = 0, par = 0;
      for (int st = 0; st < nstages; ++st) {
        mbar_wait(&b->conv[slot], par, 20000 + __LINE__);      // stage landed and its h1 part converted to a bf16 pair
        tc_fence_after();
        const uint32_t base = sbase + slot * DW_STAGE;
#pragma unroll
        for (int ks = 0; ks < DW_ROWS / 16; ++ks) {
          const uint32_t acc = (st | ks) ? 1u : 0u;
          // left operand (MN-major SW128, M = 128 features = 2 blocks DW_BLK apart, 8-row groups 1024 B apart)
          auto L = [&](int sp) { return make_desc(base + DW_OFF_H1 + sp * 2 * DW_BLK + ks * 2048, DW_BLK, 1024, LAYOUT_SW128); };
          // right operand delta2 (N = 256 = 4 blocks)
          auto R2 = [&](int sp) { return make_desc(base + DW_OFF_D2 + sp * 4 * DW_BLK + ks * 2048, DW_BLK, 1024, LAYOUT_SW128); };
          // delta2 as LEFT operand for db2: its blocks 2mh, 2mh+1 inside the right-operand buffer
          auto LD2 = [&](int sp) { return make_desc(base + DW_OFF_D2 + sp * 4 * DW_BLK + mh * 2 * DW_BLK + ks * 2048, DW_BLK, 1024, LAYOUT_SW128); };
          // right operand [p|1] (MN-major INTERLEAVE, N = 16: halves 128 B apart (SBO), 8-row groups 256 B apart (LBO));
          // only its hi split is needed: the constant-1 column is exact in bf16
          const uint64_t rp = make_desc(base + DW_OFF_P + ks * 2 * P_GROUP, P_GROUP, 128, LAYOUT_NONE);
          umma_bf16(tmem + DW_TM_D2, L(0), R2(0), id256, acc);
          if (!A.hi_only) {
            umma_bf16(tmem + DW_TM_D2, L(1), R2(0), id256, 1u);
            umma_bf16(tmem + DW_TM_D2, L(0), R2(1), id256, 1u);
          }
          umma_bf16(tmem + DW_TM_DB2, LD2(0), rp, id16, acc);
          if (!A.hi_only) umma_bf16(tmem + DW_TM_DB2, LD2(1), rp, id16, 1u);
        }
        umma_commit(&b->empty[slot]);
        if (++slot == DW_NSTAGE) { slot = 0; par ^= 1; }
      }
      umma_commit(&b->d_full);
    }
  } else {
    // ------------- converter + epilogue warps -------------
    // The forward pass keeps h1 as an fp16 pair (the precision the layer-2 GEMM needs); delta2 is a bf16 pair (exponent
    // range) and one UMMA cannot mix the two formats, so the h1 part of every stage is rewritten in place as a bf16 pair
    // (16 significant bits: what the weight gradient had before) while the next stages are still in flight.
    {
      uint32_t slot = 0, par = 0;
      for (int st = 0; st < nstages; ++st) {
        mbar_wait(&b->full[slot], par, 20000 + __LINE__);
        uint8_t* hi = stage_buf + slot * DW_STAGE + DW_OFF_H1;
        uint8_t* lo = hi + 2 * DW_BLK;
#pragma unroll
        for (int i = 0; i < (2 * DW_BLK / 16) / (DW_CONV_WARPS * 32); ++i) {
          const int c = (int)threadIdx.x + i * (DW_CONV_WARPS * 32);
          const uint4 h = *reinterpret_cast<const uint4*>(hi + c * 16);
          const uint4 l = A.hi_only ? make_uint4(0u, 0u, 0u, 0u) : *reinterpret_cast<const uint4*>(lo + c * 16);
          const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
          uint32_t oh[4], ol[4];
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hw[w]));
            const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&lw[w]));
            split2(a.x + d.x, a.y + d.y, oh[w], ol[w]);
          }
          *reinterpret_cast<uint4*>(hi + c * 16) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
          if (!A.hi_only) *reinterpret_cast<uint4*>(lo + c * 16) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
        }
        fence_proxy_async();
        mbar_arrive(&b->conv[slot]);
        if (++slot == DW_NSTAGE) { slot = 0; par ^= 1; }
      }
    }
    // ------------------------------- epilogue: TMEM -> this CTA's partial gradient -------------------------------
    const GradLayout L(A.in_dim, A.out_dim, H, 2);
    float* partial = A.partial + (size_t)blockIdx.x * A.partial_stride;
    const int f = mh * 128 + warp * 32 + lane;                   // feature owned by this thread (TMEM lane)
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    if (nstages > 0 && warp < 4) {
      mbar_wait(&b->d_full, 0, 20000 + __LINE__);
      tc_fence_after();
      for (int c0 = 0; c0 < 256; c0 += 32) {
        float v[32];
        tmem_ld32(tmem + DW_TM_D2 + lane_off + c0, v);
        float4* dst = reinterpret_cast<float4*>(partial + L.oW(2) + (size_t)f * H + c0);
#pragma unroll
        for (int i = 0; i < 8; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      float v[16];
      tmem_ld16(tmem + DW_TM_DB2 + lane_off, v);
      partial[L.ob(2) + f] = v[BIAS_K];
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == DW_CONV_WARPS + 1) tmem_dealloc(tmem, TMEM_COLS);
}

}  // namespace tc
}  // namespace mpg
