// Tensor-core (tcgen05) path: state owned by the handle, weight-image packing, development self tests.  Included by api.cu
// only; the rollout kernel, which depends on the hidden activation, is launched through mlp_kernels.cuh.
#pragma once
#include "tc_dw.cuh"
#ifdef MPG_DEBUG_PROBES
#include "tc_pair_probe.cuh"
#endif

namespace mpg {
namespace tc {

// ---- global weight-image packing (run once per set_weights) ------------------------------------------------
// big image: value(row, k) = src[row * rs + k * cs], 256 rows x 256 k -> 16 stages (kb, split, kh) of 256 rows x 64 B,
// SW64 K-major (8-row groups of 512 B, 16-byte chunk index ^ ((row >> 1) & 3))
template <bool F16>
__global__ void pack_big_image(const float* __restrict__ src, int rs, int cs, uint8_t* __restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // one thread per (row, 8-element chunk): 256 x 32
  if (idx >= 256 * 32) return;
  const int row = idx >> 5, cc = idx & 31;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = src[(size_t)row * rs + (size_t)(cc * 8 + e) * cs];
  uint4 h, l;
  split2x<F16>(x[0], x[1], h.x, l.x); split2x<F16>(x[2], x[3], h.y, l.y); split2x<F16>(x[4], x[5], h.z, l.z); split2x<F16>(x[6], x[7], h.w, l.w);
  const int kb = cc >> 3, kh = (cc >> 2) & 1, c = cc & 3;
  const size_t stage = (size_t)(kb * 4 + kh) * STAGE_BYTES;   // streamed in (k-block, split, k-half) order
  const uint32_t off = (row >> 3) * 512 + (row & 7) * 64 + ((c ^ ((row >> 1) & 3)) << 4);
  *reinterpret_cast<uint4*>(img + stage + off) = h;
  *reinterpret_cast<uint4*>(img + stage + 2 * STAGE_BYTES + off) = l;
}
// first-layer image: value(n, k) = scale * (k < in_dim ? W1[k][n] : (k == bias_k ? b1[n] : 0)); 256 rows x 16 k,
// (scale = log2(e) for the bf16 image of the BPTT recompute, whose z1 only feeds act'(z1), e.g. elu'(z1) = 2^(min(z1, 0) log2 e))
// INTERLEAVE K-major: [hi 8 KB | lo 8 KB]
template <bool F16>
__global__ void pack_l1_image(const float* __restrict__ W1, const float* __restrict__ b1, int in_dim, int bias_k,
                              uint8_t* __restrict__ img, float scale = 1.f) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (n, k-half): 256 x 2
  if (idx >= 512) return;
  const int n = idx >> 1, kh = idx & 1;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = kh * 8 + e;
    x[e] = scale * (k < in_dim ? W1[(size_t)k * H + n] : (k == bias_k ? b1[n] : 0.f));
  }
  uint4 h, l;
  split2x<F16>(x[0], x[1], h.x, l.x); split2x<F16>(x[2], x[3], h.y, l.y); split2x<F16>(x[4], x[5], h.z, l.z); split2x<F16>(x[6], x[7], h.w, l.w);
  const uint32_t off = il_chunk_off(n, kh);
  *reinterpret_cast<uint4*>(img + off) = h;
  *reinterpret_cast<uint4*>(img + 8192 + off) = l;
}
// input-gradient image: value(i, n) = i < in_dim ? W1[i][n] : 0; per 64-k block 32 rows (hi of rows 0..15, then lo of rows
// 0..15) x 128 B, SW128 K-major: 4 x 4 KB
__global__ void pack_in_image(const float* __restrict__ W1, int in_dim, uint8_t* __restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (i, chunk): 16 x 32
  if (idx >= 512) return;
  const int i = idx >> 5, cc = idx & 31;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = i < in_dim ? W1[(size_t)i * H + cc * 8 + e] : 0.f;
  uint4 h, l;
  split2(x[0], x[1], h.x, l.x); split2(x[2], x[3], h.y, l.y); split2(x[4], x[5], h.z, l.z); split2(x[6], x[7], h.w, l.w);
  const int kb = cc >> 3, c = cc & 7;
  auto off = [&](int row) { return (uint32_t)(kb * 4096 + (row >> 3) * 1024 + (row & 7) * 128 + ((c ^ (row & 7)) << 4)); };
  *reinterpret_cast<uint4*>(img + off(i)) = h;
  *reinterpret_cast<uint4*>(img + off(16 + i)) = l;
}

#ifdef MPG_DEBUG_PROBES
// ---- self test: the three GEMM kinds against caller-provided fp32 data ---------------------------------------
//   kind 0: Z[128 x 256] = X[128 x 256] . (image of Wt[256 x 256])^T
//   kind 1: Z[128 x 256] = X16[128 x 16] . (first-layer image)^T
//   kind 2: Z[128 x 16]  = X[128 x 256] . (input-gradient image)^T
__global__ void __launch_bounds__(CTA_THREADS, 1) selftest_kernel(int kind, const float* __restrict__ X,
                                                                 const uint8_t* __restrict__ img, float* __restrict__ Z,
                                                                 int repeats) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SW128 needs 1024-byte alignment
  Bars* b = cta_setup(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem = b->tmem_base;
  Sync s;
  if (warp < EPI_WARPS) {
    const int row = (warp & 3) * 32 + lane, hc = warp >> 2;
    constexpr int CW = COLS_PER_WARP;
    for (int rep = 0; rep < repeats; ++rep) {
      if (kind >= 3) {          // timing probes: back-to-back big GEMMs on whatever the images hold, one wait at the end
        if (rep == repeats - 1) epi_wait_d(b, s);
        continue;
      }
      if (kind == 1) {
        if (hc == 0) {
          for (int kh = 0; kh < 2; ++kh) {
            float x[8];
            for (int e = 0; e < 8; ++e) x[e] = X[row * 16 + kh * 8 + e];
            uint4 h, l;
            split2h(x[0], x[1], h.x, l.x); split2h(x[2], x[3], h.y, l.y); split2h(x[4], x[5], h.z, l.z); split2h(x[6], x[7], h.w, l.w);
            *reinterpret_cast<uint4*>(smem + SmemMap::PIMG + p_chunk_off(row, kh)) = h;
            *reinterpret_cast<uint4*>(smem + SmemMap::PIMG + p_chunk_off(row, 2 + kh)) = l;
          }
        }
      } else {
        for (int cc = hc * (CW / 8); cc < (hc + 1) * (CW / 8); ++cc) {
          float x[8];
          for (int e = 0; e < 8; ++e) x[e] = X[row * 256 + cc * 8 + e];
          act_store8(smem + SmemMap::ACT, smem + SmemMap::ACT + ACT_SPLIT, row, cc, x);
        }
      }
      gemm<ROLE_EPI>(kind, b, smem, s, img, tmem + TM_WORK);
      const uint32_t lane_base = tmem + TM_WORK + ((uint32_t)((warp & 3) * 32) << 16);
      if (kind == 2) {
        if (hc == 0) {
          float v[16], v2[16];
          tmem_ld16(lane_base, v);
          tmem_ld16(lane_base + 16, v2);
          for (int j = 0; j < 16; ++j) Z[row * 16 + j] = v[j] + v2[j];
        }
      } else {
        for (int c0 = hc * CW; c0 < (hc + 1) * CW; c0 += 32) {
          float v[32];
          tmem_ld32(lane_base + c0, v);
          for (int j = 0; j < 32; ++j) Z[row * 256 + c0 + j] = v[j];
        }
      }
    }
    tc_fence_before();
  } else if (warp == EPI_WARPS) {
    if (lane == 0)
      for (int rep = 0; rep < repeats; ++rep)
        if (kind != 4) gemm<ROLE_PRODUCER>(kind == 3 ? 0 : kind, b, smem, s, img, 0);
  } else {
    if (lane == 0)
      for (int rep = 0; rep < repeats; ++rep) {
        if (kind == 3) {          // weights streamed through the ring, no epilogue in the loop
          mma_big<FMT_BF16>(b, smem_u32(smem) + SmemMap::ACT, smem_u32(smem) + SmemMap::RING, s, tmem + TM_WORK, false);
          if (rep == repeats - 1) mma_publish_d(b);
        } else if (kind == 4) {   // operands resident, no streaming: the tensor pipe's own rate for this shape
          constexpr uint32_t idesc = make_idesc(128, 256, 0, 0);
          const uint32_t act = smem_u32(smem) + SmemMap::ACT, ring = smem_u32(smem) + SmemMap::RING;
          for (int k = 0; k < 16; ++k) {
            const uint64_t ko = (uint64_t)((k & 3) * 2);
            const uint64_t dah = make_desc(act + (k >> 2) * ACT_BLOCK, 16, 1024, LAYOUT_SW128) + ko;
            const uint64_t dal = make_desc(act + ACT_SPLIT + (k >> 2) * ACT_BLOCK, 16, 1024, LAYOUT_SW128) + ko;
            const uint64_t dbh = make_desc(ring, 16, 1024, LAYOUT_SW128) + ko;
            const uint64_t dbl = make_desc(ring + 32768, 16, 1024, LAYOUT_SW128) + ko;
            umma_bf16(tmem + TM_WORK, dah, dbh, idesc, 1u);
            umma_bf16(tmem + TM_WORK, dal, dbh, idesc, 1u);
            umma_bf16(tmem + TM_WORK, dah, dbl, idesc, 1u);
          }
          if (rep == repeats - 1) mma_publish_d(b);
        } else {
          gemm<ROLE_MMA>(kind, b, smem, s, img, tmem + TM_WORK);
        }
      }
  }
  cta_teardown(b);
}
#endif

}  // namespace tc

struct TcNetImages {
  uint8_t* big_fwd = nullptr;   // Wt[n][k] = W2[k][n]   (z2 = h1 . W2)
  uint8_t* big_dx = nullptr;    // Wt[k][n] = W2[k][n]   (g_h1 = delta2 . W2^T)
  uint8_t* l1 = nullptr;        // [W1; b1] as 256 x 16, fp16 pair (forward)
  uint8_t* l1b = nullptr;       // the same as a bf16 pair (BPTT)
  uint8_t* in = nullptr;        // W1 as 16 x 256 (input gradient)
};

struct TcState {
  bool ready = false;
  TcNetImages nets[MPG_NUM_NETS];
  uint8_t* scratch_img = nullptr;   // self-test image
  DevBuf<float> act_ckpt;           // [n_list][max_rows][MAX_A]: MPG_MAX_LIST entries at creation, grows with longer lists
  float* z_ckpt = nullptr;          // [max_horizon+1][max_rows][2 MAX_A] action and head derivative of every step (BPTT)
  DevBuf<uint8_t> store;            // dW operand store (allocated on first use)
  DevBuf<uint8_t> h2store;          // h2 images of the forward pass, [tile][step][128 KB] (allocated on first use)
};

template <typename K>
inline bool tc_set_smem(K kernel, int bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess;
}

inline bool tc_init(TcState& t, const mpg_config& cfg, int hidden_layers, int /*sms*/, size_t& ws_bytes) {
  if (cfg.hidden != tc::H) return true;                  // every layout of this path is built for 256; stay on FFMA
  if (hidden_layers != 2) return true;                   // and for two hidden layers; stay on FFMA
  if (cfg.obs_dim + cfg.act_dim + 1 > 16) return true;   // first-layer K must fit one UMMA k-step; stay on FFMA
  auto alloc = [&](void** p, size_t n) {
    if (cudaMalloc(p, n) != cudaSuccess) return false;
    ws_bytes += n;
    return true;
  };
  const size_t act_ckpt_n = (size_t)MPG_MAX_LIST * cfg.max_rows * MAX_A;
  bool ok = alloc((void**)&t.scratch_img, tc::BIG_IMAGE_BYTES) && t.act_ckpt.grow(act_ckpt_n) == cudaSuccess
            && alloc((void**)&t.z_ckpt, (size_t)(cfg.max_horizon + 1) * cfg.max_rows * 2 * MAX_A * sizeof(float));
  if (ok) ws_bytes += act_ckpt_n * sizeof(float);
  for (int n = 0; n < MPG_NUM_NETS && ok; ++n)
    ok = alloc((void**)&t.nets[n].big_fwd, tc::BIG_IMAGE_BYTES) && alloc((void**)&t.nets[n].big_dx, tc::BIG_IMAGE_BYTES)
         && alloc((void**)&t.nets[n].l1, 16384) && alloc((void**)&t.nets[n].l1b, 16384) && alloc((void**)&t.nets[n].in, 16384);
  if (!ok) return false;
  // the rollout kernels are set up with the other activation-dependent kernels (MlpKernels::set_smem)
  ok = tc_set_smem(tc::tc_dw_kernel, tc::DW_SMEM);
#ifdef MPG_DEBUG_PROBES
  ok = ok && tc_set_smem(tc::selftest_kernel, tc::SmemMap::TOTAL + 1024) && tc_set_smem(tc::pair_probe_kernel, tc::PAIR_SMEM);
#endif
  t.ready = ok;
  return ok;
}

inline void tc_destroy(TcState& t) {
  cudaFree(t.scratch_img); t.act_ckpt.release(); cudaFree(t.z_ckpt); t.h2store.release(); t.store.release();
  for (int n = 0; n < MPG_NUM_NETS; ++n) {
    cudaFree(t.nets[n].big_fwd); cudaFree(t.nets[n].big_dx); cudaFree(t.nets[n].l1); cudaFree(t.nets[n].l1b); cudaFree(t.nets[n].in);
  }
}

// flat: Keras-order natural weights W1|b1|W2|b2|W3|b3 on the device
inline bool tc_pack_weights(TcState& t, int net, const float* flat, int in_dim, int out_dim, cudaStream_t st) {
  if (!t.nets[net].big_fwd) return true;   // tensor-core path not configured for this handle
  const GradLayout L(in_dim, out_dim, tc::H, 2);
  tc::pack_big_image<true><<<32, 256, 0, st>>>(flat + L.oW(2), 1, tc::H, t.nets[net].big_fwd);     // value(n,k) = W2[k][n]
  tc::pack_big_image<false><<<32, 256, 0, st>>>(flat + L.oW(2), tc::H, 1, t.nets[net].big_dx);      // value(k,n) = W2[k][n]
  tc::pack_l1_image<true><<<2, 256, 0, st>>>(flat + L.oW1, flat + L.ob1, in_dim, tc::BIAS_K, t.nets[net].l1);
  tc::pack_l1_image<false><<<2, 256, 0, st>>>(flat + L.oW1, flat + L.ob1, in_dim, tc::BIAS_K, t.nets[net].l1b, 1.4426950408889634f);   // z1 log2(e) for every activation, see act_grad_log2e
  tc::pack_in_image<<<2, 256, 0, st>>>(flat + L.oW1, in_dim, t.nets[net].in);
  return cudaGetLastError() == cudaSuccess;
}

inline tc::TcNet tc_net(const TcState& t, int net, const float* flat, int in_dim, int out_dim) {
  const GradLayout L(in_dim, out_dim, tc::H, 2);
  tc::TcNet n;
  n.big_fwd = t.nets[net].big_fwd; n.big_dx = t.nets[net].big_dx; n.l1 = t.nets[net].l1; n.l1b = t.nets[net].l1b; n.in = t.nets[net].in;
  n.W3 = flat + L.oWout; n.b2 = flat + L.ob(2); n.b3 = flat + L.obout;
  n.in_dim = in_dim; n.out_dim = out_dim;
  return n;
}

#ifdef MPG_DEBUG_PROBES
// self test of one GEMM kind (see tc_gemm.cuh): W is fp32 [256 x 256] (kind 0), [16 x 256] (kinds 1, 2)
inline cudaError_t tc_selftest(TcState& t, int kind, const float* X, const float* W, float* Z, int repeats, cudaStream_t st) {
  if (!t.scratch_img) return cudaErrorNotSupported;
  if (kind == 5) {   // CTA-pair probe: X is [256 x 256], Z is [256 x 256]; MPG_SELFTEST_GRID CTAs (even), default 2
    const char* g = getenv("MPG_SELFTEST_GRID");
    int grid = g ? atoi(g) & ~1 : 2;
    if (grid < 2) grid = 2;
    tc::pack_pair_image<<<32, 256, 0, st>>>(W, tc::H, 1, t.scratch_img);
    tc::pair_probe_kernel<<<grid, 192, tc::PAIR_SMEM, st>>>(X, t.scratch_img, Z, repeats);
    return cudaGetLastError();
  }
  if (kind >= 3) {   // timing probes (tools/gemm_probe.py): MPG_SELFTEST_GRID CTAs run the big GEMM `repeats` times
    const char* g = getenv("MPG_SELFTEST_GRID");
    tc::selftest_kernel<<<g ? atoi(g) : 1, tc::CTA_THREADS, tc::SmemMap::TOTAL + 1024, st>>>(kind, X, t.scratch_img, Z, repeats);
    return cudaGetLastError();
  }
  if (kind == 0) tc::pack_big_image<false><<<32, 256, 0, st>>>(W, tc::H, 1, t.scratch_img);
  else if (kind == 1) tc::pack_l1_image<true><<<2, 256, 0, st>>>(W, W, 16, -1, t.scratch_img);
  else tc::pack_in_image<<<2, 256, 0, st>>>(W, 16, t.scratch_img);
  tc::selftest_kernel<<<1, tc::CTA_THREADS, tc::SmemMap::TOTAL + 1024, st>>>(kind, X, t.scratch_img, Z, repeats);
  return cudaGetLastError();
}
#endif

}  // namespace mpg
