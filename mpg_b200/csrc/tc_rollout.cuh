// Tensor-core (tcgen05) path: state owned by the handle, weight-image packing, launchers.
#pragma once
#include <type_traits>

#include "tc_kernels.cuh"
#ifdef MPG_DEBUG_PROBES
#include "tc_pair_probe.cuh"
#endif

namespace mpg {

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
  float* act_ckpt = nullptr;        // [MPG_MAX_LIST][max_rows][MAX_A]
  float* qtmp = nullptr;            // [max_rows] Q values of the regression pass / of the target evaluations
  float* qtmp2 = nullptr;           // [max_rows] second Q value (double-Q minimum, TD error)
  float* z_ckpt = nullptr;          // [max_horizon+1][max_rows][2 MAX_A] action and head derivative of every step (BPTT)
  uint8_t* store = nullptr;         // dW operand store (allocated on first use, grows)
  size_t store_bytes = 0;
  uint8_t* h2store = nullptr;       // h2 images of the forward pass, [tile][step][128 KB] (allocated on first use, grows)
  size_t h2store_bytes = 0;
};

template <typename K>
inline bool tc_set_smem(K kernel, int bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess;
}

inline bool tc_init(TcState& t, const mpg_config& cfg, int /*sms*/, size_t& ws_bytes) {
  if (cfg.hidden != tc::H) return true;                  // every layout of this path is built for 256; stay on FFMA
  if (cfg.obs_dim + cfg.act_dim + 1 > 16) return true;   // first-layer K must fit one UMMA k-step; stay on FFMA
  auto alloc = [&](void** p, size_t n) {
    if (cudaMalloc(p, n) != cudaSuccess) return false;
    ws_bytes += n;
    return true;
  };
  bool ok = alloc((void**)&t.scratch_img, tc::BIG_IMAGE_BYTES)
            && alloc((void**)&t.act_ckpt, (size_t)MPG_MAX_LIST * cfg.max_rows * MAX_A * sizeof(float))
            && alloc((void**)&t.z_ckpt, (size_t)(cfg.max_horizon + 1) * cfg.max_rows * 2 * MAX_A * sizeof(float))
            && alloc((void**)&t.qtmp, (size_t)cfg.max_rows * sizeof(float))
            && alloc((void**)&t.qtmp2, (size_t)cfg.max_rows * sizeof(float));
  for (int n = 0; n < MPG_NUM_NETS && ok; ++n)
    ok = alloc((void**)&t.nets[n].big_fwd, tc::BIG_IMAGE_BYTES) && alloc((void**)&t.nets[n].big_dx, tc::BIG_IMAGE_BYTES)
         && alloc((void**)&t.nets[n].l1, 16384) && alloc((void**)&t.nets[n].l1b, 16384) && alloc((void**)&t.nets[n].in, 16384);
  if (!ok) return false;
  const int sm = tc::SM_TOTAL + 1024;
  auto set_act = [&](auto ac) {
    constexpr int ACT = decltype(ac)::value;
    return tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING, true, ACT>, sm)
           && tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING, false, ACT>, sm)
           && tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_INVERTED_PENDULUM, true, ACT>, sm)
           && tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_INVERTED_PENDULUM, false, ACT>, sm)
           && tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_INVERTED_DOUBLE_PENDULUM, true, ACT>, sm)
           && tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_INVERTED_DOUBLE_PENDULUM, false, ACT>, sm)
           && tc_set_smem(tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING_REAL, false, ACT>, sm);
  };
  ok = set_act(std::integral_constant<int, MPG_ACT_ELU>()) && set_act(std::integral_constant<int, MPG_ACT_RELU>())
       && set_act(std::integral_constant<int, MPG_ACT_TANH>()) && tc_set_smem(tc::tc_dw_kernel, tc::DW_SMEM);
#ifdef MPG_DEBUG_PROBES
  ok = ok && tc_set_smem(tc::selftest_kernel, tc::SmemMap::TOTAL + 1024) && tc_set_smem(tc::pair_probe_kernel, tc::PAIR_SMEM);
#endif
  t.ready = ok;
  return ok;
}

inline void tc_destroy(TcState& t) {
  cudaFree(t.scratch_img); cudaFree(t.act_ckpt); cudaFree(t.z_ckpt); cudaFree(t.h2store); cudaFree(t.qtmp); cudaFree(t.qtmp2); cudaFree(t.store);
  for (int n = 0; n < MPG_NUM_NETS; ++n) {
    cudaFree(t.nets[n].big_fwd); cudaFree(t.nets[n].big_dx); cudaFree(t.nets[n].l1); cudaFree(t.nets[n].l1b); cudaFree(t.nets[n].in);
  }
}

// flat: Keras-order natural weights W1|b1|W2|b2|W3|b3 on the device
inline bool tc_pack_weights(TcState& t, int net, const float* flat, int in_dim, int out_dim, cudaStream_t st) {
  if (!t.nets[net].big_fwd) return true;   // tensor-core path not configured for this handle
  const GradLayout L(in_dim, out_dim, tc::H);
  tc::pack_big_image<true><<<32, 256, 0, st>>>(flat + L.oW2, 1, tc::H, t.nets[net].big_fwd);     // value(n,k) = W2[k][n]
  tc::pack_big_image<false><<<32, 256, 0, st>>>(flat + L.oW2, tc::H, 1, t.nets[net].big_dx);      // value(k,n) = W2[k][n]
  tc::pack_l1_image<true><<<2, 256, 0, st>>>(flat + L.oW1, flat + L.ob1, in_dim, tc::BIAS_K, t.nets[net].l1);
  tc::pack_l1_image<false><<<2, 256, 0, st>>>(flat + L.oW1, flat + L.ob1, in_dim, tc::BIAS_K, t.nets[net].l1b, 1.4426950408889634f);   // z1 log2(e) for every activation, see act_grad_log2e
  tc::pack_in_image<<<2, 256, 0, st>>>(flat + L.oW1, in_dim, t.nets[net].in);
  return cudaGetLastError() == cudaSuccess;
}

inline tc::TcNet tc_net(const TcState& t, int net, const float* flat, int in_dim, int out_dim) {
  const GradLayout L(in_dim, out_dim, tc::H);
  tc::TcNet n;
  n.big_fwd = t.nets[net].big_fwd; n.big_dx = t.nets[net].big_dx; n.l1 = t.nets[net].l1; n.l1b = t.nets[net].l1b; n.in = t.nets[net].in;
  n.W3 = flat + L.oW3; n.b2 = flat + L.ob2; n.b3 = flat + L.ob3;
  n.in_dim = in_dim; n.out_dim = out_dim;
  return n;
}

inline bool tc_ensure_buf(uint8_t*& buf, size_t& have, size_t bytes) {
  if (bytes <= have) return true;
  cudaFree(buf);
  buf = nullptr; have = 0;
  if (cudaMalloc((void**)&buf, bytes) != cudaSuccess) { cudaGetLastError(); return false; }
  have = bytes;
  return true;
}
inline bool tc_ensure_store(TcState& t, size_t bytes) { return tc_ensure_buf(t.store, t.store_bytes, bytes); }
inline bool tc_ensure_h2store(TcState& t, size_t bytes) { return tc_ensure_buf(t.h2store, t.h2store_bytes, bytes); }

// act: MPG_ACT_* of the handle
template <bool BWD>
inline cudaError_t tc_launch_rollout(int env, int act, const tc::TcArgs& a, int grid, cudaStream_t st) {
  const size_t smem = tc::SM_TOTAL + 1024;
  auto launch = [&](auto ac) {
    constexpr int ACT = decltype(ac)::value;
    if (env == MPG_ENV_PATH_TRACKING_REAL) {
      if (BWD) return cudaErrorNotSupported;
      tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING_REAL, false, ACT><<<grid, tc::ROLLOUT_THREADS, smem, st>>>(a);
      return cudaGetLastError();
    }
    switch (env) {
      case MPG_ENV_PATH_TRACKING: tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING, BWD, ACT><<<grid, tc::ROLLOUT_THREADS, smem, st>>>(a); break;
      case MPG_ENV_INVERTED_PENDULUM: tc::tc_rollout_kernel<MPG_ENV_INVERTED_PENDULUM, BWD, ACT><<<grid, tc::ROLLOUT_THREADS, smem, st>>>(a); break;
      default: tc::tc_rollout_kernel<MPG_ENV_INVERTED_DOUBLE_PENDULUM, BWD, ACT><<<grid, tc::ROLLOUT_THREADS, smem, st>>>(a); break;
    }
    return cudaGetLastError();
  };
  switch (act) {
    case MPG_ACT_RELU: return launch(std::integral_constant<int, MPG_ACT_RELU>());
    case MPG_ACT_TANH: return launch(std::integral_constant<int, MPG_ACT_TANH>());
    default: return launch(std::integral_constant<int, MPG_ACT_ELU>());
  }
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
