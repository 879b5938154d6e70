// Every kernel whose code depends on the hidden activation ACT (MPG_ACT_*): the FFMA tile kernels at each hidden width and
// the tensor-core rollout kernel, behind one table per (H, ACT).  act_elu.cu, act_relu.cu and act_tanh.cu each instantiate
// the tables of one activation, so that the three sets compile in parallel translation units, and each unit launches only
// the kernels it instantiates.  api.cu reaches them only through mlp_kernels().
#pragma once
#include "rollout_kernels.cuh"
#include "tc_kernels.cuh"

namespace mpg {

// every kernel whose code depends on the hidden activation, at one (H, ACT).  The launches return nothing about the launch
// itself: the caller reads that with cudaGetLastError(), as after any <<<...>>>.
struct MlpKernels {
  cudaError_t (*set_smem)();   // max dynamic shared memory of each kernel below
  // false: no such kernel (backward on the real environment, see with_env)
  bool (*rollout)(int env, bool bwd, const RolloutArgs& a, int grid, cudaStream_t st);
  void (*q_grad)(const QGradArgs& a, int grid, cudaStream_t st);
  void (*eval)(const EvalArgs& a, int grid, cudaStream_t st);
  void (*env_sample)(const SampleArgs& a, int grid, cudaStream_t st);
  bool (*tc_rollout)(int env, bool bwd, const tc::TcArgs& a, int grid, cudaStream_t st);   // H = tc::H only, else null
  bool (*attach_watchdog)(unsigned long long* dev_ptr);   // this unit's copy of the mbarrier watchdog (tc_common.cuh)
};

// the tables of one activation at hidden width 64, 128 or 256, defined by act_elu.cu, act_relu.cu and act_tanh.cu
const MlpKernels& elu_kernels(int hidden);
const MlpKernels& relu_kernels(int hidden);
const MlpKernels& tanh_kernels(int hidden);

// the kernels of a handle: mpg_create admits widths 64, 128 and 256 only, mpg_set_activation the three MPG_ACT_* values
inline const MlpKernels& mlp_kernels(int hidden, int act) {
  switch (act) {
    case MPG_ACT_RELU: return relu_kernels(hidden);
    case MPG_ACT_TANH: return tanh_kernels(hidden);
    default: return elu_kernels(hidden);
  }
}

// the table of one (H, ACT); only the unit of activation ACT instantiates it
template <int H, int ACT>
struct MlpLaunch {
  static constexpr int SMEM = Smem<H>::FLOATS * 4, TC_SMEM = tc::SM_TOTAL + 1024;
  static constexpr int ROLLOUT_SMEM = SMEM + (int)((sizeof(StepTab) + 15) / 16 * 16);   // + the list's step tables

  static cudaError_t set_smem() {
    cudaError_t e = cudaSuccess;
    auto set = [&](auto kernel, int bytes) {
      if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    };
    for_each_env([&](auto env, auto bwd) {
      constexpr int ENV = decltype(env)::value;
      constexpr bool BWD = decltype(bwd)::value;
      set(rollout_kernel<H, ACT, ENV, BWD>, ROLLOUT_SMEM);
      if constexpr (H == tc::H) set(tc::tc_rollout_kernel<ENV, BWD, ACT>, TC_SMEM);
    });
    set(q_grad_kernel<H, ACT>, SMEM);
    set(eval_kernel<H, ACT>, SMEM);
    set(env_sample_kernel<H, ACT>, SMEM);
    return e;
  }
  static bool rollout(int env, bool bwd, const RolloutArgs& a, int grid, cudaStream_t st) {
    return with_env(env, bwd, [&](auto e, auto b) {
      rollout_kernel<H, ACT, decltype(e)::value, decltype(b)::value><<<grid, NT, ROLLOUT_SMEM, st>>>(a);
    });
  }
  static void q_grad(const QGradArgs& a, int grid, cudaStream_t st) { q_grad_kernel<H, ACT><<<grid, NT, SMEM, st>>>(a); }
  static void eval(const EvalArgs& a, int grid, cudaStream_t st) { eval_kernel<H, ACT><<<grid, NT, SMEM, st>>>(a); }
  static void env_sample(const SampleArgs& a, int grid, cudaStream_t st) {
    env_sample_kernel<H, ACT><<<grid, NT, SMEM, st>>>(a);
  }
  static bool tc_rollout(int env, bool bwd, const tc::TcArgs& a, int grid, cudaStream_t st) {
    return with_env(env, bwd, [&](auto e, auto b) {
      tc::tc_rollout_kernel<decltype(e)::value, decltype(b)::value, ACT><<<grid, tc::ROLLOUT_THREADS, TC_SMEM, st>>>(a);
    });
  }

  static constexpr MlpKernels table() {
    MlpKernels t = {set_smem, rollout, q_grad, eval, env_sample, nullptr, tc::wait_dbg_attach};
    if constexpr (H == tc::H) t.tc_rollout = tc_rollout;
    return t;
  }
};

}  // namespace mpg
