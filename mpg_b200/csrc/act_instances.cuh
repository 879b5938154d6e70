// Explicit instantiations of the kernels that depend on the hidden activation ACT (MPG_ACT_*): the FFMA tile kernels at
// every width and the tensor-core rollout kernel.  api.cu instantiates the ELU set itself and declares the relu and tanh
// sets extern; act_relu.cu and act_tanh.cu define them, so that the three sets compile in parallel translation units.
// Those units define MPG_ACT_UNIT, which leaves out the kernels that do not depend on the activation (api.cu owns them)
// and gives the unit its own copy of the mbarrier-watchdog pointer (attached by wait_dbg_attach_*).
#pragma once
#include "rollout_kernels.cuh"
#include "tc_kernels.cuh"

#define MPG_FFMA_INSTANCES(EXT, H, ACT)                                                                                  \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_PATH_TRACKING, true>(const __grid_constant__ RolloutArgs);  \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_PATH_TRACKING, false>(const __grid_constant__ RolloutArgs); \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_INVERTED_PENDULUM, true>(const __grid_constant__ RolloutArgs); \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_INVERTED_PENDULUM, false>(const __grid_constant__ RolloutArgs); \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_INVERTED_DOUBLE_PENDULUM, true>(                             \
      const __grid_constant__ RolloutArgs);                                                                              \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_INVERTED_DOUBLE_PENDULUM, false>(                            \
      const __grid_constant__ RolloutArgs);                                                                              \
  EXT template __global__ void rollout_kernel<H, ACT, MPG_ENV_PATH_TRACKING_REAL, false>(const __grid_constant__ RolloutArgs); \
  EXT template __global__ void q_grad_kernel<H, ACT>(const __grid_constant__ QGradArgs);                                 \
  EXT template __global__ void eval_kernel<H, ACT>(const __grid_constant__ EvalArgs);                                    \
  EXT template __global__ void env_sample_kernel<H, ACT>(const __grid_constant__ SampleArgs);

#define MPG_ACT_INSTANCES(EXT, ACT)                                                                                      \
  MPG_FFMA_INSTANCES(EXT, 64, ACT)                                                                                       \
  MPG_FFMA_INSTANCES(EXT, 128, ACT)                                                                                      \
  MPG_FFMA_INSTANCES(EXT, 256, ACT)                                                                                      \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING, true, ACT>(const __grid_constant__ tc::TcArgs); \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING, false, ACT>(const __grid_constant__ tc::TcArgs); \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_INVERTED_PENDULUM, true, ACT>(                               \
      const __grid_constant__ tc::TcArgs);                                                                               \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_INVERTED_PENDULUM, false, ACT>(                              \
      const __grid_constant__ tc::TcArgs);                                                                               \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_INVERTED_DOUBLE_PENDULUM, true, ACT>(                        \
      const __grid_constant__ tc::TcArgs);                                                                               \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_INVERTED_DOUBLE_PENDULUM, false, ACT>(                       \
      const __grid_constant__ tc::TcArgs);                                                                               \
  EXT template __global__ void tc::tc_rollout_kernel<MPG_ENV_PATH_TRACKING_REAL, false, ACT>(                             \
      const __grid_constant__ tc::TcArgs);

namespace mpg {
// point the watchdog record of the relu / tanh units' kernels at the handle's mapped host memory (see tc_common.cuh)
bool wait_dbg_attach_relu(unsigned long long* dev_ptr);
bool wait_dbg_attach_tanh(unsigned long long* dev_ptr);
}  // namespace mpg
