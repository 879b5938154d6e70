// Environment-only kernels, one thread per row: single model steps and the real PathTracking environment step.  They do
// not depend on the hidden activation, so only api.cu compiles them.
#pragma once
#include "env_models.cuh"

namespace mpg {

// ---------------------------------------------------------------------------------------------
// single model step (backs <Env>Model.rollout_out / reset / compute_rewards and their autograd)
// ---------------------------------------------------------------------------------------------
template <int ENV>
__global__ void model_reset_kernel(int rows, int obs_dim, const float* __restrict__ obs, float* __restrict__ state) {
  using E = Env<ENV>;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float o[MPG_MAX_OBS], s[E::S];
  for (int i = 0; i < obs_dim; ++i) o[i] = obs[(size_t)r * obs_dim + i];
  E::reset(o, s);
#pragma unroll
  for (int j = 0; j < E::S; ++j) state[(size_t)r * E::S + j] = s[j];
}

template <int ENV>
__global__ void model_step_kernel(int rows, int obs_dim, int nfd, const float* __restrict__ state_in,
                                  const float* __restrict__ action, const float* __restrict__ eps,
                                  float* __restrict__ state_out, float* __restrict__ obs_out, float* __restrict__ rew_out) {
  using E = Env<ENV>;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float s[E::S], act[E::A], o[MPG_MAX_OBS];
#pragma unroll
  for (int j = 0; j < E::S; ++j) s[j] = state_in[(size_t)r * E::S + j];
#pragma unroll
  for (int j = 0; j < E::A; ++j) act[j] = action[(size_t)r * E::A + j];
  const float rew = E::step(s, act, eps ? eps[r] : 0.f, eps != nullptr);
#pragma unroll
  for (int j = 0; j < E::S; ++j) state_out[(size_t)r * E::S + j] = s[j];
  E::get_obs(s, o, nfd);
  if (obs_out) for (int i = 0; i < obs_dim; ++i) obs_out[(size_t)r * obs_dim + i] = o[i];
  if (rew_out) rew_out[r] = rew;
}

// real PathTracking environment step with the done flag
__global__ void env_step_kernel(int rows, int obs_dim, int nfd, const float* __restrict__ state_in,
                                const float* __restrict__ action, float* __restrict__ state_out,
                                float* __restrict__ obs_out, float* __restrict__ rew_out, int* __restrict__ done_out) {
  using E = Env<MPG_ENV_PT_REAL>;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float s[E::S], act[E::A], o[MPG_MAX_OBS];
#pragma unroll
  for (int j = 0; j < E::S; ++j) s[j] = state_in[(size_t)r * E::S + j];
  act[0] = action[(size_t)r * 2]; act[1] = action[(size_t)r * 2 + 1];
  int done = 0;
  const float rew = E::step_done(s, act, &done);
#pragma unroll
  for (int j = 0; j < E::S; ++j) state_out[(size_t)r * E::S + j] = s[j];
  E::get_obs(s, o, nfd);
  if (obs_out) for (int i = 0; i < obs_dim; ++i) obs_out[(size_t)r * obs_dim + i] = o[i];
  if (rew_out) rew_out[r] = rew;
  if (done_out) done_out[r] = done;
}

// g_state_in = J_s^T (E^T g_obs_out + g_state_out) + g_rew dr/ds ; g_action likewise
template <int ENV>
__global__ void model_step_bwd_kernel(int rows, int obs_dim, int nfd, const float* __restrict__ state_in,
                                      const float* __restrict__ action, const float* __restrict__ eps,
                                      const float* __restrict__ g_obs_out,
                                      const float* __restrict__ g_rew_out, const float* __restrict__ g_state_out,
                                      float* __restrict__ g_state_in, float* __restrict__ g_action) {
  using E = Env<ENV>;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float s[E::S], s1[E::S], act[E::A], lam[E::S], gs[E::S], ga[E::A];
#pragma unroll
  for (int j = 0; j < E::S; ++j) { s[j] = state_in[(size_t)r * E::S + j]; s1[j] = s[j]; gs[j] = 0.f; }
#pragma unroll
  for (int j = 0; j < E::A; ++j) { act[j] = action[(size_t)r * E::A + j]; ga[j] = 0.f; }
  // recompute the post-step state (the pendulum rewards and the obs map are taken there)
  E::step(s1, act, eps ? eps[r] : 0.f, eps != nullptr);
#pragma unroll
  for (int j = 0; j < E::S; ++j) lam[j] = g_state_out ? g_state_out[(size_t)r * E::S + j] : 0.f;
  if (g_obs_out) {
    float go[MPG_MAX_OBS];
    for (int i = 0; i < obs_dim; ++i) go[i] = g_obs_out[(size_t)r * obs_dim + i];
    E::obs_grad_to_state(s1, go, nfd, lam);
  }
  env_step_bwd<ENV>(s, act, lam, g_rew_out ? g_rew_out[r] : 0.f, gs, ga, s1);
#pragma unroll
  for (int j = 0; j < E::S; ++j) g_state_in[(size_t)r * E::S + j] = gs[j];
#pragma unroll
  for (int j = 0; j < E::A; ++j) g_action[(size_t)r * E::A + j] = ga[j];
}

template <int ENV>
__global__ void rewards_kernel(int rows, const float* __restrict__ state, const float* __restrict__ scaled_action,
                               float* __restrict__ rew) {
  using E = Env<ENV>;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float s[E::S];
#pragma unroll
  for (int j = 0; j < E::S; ++j) s[j] = state[(size_t)r * E::S + j];
  if constexpr (ENV == MPG_ENV_PATH_TRACKING || ENV == MPG_ENV_PT_REAL)
    rew[r] = Env<MPG_ENV_PATH_TRACKING>::reward_pre(s, scaled_action[(size_t)r * 2], scaled_action[(size_t)r * 2 + 1]);
  else
    rew[r] = E::reward_post(s);
}

}  // namespace mpg
