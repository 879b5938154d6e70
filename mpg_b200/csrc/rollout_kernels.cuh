// Fused, persistent model-rollout kernels (fp32 FFMA path).
//   forward : mpg_learner.py:226-286 / nadp.py:87-171 rollout loop with per-step state checkpoints
//   backward: BPTT with recompute of the policy forward from the checkpoints (SURVEY.md 8(a) adjoint)
// One CTA owns a tile of TILE_R trajectories and walks the whole horizon; activations never leave
// shared memory; per-CTA parameter-gradient partials are combined later in a fixed order.
#pragma once
#include "env_models.cuh"
#include "mlp_tile.cuh"

namespace mpg {

struct RolloutArgs {
  // learner config
  int obs_dim, act_dim, nfd, policy_out_tanh;
  float action_range;
  float obs_scale[MPG_MAX_OBS];
  float rew_scale, rew_shift, gamma;
  // rollout
  int rows, M, horizon, n_list;
  int list[MPG_MAX_LIST];
  float list_w[MPG_MAX_LIST];
  int full_bptt, has_q, use_start_actions, noise_mode;  // noise_mode: 0 none, 1 tensor, 2 philox
  long long global_rows, row_offset;
  unsigned long long seed;
  // pointers
  const float* obs;
  const float* start_actions;
  const float* noise;
  float* returns_out;
  float* traj_obs;
  float* traj_rew;
  float* traj_act;
  float* ckpt;      // [horizon+1][M*rows][S]
  float* partial;   // [grid][partial_stride]
  long long partial_stride;   // floats, multiple of 4 (float4 accesses into the dW2 region)
  NetDev pol, q;
};

// policy head (policy.py:193-199): z -> m = out_act(z) -> a = action_range * tanh(m) | m
__device__ __forceinline__ float head_fwd(float z, int out_tanh, float range) {
  float m = out_tanh ? tanhf(z) : z;
  return range > 0.f ? range * tanhf(m) : m;
}
__device__ __forceinline__ float head_grad(float z, int out_tanh, float range) {
  float m = out_tanh ? tanhf(z) : z;
  float g = out_tanh ? 1.f - m * m : 1.f;
  if (range > 0.f) { float th = tanhf(m); g *= range * (1.f - th * th); }
  return g;
}

// action and d action / d z in one evaluation (same operations as head_fwd / head_grad)
__device__ __forceinline__ void head_fwd_grad(float z, int out_tanh, float range, float& act, float& g) {
  const float m = out_tanh ? tanhf(z) : z;
  g = out_tanh ? 1.f - m * m : 1.f;
  act = m;
  if (range > 0.f) { const float th = tanhf(m); g *= range * (1.f - th * th); act = range * th; }
}

template <int H, int ACT, int ENV, bool BWD>
__global__ void __launch_bounds__(NT, 1) rollout_kernel(const __grid_constant__ RolloutArgs a) {
  extern __shared__ float4 smem_raw[];
  Smem<H> sm(reinterpret_cast<float*>(smem_raw));
  using E = Env<ENV>;
  constexpr int S = E::S, A = E::A;
  const int tid = threadIdx.x;
  const int MB = a.rows * a.M;
  const int ntiles = (MB + TILE_R - 1) / TILE_R;
  const bool rowthread = tid < TILE_R;
  const GradLayout L(a.pol.in_dim, a.pol.out_dim, H);
  float* partial = a.partial + (size_t)blockIdx.x * a.partial_stride;
  GradAcc<H> ga;
  ga.zero();
  const float cscale = -1.f / ((float)a.M * (float)a.global_rows);

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int grow = tile * TILE_R + tid;          // local tiled row
    const bool valid = rowthread && grow < MB;
    const int m_idx = valid ? grow / a.rows : 0, i_idx = valid ? grow % a.rows : 0;
    const unsigned long long noise_row = (unsigned long long)m_idx * (unsigned long long)a.global_rows
                                         + (unsigned long long)(a.row_offset + i_idx);
    float s[S];
#pragma unroll
    for (int j = 0; j < S; ++j) s[j] = 0.f;
    if (valid) {
      float o[MPG_MAX_OBS];
      for (int i = 0; i < a.obs_dim; ++i) o[i] = a.obs[(size_t)i_idx * a.obs_dim + i];
      E::reset(o, s);
    }
    float rsum = 0.f, gpow = 1.f;
    // ------------------------------- forward -------------------------------
    for (int t = 0; t <= a.horizon; ++t) {
      float act[A];
      if (rowthread) {
        float o[MPG_MAX_OBS];
        if (valid) {
          E::get_obs(s, o, a.nfd);
          if (BWD) {
            float* c = a.ckpt + ((size_t)t * MB + grow) * S;
#pragma unroll
            for (int j = 0; j < S; ++j) c[j] = s[j];
          }
        }
        for (int i = 0; i < a.obs_dim; ++i) sm.xin[i * RP + tid] = valid ? o[i] * a.obs_scale[i] : 0.f;
      }
      const bool given = (t == 0 && a.use_start_actions);
      if (!given) {
        __syncthreads();
        mlp_forward_tile<H, ACT>(a.pol, sm, A);
      }
      if (rowthread) {
#pragma unroll
        for (int j = 0; j < A; ++j) {
          if (given) act[j] = valid ? a.start_actions[(size_t)i_idx * A + j] : 0.f;
          else act[j] = head_fwd(sm.y3[j * RP + tid], a.policy_out_tanh, a.action_range);
          sm.xin[(a.obs_dim + j) * RP + tid] = act[j];
          if (a.traj_act && valid) a.traj_act[((size_t)t * MB + grow) * A + j] = act[j];
        }
      }
      int kidx = -1;
      for (int k = 0; k < a.n_list; ++k) if (a.list[k] == t) kidx = k;
      if (kidx >= 0) {
        float qv = 0.f;
        if (a.has_q) {
          __syncthreads();
          mlp_forward_tile<H, ACT>(a.q, sm, 1);
          if (rowthread) qv = sm.y3[tid];
        }
        if (valid && a.returns_out) a.returns_out[(size_t)kidx * MB + grow] = rsum + gpow * qv;
      }
      if (t < a.horizon && rowthread && valid) {
        float eps = 0.f;
        if (E::HAS_NOISE) {
          if (a.noise_mode == 1) eps = a.noise[(size_t)t * MB + grow];
          else if (a.noise_mode == 2) eps = philox_normal(a.seed, noise_row, (uint32_t)t);
        }
        const float rew = E::step(s, act, eps, a.noise_mode != 0);
        const float prew = (rew + a.rew_shift) * a.rew_scale;   // preprocessor.py:147-159
        rsum += gpow * prew;
        gpow *= a.gamma;
        if (a.traj_rew) a.traj_rew[(size_t)t * MB + grow] = prew;
        if (a.traj_obs) {
          float o[MPG_MAX_OBS];
          E::get_obs(s, o, a.nfd);
          for (int i = 0; i < a.obs_dim; ++i) a.traj_obs[((size_t)t * MB + grow) * a.obs_dim + i] = o[i];
        }
      }
      __syncthreads();
    }
    // ------------------------------- backward -------------------------------
    if (BWD) {
      float lam[S], snext[S];
#pragma unroll
      for (int j = 0; j < S; ++j) { lam[j] = 0.f; snext[j] = s[j]; }
      for (int t = a.horizon; t >= 0; --t) {
        float gp = 1.f;
        for (int i = 0; i < t; ++i) gp *= a.gamma;
        if (rowthread) {
          float o[MPG_MAX_OBS];
          if (valid) {
            const float* c = a.ckpt + ((size_t)t * MB + grow) * S;
#pragma unroll
            for (int j = 0; j < S; ++j) s[j] = c[j];
            E::get_obs(s, o, a.nfd);
          }
          for (int i = 0; i < a.obs_dim; ++i) sm.xin[i * RP + tid] = valid ? o[i] * a.obs_scale[i] : 0.f;
        }
        __syncthreads();
        mlp_forward_tile<H, ACT>(a.pol, sm, A);
        float act[A], g_a[A], g_s[S], zpre[A];
#pragma unroll
        for (int j = 0; j < A; ++j) { act[j] = 0.f; g_a[j] = 0.f; zpre[j] = 0.f; }
#pragma unroll
        for (int j = 0; j < S; ++j) g_s[j] = 0.f;
        if (rowthread) {
#pragma unroll
          for (int j = 0; j < A; ++j) {
            zpre[j] = sm.y3[j * RP + tid];
            act[j] = head_fwd(zpre[j], a.policy_out_tanh, a.action_range);
          }
        }
        int kidx = -1;
        for (int k = 0; k < a.n_list; ++k) if (a.list[k] == t) kidx = k;
        if (kidx >= 0 && a.has_q && a.list_w[kidx] != 0.f) {   // zero-weight entries are stats only
          // Q input-gradient: upstream c w_k gamma^t on Q1(p_t, a_t)
          if (rowthread) {
#pragma unroll
            for (int j = 0; j < A; ++j) sm.xin[(a.obs_dim + j) * RP + tid] = act[j];
          }
          __syncthreads();
          mlp_forward_tile<H, ACT>(a.q, sm, 1);
          if (rowthread) sm.d3[tid] = valid ? cscale * a.list_w[kidx] * gp : 0.f;
          __syncthreads();
          mlp_backward_tile<H, ACT>(a.q, sm, 1, false, true, ga, nullptr);
          if (rowthread && valid) {
            float go[MPG_MAX_OBS];
            for (int i = 0; i < a.obs_dim; ++i) go[i] = sm.gx[i * RP + tid] * a.obs_scale[i];
            E::obs_grad_to_state(s, go, a.nfd, g_s);
#pragma unroll
            for (int j = 0; j < A; ++j) g_a[j] += sm.gx[(a.obs_dim + j) * RP + tid];
          }
          __syncthreads();
          mlp_forward_tile<H, ACT>(a.pol, sm, A);   // the Q pass reused bufA/bufB: recompute h1, h2 of the policy
        }
        if (t < a.horizon && rowthread && valid) {
          float Wt = 0.f;
          for (int k = 0; k < a.n_list; ++k) if (a.list[k] > t) Wt += a.list_w[k];
          const float rc = cscale * Wt * gp * a.rew_scale;
          env_step_bwd<ENV>(s, act, lam, rc, g_s, g_a, snext);
        }
        if (rowthread) {
#pragma unroll
          for (int j = 0; j < A; ++j)
            sm.d3[j * RP + tid] = valid ? g_a[j] * head_grad(zpre[j], a.policy_out_tanh, a.action_range) : 0.f;
        }
        __syncthreads();
        const bool want_dw = a.full_bptt || t == 0;
        const bool want_gin = t > 0;
        mlp_backward_tile<H, ACT>(a.pol, sm, A, want_dw, want_gin, ga, partial + L.oW2);
        if (rowthread && valid) {
#pragma unroll
          for (int j = 0; j < S; ++j) { lam[j] = g_s[j]; snext[j] = s[j]; }
          if (t > 0) {
            float go[MPG_MAX_OBS];
            for (int i = 0; i < a.obs_dim; ++i) go[i] = sm.gx[i * RP + tid] * a.obs_scale[i];
            E::obs_grad_to_state(s, go, a.nfd, lam);
          }
        }
        __syncthreads();
      }
    }
  }
  if (BWD) flush_grad_acc(a.pol, ga, partial);
}

// ---------------------------------------------------------------------------------------------
// Q-net regression gradient: q_forward_and_backward (mpg_learner.py:326-354, nadp.py:173-184)
// ---------------------------------------------------------------------------------------------
struct QGradArgs {
  int obs_dim, act_dim, rows;
  float obs_scale[MPG_MAX_OBS];
  float inv_global_rows;
  const float* obs;
  const float* act;
  const float* target;
  float* partial;       // [grid][partial_stride]
  long long partial_stride;
  float* loss_partial;  // [grid]
  NetDev q;
};

template <int H, int ACT>
__global__ void __launch_bounds__(NT, 1) q_grad_kernel(const __grid_constant__ QGradArgs a) {
  extern __shared__ float4 smem_raw[];
  Smem<H> sm(reinterpret_cast<float*>(smem_raw));
  __shared__ float red[TILE_R];
  const int tid = threadIdx.x;
  const int ntiles = (a.rows + TILE_R - 1) / TILE_R;
  const GradLayout L(a.q.in_dim, a.q.out_dim, H);
  float* partial = a.partial + (size_t)blockIdx.x * a.partial_stride;
  GradAcc<H> ga;
  ga.zero();
  float loss = 0.f;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row = tile * TILE_R + tid;
    const bool valid = tid < TILE_R && row < a.rows;
    if (tid < TILE_R) {
      for (int i = 0; i < a.obs_dim; ++i)
        sm.xin[i * RP + tid] = valid ? a.obs[(size_t)row * a.obs_dim + i] * a.obs_scale[i] : 0.f;
      for (int j = 0; j < a.act_dim; ++j)
        sm.xin[(a.obs_dim + j) * RP + tid] = valid ? a.act[(size_t)row * a.act_dim + j] : 0.f;
    }
    __syncthreads();
    mlp_forward_tile<H, ACT>(a.q, sm, 1);
    if (tid < TILE_R) {
      float diff = valid ? sm.y3[tid] - a.target[row] : 0.f;
      loss += 0.5f * diff * diff;
      sm.d3[tid] = diff * a.inv_global_rows;
    }
    __syncthreads();
    mlp_backward_tile<H, ACT>(a.q, sm, 1, true, false, ga, partial + L.oW2);
  }
  flush_grad_acc(a.q, ga, partial);
  if (tid < TILE_R) red[tid] = loss;
  __syncthreads();
  if (tid == 0) {
    float sum = 0.f;
    for (int i = 0; i < TILE_R; ++i) sum += red[i];
    a.loss_partial[blockIdx.x] = sum;
  }
}

// ---------------------------------------------------------------------------------------------
// forward-only evaluations on a replay batch
//   mode 0: act_out = pi_net0(sigma obs)                    (policy.py:193-212)
//   mode 1: out = Q_net0(sigma obs, act)                    (policy.py:219-241)
//   mode 2: out = rho(r+shift) + gamma min(Q_net1, Q_net2)(sigma o', pi_net0(sigma o'))  (mpg_learner.py:126-134);
//           single-Q when n_q == 1 (mpg_learner.py:147-152)
//   mode 3: out = rho(r+shift) + gamma Q_net1(sigma o', pi_net0(sigma o')) - Q_net2(sigma o, a)  (mpg_learner.py:136-144)
//   mode 4: out = rew[row] + gamma * Q_net1(sigma o, pi_net0(sigma o))   (n-step bootstrap, mpg_learner.py:153-169;
//           `rew` carries the partial return, `gamma` the coefficient gamma^T)
// ---------------------------------------------------------------------------------------------
struct EvalArgs {
  int mode, obs_dim, act_dim, rows, n_q, policy_out_tanh;
  float action_range, rew_scale, rew_shift, gamma;
  float obs_scale[MPG_MAX_OBS];
  const float* obs;      // obs (modes 0,1,3) / obs_tp1 (mode 2)
  const float* obs2;     // obs_tp1 (mode 3)
  const float* act;
  const float* rew;
  float* out;
  NetDev net0, net1, net2;
};

template <int H, int ACT>
__global__ void __launch_bounds__(NT, 1) eval_kernel(const __grid_constant__ EvalArgs a) {
  extern __shared__ float4 smem_raw[];
  Smem<H> sm(reinterpret_cast<float*>(smem_raw));
  const int tid = threadIdx.x;
  const int ntiles = (a.rows + TILE_R - 1) / TILE_R;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row = tile * TILE_R + tid;
    const bool rt = tid < TILE_R, valid = rt && row < a.rows;
    auto load_obs = [&](const float* src) {
      if (rt)
        for (int i = 0; i < a.obs_dim; ++i)
          sm.xin[i * RP + tid] = valid ? src[(size_t)row * a.obs_dim + i] * a.obs_scale[i] : 0.f;
    };
    auto load_act = [&]() {
      if (rt)
        for (int j = 0; j < a.act_dim; ++j)
          sm.xin[(a.obs_dim + j) * RP + tid] = valid ? a.act[(size_t)row * a.act_dim + j] : 0.f;
    };
    auto policy_to_xin = [&](const NetDev& net) {   // a = pi(xin obs rows) -> xin action rows
      __syncthreads();
      mlp_forward_tile<H, ACT>(net, sm, a.act_dim);
      if (rt)
        for (int j = 0; j < a.act_dim; ++j)
          sm.xin[(a.obs_dim + j) * RP + tid] = head_fwd(sm.y3[j * RP + tid], a.policy_out_tanh, a.action_range);
    };
    auto q_eval = [&](const NetDev& net) -> float {
      __syncthreads();
      mlp_forward_tile<H, ACT>(net, sm, 1);
      return rt ? sm.y3[tid] : 0.f;
    };
    if (a.mode == 0) {
      load_obs(a.obs);
      policy_to_xin(a.net0);
      if (valid)
        for (int j = 0; j < a.act_dim; ++j) a.out[(size_t)row * a.act_dim + j] = sm.xin[(a.obs_dim + j) * RP + tid];
    } else if (a.mode == 1) {
      load_obs(a.obs);
      load_act();
      float q = q_eval(a.net0);
      if (valid) a.out[row] = q;
    } else if (a.mode == 2) {
      load_obs(a.obs);
      policy_to_xin(a.net0);
      float q = q_eval(a.net1);
      if (a.n_q == 2) q = fminf(q, q_eval(a.net2));
      if (valid) a.out[row] = (a.rew[row] + a.rew_shift) * a.rew_scale + a.gamma * q;
    } else if (a.mode == 4) {
      load_obs(a.obs);
      policy_to_xin(a.net0);
      float q = q_eval(a.net1);
      if (valid) a.out[row] = a.rew[row] + a.gamma * q;
    } else {
      load_obs(a.obs2);
      policy_to_xin(a.net0);
      float q1 = q_eval(a.net1);
      __syncthreads();
      load_obs(a.obs);
      load_act();
      float q0 = q_eval(a.net2);
      if (valid) a.out[row] = (a.rew[row] + a.rew_shift) * a.rew_scale + a.gamma * q1 - q0;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// Fused exploration sampler (OffPolicyWorker.sample, worker.py:91-119, with the real PathTracking environment):
// `steps` iterations of  a = pi(sigma obs) + explore_sigma eps ; (obs', r, done) = env.step(a) ; record the
// transition ; re-draw the agents that are done  -- in ONE launch, one 64-agent tile per CTA, the environment state
// in the registers of the thread that owns the agent.  eps and the reset observations are drawn by the caller, so
// the step-by-step path (mpg_policy_forward + mpg_env_step per step) gives the same numbers.
// ---------------------------------------------------------------------------------------------
struct SampleArgs {
  int agents, steps, obs_dim, act_dim, nfd, policy_out_tanh;
  float action_range, sigma;
  float obs_scale[MPG_MAX_OBS];
  const float* explore_noise;   // (steps, agents, act_dim) standard normal, or nullptr
  const float* reset_obs;       // (steps, agents, obs_dim): observation an agent restarts from when done at that step;
                                // nullptr: never restart (fixed-step evaluation episodes, evaluator.py run_an_episode)
  float* state;                 // (agents, 8)        in/out
  float* obs;                   // (agents, obs_dim)  in/out
  float *out_obs, *out_act, *out_rew, *out_obs_tp1, *out_done;   // (steps, agents, ...)
  NetDev net;
};

template <int H, int ACT>
__global__ void __launch_bounds__(NT, 1) env_sample_kernel(const __grid_constant__ SampleArgs a) {
  using E = Env<MPG_ENV_PT_REAL>;
  extern __shared__ float4 smem_raw[];
  Smem<H> sm(reinterpret_cast<float*>(smem_raw));
  const int tid = threadIdx.x, row = blockIdx.x * TILE_R + tid;
  const bool rt = tid < TILE_R, valid = rt && row < a.agents;
  float s[E::S], o[MPG_MAX_OBS];
#pragma unroll
  for (int j = 0; j < E::S; ++j) s[j] = valid ? a.state[(size_t)row * E::S + j] : 0.f;
  for (int i = 0; i < a.obs_dim; ++i) o[i] = valid ? a.obs[(size_t)row * a.obs_dim + i] : 0.f;
  for (int t = 0; t < a.steps; ++t) {
    if (rt)
      for (int i = 0; i < a.obs_dim; ++i) sm.xin[i * RP + tid] = o[i] * a.obs_scale[i];
    __syncthreads();
    mlp_forward_tile<H, ACT>(a.net, sm, a.act_dim);
    if (valid) {
      const size_t tr = (size_t)t * a.agents + row;
      float act[E::A], o1[MPG_MAX_OBS];
#pragma unroll
      for (int j = 0; j < E::A; ++j) {
        act[j] = head_fwd(sm.y3[j * RP + tid], a.policy_out_tanh, a.action_range);
        if (a.explore_noise) act[j] += a.sigma * a.explore_noise[tr * E::A + j];
        a.out_act[tr * E::A + j] = act[j];
      }
      for (int i = 0; i < a.obs_dim; ++i) a.out_obs[tr * a.obs_dim + i] = o[i];
      int done = 0;
      const float rew = E::step_done(s, act, &done);
      E::get_obs(s, o1, a.nfd);
      a.out_rew[tr] = rew;
      a.out_done[tr] = (float)done;
      for (int i = 0; i < a.obs_dim; ++i) a.out_obs_tp1[tr * a.obs_dim + i] = o1[i];
      if (done && a.reset_obs) {                    // env.reset(): only the finished agents restart
        for (int i = 0; i < a.obs_dim; ++i) o[i] = a.reset_obs[tr * a.obs_dim + i];
        E::reset(o, s);
      } else {
        for (int i = 0; i < a.obs_dim; ++i) o[i] = o1[i];
      }
    }
    __syncthreads();
  }
  if (valid) {
#pragma unroll
    for (int j = 0; j < E::S; ++j) a.state[(size_t)row * E::S + j] = s[j];
    for (int i = 0; i < a.obs_dim; ++i) a.obs[(size_t)row * a.obs_dim + i] = o[i];
  }
}

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

#ifndef MPG_ACT_UNIT   // non-template kernels are defined in api.cu's unit only (act_instances.cuh)
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
#endif

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
