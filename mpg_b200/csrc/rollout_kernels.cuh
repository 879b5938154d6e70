// Fused, persistent model-rollout kernels (fp32 FFMA path).
//   forward : mpg_learner.py:226-286 / nadp.py:87-171 rollout loop with per-step state checkpoints
//   backward: BPTT with recompute of the policy forward from the checkpoints (SURVEY.md 8(a) adjoint)
// One CTA owns a tile of TILE_R trajectories and walks the whole horizon; activations never leave
// shared memory; per-CTA parameter-gradient partials are combined later in a fixed order.
#pragma once
#include "env_models.cuh"
#include "mlp_tile.cuh"

namespace mpg {

struct FarStep { float wq, wlater; int first, q; };   // one step of the rollout list, see list_step

struct RolloutArgs {
  // learner config
  int obs_dim, act_dim, nfd, policy_out_tanh;
  float action_range;
  float obs_scale[MPG_MAX_OBS];
  float rew_scale, rew_shift, gamma;
  // rollout
  int rows, M, horizon, n_list;
  int list[MPG_MAX_LIST_LONG];
  float list_w[MPG_MAX_LIST_LONG];
  int full_bptt, has_q, use_start_actions, noise_mode;  // noise_mode: 0 none, 1 tensor, 2 philox
  const FarStep* far_steps;   // [horizon + 1 - STEP_TAB] the list at steps >= STEP_TAB (nullptr: the horizon stays below)
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
  long long partial_stride;   // floats, multiple of 4 (float4 accesses into the hidden -> hidden dW regions)
  NetDev pol, q;
};

// One step of the rollout list: the summed weight of the entries at step t (the upstream of Q(p_t, a_t)), the summed
// weight of the entries at steps > t (the weight of the reward of step t), the first entry at t (-1: t is not in the list)
// and whether some entry at t has a non-zero weight (step t has a Q part).  The sums run over the entries in list order.
__device__ __forceinline__ FarStep list_step(const int* list, const float* list_w, int n, int t) {
  FarStep r{0.f, 0.f, -1, 0};
  for (int k = 0; k < n; ++k) {
    const int l = list[k];
    const float w = list_w[k];
    if (l == t) {
      r.wq += w;
      if (r.first < 0) r.first = k;
      if (w != 0.f) r.q = 1;
    } else if (l > t) {
      r.wlater += w;
    }
  }
  return r;
}

// What the rollout list means at each step, built once per CTA so that no step scans the list (an indexed load of the list
// from the kernel parameters costs ~1.5 K cycles on the row threads).  Steps [0, STEP_TAB) are tables in 3.1 KB of shared
// memory (what the tensor-core kernel has left beside its 221 KB of images, DESIGN 4.2); a later step -- only horizons
// beyond STEP_TAB reach one -- reads its FarStep from a global table the host side builds before the launch
// (RolloutArgs::far_steps).  Either way a per-step question is one load.  Both kernels keep the tables behind their other
// shared memory (ROLLOUT_SMEM, SM_TAB), which stays where it was.
constexpr int STEP_TAB = 256;
struct StepTab {
  float wq_[STEP_TAB];
  float wlater_[STEP_TAB];
  int list[MPG_MAX_LIST_LONG];              // the list, staged for the build
  float w[MPG_MAX_LIST_LONG];
  const FarStep* far;                       // steps >= STEP_TAB
  signed char first_[STEP_TAB];
  signed char next[MPG_MAX_LIST_LONG];      // next entry at the step of entry k, -1: none
  unsigned char q_[STEP_TAB];

  __device__ __forceinline__ float wq(int t) const { return t < STEP_TAB ? wq_[t] : far[t - STEP_TAB].wq; }
  __device__ __forceinline__ float wlater(int t) const { return t < STEP_TAB ? wlater_[t] : far[t - STEP_TAB].wlater; }
  __device__ __forceinline__ int first(int t) const { return t < STEP_TAB ? first_[t] : far[t - STEP_TAB].first; }
  __device__ __forceinline__ bool q_part(int t) const { return t < STEP_TAB ? q_[t] != 0 : far[t - STEP_TAB].q != 0; }
};

// every thread of the CTA takes part (contains __syncthreads()); the caller synchronises the CTA before the first read.
// The list is staged in shared memory first: one parameter load per entry instead of one per entry and table step.
__device__ __forceinline__ void build_step_tab(StepTab& T, const int* list, const float* list_w, int n, const FarStep* far,
                                               int tid, int nthreads) {
  for (int k = tid; k < MPG_MAX_LIST_LONG; k += nthreads) {
    T.list[k] = k < n ? list[k] : -1;
    T.w[k] = k < n ? list_w[k] : 0.f;
  }
  if (tid == 0) T.far = far;
  __syncthreads();
  for (int i = tid; i < STEP_TAB + MPG_MAX_LIST_LONG; i += nthreads) {
    if (i < STEP_TAB) {
      const FarStep r = list_step(T.list, T.w, n, i);
      T.wq_[i] = r.wq; T.wlater_[i] = r.wlater; T.first_[i] = (signed char)r.first; T.q_[i] = (unsigned char)r.q;
    } else {
      const int k = i - STEP_TAB;
      int nx = -1;
      for (int j = n - 1; j > k; --j) if (T.list[j] == T.list[k]) nx = j;
      T.next[k] = (signed char)nx;
    }
  }
}

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
  StepTab& tab = *reinterpret_cast<StepTab*>(reinterpret_cast<float*>(smem_raw) + Smem<H>::FLOATS);   // behind the tiles
  using E = Env<ENV>;
  constexpr int S = E::S, A = E::A;
  const int tid = threadIdx.x;
  build_step_tab(tab, a.list, a.list_w, a.n_list, a.far_steps, tid, blockDim.x);
  __syncthreads();
  const int MB = a.rows * a.M;
  const int ntiles = (MB + TILE_R - 1) / TILE_R;
  const bool rowthread = tid < TILE_R;
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
      const int k0 = tab.first(t);
      if (k0 >= 0) {
        float qv = 0.f;
        if (a.has_q) {
          __syncthreads();
          mlp_forward_tile<H, ACT>(a.q, sm, 1);
          if (rowthread) qv = sm.y3[tid];
        }
        // every entry of step t gets its row, repeated entries included
        if (valid && a.returns_out)
          for (int k = k0; k >= 0; k = tab.next[k]) a.returns_out[(size_t)k * MB + grow] = rsum + gpow * qv;
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
        // Q part of step t: the summed weight of every entry at t; entries that all weigh zero are stats only
        if (tab.q_part(t) && a.has_q) {
          const float w_t = tab.wq(t);
          // Q input-gradient: upstream c w_t gamma^t on Q1(p_t, a_t)
          if (rowthread) {
#pragma unroll
            for (int j = 0; j < A; ++j) sm.xin[(a.obs_dim + j) * RP + tid] = act[j];
          }
          __syncthreads();
          mlp_forward_tile<H, ACT>(a.q, sm, 1);
          if (rowthread) sm.d3[tid] = valid ? cscale * w_t * gp : 0.f;
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
          mlp_forward_tile<H, ACT>(a.pol, sm, A);   // the Q pass reused bufA/bufB: recompute every layer of the policy
        }
        if (t < a.horizon && rowthread && valid) {
          const float rc = cscale * tab.wlater(t) * gp * a.rew_scale;
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
        mlp_backward_tile<H, ACT>(a.pol, sm, A, want_dw, want_gin, ga, partial);
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
    mlp_backward_tile<H, ACT>(a.q, sm, 1, true, false, ga, partial);
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

}  // namespace mpg
