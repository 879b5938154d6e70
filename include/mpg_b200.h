/*
 * mpg_b200 -- C ABI of the B200-native MPG model-based learner hot path.
 *
 * The reference (idthanm/mpg) has NO FFI: its two plugin boundaries are duck-typed Python classes
 * (learners/*.py selected at train_scripts/train_script.py:40-46; env models selected at
 * envs_and_models/__init__.py:13-15).  This header is the boundary a maintainer would bind with
 * ctypes from those classes (see INTEGRATION.md); every entry point names the reference code it
 * replaces.  Plain C: opaque handle, POD structs, raw device pointers, explicit sizes, a
 * caller-supplied cudaStream_t (passed as void*).  No torch types, no C++ exceptions.
 *
 * Conventions
 *   - all tensors fp32, row-major, DEVICE pointers unless the name ends in _host;
 *   - network weights use the Keras layout of the reference: kernels (in, out), list order
 *     [W1, b1, W2, b2, W3, b3] (model.py:20-43); gradients are written in the same order into one
 *     flat buffer (W1|b1|W2|b2|W3|b3);
 *   - every function returns 0 on success, <0 on error; mpg_last_error() gives the message;
 *   - nothing is freed or retained from caller memory; workspace belongs to the handle;
 *   - all work is enqueued on `stream`; no hidden synchronisation.
 */
#ifndef MPG_B200_H
#define MPG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mpg_ctx mpg_ctx;

/* env_id registry: envs_and_models/__init__.py:13-15 */
enum {
  MPG_ENV_PATH_TRACKING = 0,            /* 'PathTracking-v0'            path_tracking_env.py:245-297 */
  MPG_ENV_INVERTED_PENDULUM = 1,        /* 'InvertedPendulumConti-v0'   inverted_pendulum_model.py:77-97 */
  MPG_ENV_INVERTED_DOUBLE_PENDULUM = 2, /* 'InvertedDoublePendulum-v2'  inverted_double_pendulum_model.py:103-144 */
  /* the REAL PathTracking environment (PathTrackingEnv, path_tracking_env.py:356-487: 200 Hz x 20 sub-steps, reference
   * path projection). Forward only: as mpg_config.env it backs mpg_model_reset / mpg_env_step (state_dim 8); inside a
   * PathTracking handle it is selected per call with mpg_rollout_params.real_env (MPG-v1 n-step targets). */
  MPG_ENV_PATH_TRACKING_REAL = 3
};

/* network slots: PolicyWithQs.models + target_models (policy.py:72-89) */
enum {
  MPG_NET_Q1 = 0, MPG_NET_Q2 = 1, MPG_NET_POLICY = 2,
  MPG_NET_Q1_TARGET = 3, MPG_NET_Q2_TARGET = 4, MPG_NET_POLICY_TARGET = 5,
  MPG_NUM_NETS = 6
};

enum { MPG_OK = 0, MPG_ERR_ARG = -1, MPG_ERR_CUDA = -2, MPG_ERR_UNSUPPORTED = -3, MPG_ERR_STATE = -4 };

#define MPG_MAX_OBS 16
#define MPG_MAX_LIST 8

/* What the learner constructors read from `args` (mpg_learner.py:30-58, nadp.py:29-47) that the
 * device path needs. */
typedef struct {
  int32_t env;               /* MPG_ENV_* */
  int32_t num_future_data;   /* PathTracking only (path_tracking_env.py:265-271) */
  int32_t obs_dim;           /* 6+nfd | 4 | 11 */
  int32_t act_dim;           /* 2 | 1 | 1 */
  int32_t hidden;            /* *_num_hidden_units of every net of the handle: 64, 128 or 256 (2 hidden layers) */
  int32_t policy_out_tanh;   /* policy_out_activation == 'tanh' */
  float action_range;        /* policy.py:197; <= 0 means None */
  float obs_scale[MPG_MAX_OBS]; /* preprocessor.py:134-145, 'scale' mode */
  float rew_scale;           /* preprocessor.py:147-159 */
  float rew_shift;
  float gamma;
  int32_t max_rows;          /* capacity: M * rows per call on this device */
  int32_t max_horizon;       /* capacity: max rollout length n */
} mpg_config;

/* One model rollout (mpg_learner.py:226-286, nadp.py:87-171). */
typedef struct {
  int32_t rows;              /* B on this device (before M-tiling) */
  int32_t M;                 /* args.M: tf.tile factor */
  int32_t horizon;           /* n = max(rollout list) */
  int32_t n_list;            /* len(num_rollout_list_*) <= MPG_MAX_LIST */
  int32_t list[MPG_MAX_LIST];   /* rollout indices k (each <= horizon) */
  float list_w[MPG_MAX_LIST];   /* loss weights w_k (rule_based_weights; 1 for NADP) */
  int32_t full_bptt;         /* 1: dW at every step (NADP, deriv_interval_policy); 0: a_0 only (default MPG) */
  int32_t q_net;             /* bootstrap net: MPG_NET_Q1 / MPG_NET_Q1_TARGET, or -1 for none (AMPC) */
  int32_t policy_net;        /* MPG_NET_POLICY (a_t = pi(p_t)) */
  int64_t global_rows;       /* B summed over all ranks (loss scale 1/(M*global_rows)); 0 -> rows */
  int64_t row_offset;        /* first global row of this shard (keys the noise stream) */
  uint64_t noise_seed;       /* Philox key when `noise` is NULL */
  int32_t use_philox;        /* 1: in-kernel Philox4x32-10 N(0,1); 0: read `noise` (NULL noise + 0 => no noise) */
  int32_t real_env;          /* 1: roll the REAL PathTracking env instead of the model (forward-only calls, PathTracking handles) */
} mpg_rollout_params;

/* ---- lifetime ---------------------------------------------------------------------------- */
int mpg_create(const mpg_config* cfg, mpg_ctx** out);
void mpg_destroy(mpg_ctx* ctx);
const char* mpg_last_error(const mpg_ctx* ctx);   /* ctx may be NULL: last create() error */
size_t mpg_workspace_bytes(const mpg_ctx* ctx);
int mpg_num_sms(const mpg_ctx* ctx);
int mpg_param_count(const mpg_ctx* ctx, int net); /* floats in one net's flat gradient */

/* ---- weights: PolicyWithQs.set_weights (policy.py:116-121) -------------------------------- */
/* w[0..5] = W1,b1,W2,b2,W3,b3 device pointers in Keras layout; repacked into the kernel layouts. */
int mpg_set_weights(mpg_ctx* ctx, int net, const float* const w[6], void* stream);
/* copy back in Keras layout (PolicyWithQs.get_weights, policy.py:112-114) */
int mpg_get_weights(mpg_ctx* ctx, int net, float* const w[6], void* stream);

/* ---- policy gradient through the model rollout ------------------------------------------- */
/* MPGLearner.policy_forward_and_backward (mpg_learner.py:356-365) /
 * NADPLearner.policy_forward_and_backward (nadp.py:186-194): forward rollout with per-step state
 * checkpoints, fused BPTT backward with recompute.
 *   obs        (rows, obs_dim)
 *   noise      (horizon, M*rows) standard-normal eps, or NULL (see use_philox)
 *   grad_out   (param_count(policy)) UNCLIPPED d loss / d theta, loss = sum_k w_k * (-mean R_k),
 *              scaled by 1/(M*global_rows) so that per-rank results add up under all-reduce
 *   returns_out (n_list, M*rows) per-row R_k = sum_{t<k} gamma^t rho r_t + gamma^k Q(p_k, a_k)
 */
int mpg_policy_grad(mpg_ctx* ctx, const mpg_rollout_params* p, const float* obs, const float* noise,
                    float* grad_out, float* returns_out, void* stream);

/* Forward-only rollout: NADPLearner.model_rollout_for_q_estimation (nadp.py:87-126) when
 * start_actions != NULL, and the trajectory view used by the parity tests.
 *   start_actions (rows, act_dim) or NULL (a_0 = pi(p_0))
 *   returns_out (n_list, M*rows)
 *   traj_obs (horizon, M*rows, obs_dim) raw obs_{t+1};  traj_rew (horizon, M*rows) processed
 *   rewards;  traj_act (horizon+1, M*rows, act_dim) actions; each may be NULL */
int mpg_rollout_forward(mpg_ctx* ctx, const mpg_rollout_params* p, const float* obs, const float* start_actions,
                        const float* noise, float* returns_out, float* traj_obs, float* traj_rew, float* traj_act,
                        void* stream);

/* mean over the M tiles, then sum / sum of squares over rows (mpg_learner.py:272-274):
 * out[0..n_list) = sum_i mean_m R_k ; out[n_list..2 n_list) = sum_i (mean_m R_k)^2 */
int mpg_returns_stats(mpg_ctx* ctx, const float* returns, int n_list, int rows, int M, float* out, void* stream);
/* tile mean only: out (n_list, rows) -- the stop_gradient targets of nadp.py:120-126 */
int mpg_returns_tile_mean(mpg_ctx* ctx, const float* returns, int n_list, int rows, int M, float* out, void* stream);

/* ---- Q side ------------------------------------------------------------------------------- */
/* q_forward_and_backward (mpg_learner.py:326-354, nadp.py:173-184): loss = 0.5 mean (Q(sigma o, a) - target)^2.
 *   grad_out (param_count(net)) scaled by 1/global_rows; loss_sum_out[0] = sum_i 0.5 (Q - target)^2 */
int mpg_q_grad(mpg_ctx* ctx, int net, int rows, int64_t global_rows, const float* obs, const float* act,
               const float* target, float* grad_out, float* loss_sum_out, void* stream);
/* compute_action / compute_target_action (policy.py:193-212) on RAW obs (scale applied inside) */
int mpg_policy_forward(mpg_ctx* ctx, int net, int rows, const float* obs, float* act_out, void* stream);
/* compute_Q1/Q2/Q1_target/Q2_target (policy.py:219-241) on RAW obs */
int mpg_q_forward(mpg_ctx* ctx, int net, int rows, const float* obs, const float* act, float* q_out, void* stream);
/* compute_clipped_double_q_target (mpg_learner.py:126-134) when double_q, else the 1-step target of
 * compute_n_step_target (mpg_learner.py:147-152): rho (r + shift) + gamma min(Q1t, Q2t)(o', pi_t(o')) */
int mpg_q_target(mpg_ctx* ctx, int double_q, int rows, const float* rew, const float* obs_tp1, float* target_out,
                 void* stream);
/* compute_td_error (mpg_learner.py:136-144, nadp.py:67-76) */
int mpg_td_error(mpg_ctx* ctx, int rows, const float* obs, const float* act, const float* rew, const float* obs_tp1,
                 float* td_out, void* stream);

/* Bootstrap on top of a partial return (compute_n_step_target, mpg_learner.py:153-169):
 * out = base + coef * Q1_target(sigma o, pi_target(sigma o)); base (rows) e.g. sum_t gamma^t rho r_t, coef = gamma^T */
int mpg_q_bootstrap(mpg_ctx* ctx, int rows, const float* base, float coef, const float* obs, float* out, void* stream);

/* One step of the REAL environment (handles created with env = MPG_ENV_PATH_TRACKING_REAL):
 * PathTrackingEnv.step (path_tracking_env.py:456-472). done_out (int32, may be NULL) = judge_done (:474-487). */
int mpg_env_step(mpg_ctx* ctx, int rows, const float* state_in, const float* action, float* state_out, float* obs_out,
                 float* rew_out, int32_t* done_out, void* stream);

/* ---- single model step: <Env>Model.rollout_out ------------------------------------------- */
/* state (rows, state_dim) in/out; obs_out (rows, obs_dim); rew_out (rows) RAW reward.
 * eps (rows) standard normal or NULL. */
int mpg_model_reset(mpg_ctx* ctx, int rows, const float* obs, float* state_out, void* stream);
int mpg_model_step(mpg_ctx* ctx, int rows, const float* state_in, const float* action, const float* eps,
                   float* state_out, float* obs_out, float* rew_out, void* stream);
/* adjoint of mpg_model_step: given d/d obs_out and d/d rew_out, accumulate d/d state_in, d/d action */
int mpg_model_step_bwd(mpg_ctx* ctx, int rows, const float* state_in, const float* action, const float* eps,
                       const float* g_obs_out, const float* g_rew_out, const float* g_state_out, float* g_state_in,
                       float* g_action, void* stream);
/* Fused exploration sampler: OffPolicyWorker.sample (worker.py:91-119) with the real PathTracking environment
 * (path_tracking_env.py:356-487) in one launch.  Called on the PathTracking POLICY handle (env MPG_ENV_PATH_TRACKING).
 * For t < steps:  a = pi(obs_scale * obs) + explore_sigma * explore_noise[t] ;  (obs', r, done) = env.step(a) ;
 * transition t is written to out_* (row t * agents + agent) ;  agents that are done restart from reset_obs[t]
 * (env.reset() without init_obs re-draws only the finished agents, path_tracking_env.py:422-454).
 *   explore_noise (steps, agents, act_dim) standard normal or NULL;  reset_obs (steps, agents, obs_dim), or NULL:
 *   nobody restarts (the evaluator's fixed-step episodes, evaluator.py run_an_episode with fixed_steps);
 *   state (agents, 8) and obs (agents, obs_dim) are the environment's tensors, updated in place. */
int mpg_env_sample(mpg_ctx* ctx, int policy_net, int agents, int steps, float explore_sigma, const float* explore_noise,
                   const float* reset_obs, float* state, float* obs, float* out_obs, float* out_act, float* out_rew,
                   float* out_obs_tp1, float* out_done, void* stream);

/* VehicleDynamics.compute_rewards(states, scaled actions) / Dynamics.compute_rewards(states) */
int mpg_compute_rewards(mpg_ctx* ctx, int rows, const float* state, const float* scaled_action, float* rew_out,
                        void* stream);
int mpg_state_dim(const mpg_ctx* ctx);

/* ---- optimiser step on device-resident weights (SURVEY.md 8(f) next #2) --------------------- */
/* One Keras-Adam step on the flat weights of `net` (PolicyWithQs.apply_gradients, policy.py:123-156; keras
 * OptimizerV2 Adam: m = b1 m + (1-b1) g, v = b2 v + (1-b2) g^2, w -= lr sqrt(1-b2^t)/(1-b1^t) m / (sqrt(v) + eps)).
 *   grad: flat gradient in Keras order (device);  lr: already-decayed learning rate (PolynomialDecay is evaluated
 *   by the caller);  step: t = optimizer.iterations + 1.  Kernel-layout copies of the weights are re-packed. */
int mpg_adam_step(mpg_ctx* ctx, int net, const float* grad, float lr, int64_t step, float beta1, float beta2, float eps,
                  void* stream);
/* Adam moments of `net` (flat, Keras order, device pointers) -- what tf.train.Checkpoint stores for the optimizers in
 * PolicyWithQs.save_weights / load_weights (policy.py:98-110).  Moments of a never-stepped net read as zeros. */
int mpg_get_adam_state(mpg_ctx* ctx, int net, float* m, float* v, void* stream);
int mpg_set_adam_state(mpg_ctx* ctx, int net, const float* m, const float* v, void* stream);
/* Polyak target update (policy.py:158-171): dst = tau * src + (1 - tau) * dst, then re-pack dst */
int mpg_polyak_update(mpg_ctx* ctx, int src_net, int dst_net, float tau, void* stream);

/* ---- tf.clip_by_global_norm (mpg_learner.py:415-431, nadp.py:220-225) --------------------- */
/* in place over one net's flat gradient; norm_out[0] = pre-clip global norm */
int mpg_clip_global_norm(mpg_ctx* ctx, float* grad, int n, float clip, float* norm_out, void* stream);

/* standard-normal noise of the in-kernel Philox stream, for tests: out (horizon, M*rows) */
int mpg_philox_noise(mpg_ctx* ctx, const mpg_rollout_params* p, float* out, void* stream);

/* Kernel family used by mpg_policy_grad / mpg_rollout_forward:
 *   MPG_BACKEND_FFMA  fp32 CUDA-core contractions (every env / shape this build supports)
 *   MPG_BACKEND_TC    tcgen05 tensor-core contractions with split-bf16 operands (fp32-accurate), hidden = 256 only;
 *                     returns MPG_ERR_UNSUPPORTED for configurations it does not cover
 * mpg_create selects MPG_BACKEND_TC whenever it covers the configuration (hidden = 256 and
 * obs_dim + act_dim + 1 <= 16), else
 * MPG_BACKEND_FFMA; the environment variable MPG_B200_BACKEND=ffma forces the fp32 path at creation. */
enum { MPG_BACKEND_FFMA = 0, MPG_BACKEND_TC = 1 };
int mpg_set_backend(mpg_ctx* ctx, int backend);
int mpg_get_backend(const mpg_ctx* ctx);

/* Hidden activation of every net of the handle (value_hidden_activation == policy_hidden_activation, model.py
 * Dense(activation=...)): applies to every call that evaluates an MLP, on both backends and at every width.
 * A new handle uses MPG_ACT_ELU; an unknown value returns MPG_ERR_ARG.  The weight images do not depend on it, so the
 * activation may change between calls on one handle. */
enum { MPG_ACT_ELU = 0, MPG_ACT_RELU = 1, MPG_ACT_TANH = 2 };
int mpg_set_activation(mpg_ctx* ctx, int act);
int mpg_get_activation(const mpg_ctx* ctx);

/* Optional device timing of the dominant (rollout) kernel: when enabled, CUDA events are recorded on
 * the caller's stream immediately around that launch; mpg_kernel_ms() waits for the last pair and
 * returns its duration in milliseconds (<0: nothing recorded). Used by bench.py for the roofline. */
int mpg_set_timing(mpg_ctx* ctx, int enabled);
float mpg_kernel_ms(mpg_ctx* ctx);

#ifdef MPG_DEBUG_PROBES   /* development probes: exported by libmpg_b200_dbg.so only, never by the product library */
/* Self test of the tcgen05 GEMM building blocks (tests only). kind 0: Z[128x256] = X[128x256].W[256x256]^T;
 * kind 1: Z[128x256] = X[128x16].W[16x256]; kind 2: Z[128x16] = X[128x256].W[16x256]^T. fp32 device pointers.
 * kinds 3 / 4 are timing probes (tools/gemm_probe.py): the big GEMM `repeats` times back to back with streamed /
 * resident weights on MPG_SELFTEST_GRID CTAs; Z is not written. */
int mpg_tc_selftest(mpg_ctx* ctx, int kind, const float* X, const float* W, float* Z, int repeats, void* stream);

/* Debug timeline of the tensor-core rollout kernel: when `buf` (128 int64, device) is non-NULL the next
 * mpg_policy_grad calls record clock64() stamps of one backward step of CTA 0 (see DESIGN.md 4.2). */
int mpg_set_profile_buffer(mpg_ctx* ctx, long long* buf);
#endif
/* Watchdog record of the kernels' mbarrier waits: a wait that does not complete within ~2 s traps (the launch fails
 * with a CUDA error instead of hanging the device) after storing its place. out[0] != 0: some wait has timed out in
 * this process; record k (k < 7: epilogue warpgroups 0..3, row warps, producer, mma) = out[4 + 4k ..] =
 * {source line, block, thread, parity + 1} (all zero: that role was not stuck). */
int mpg_wait_debug(unsigned long long out[32]);

/* counters for bench.py: kernels launched by this handle since creation */
uint64_t mpg_launch_count(const mpg_ctx* ctx);

/* ---- GPU prioritized replay (SURVEY.md 8(f) next #1) ------------------------------------------ */
/* PrioritizedReplayBuffer (buffer.py:94-189) over sum/min segment trees (utils/segment_tree.py:13-151). */
typedef struct mpg_replay mpg_replay;
int mpg_replay_create(int capacity, int obs_dim, int act_dim, double alpha, double beta, mpg_replay** out);
void mpg_replay_destroy(mpg_replay* rb);
const char* mpg_replay_last_error(const mpg_replay* rb);
int mpg_replay_size(const mpg_replay* rb);
/* add n transitions (device pointers); priorities NULL -> current max priority (buffer.py:128-136) */
int mpg_replay_add(mpg_replay* rb, int n, const float* obs, const float* act, const float* rew, const float* obs_tp1,
                   const float* done, const float* priorities, void* stream);
/* proportional sampling (buffer.py:138-165): u = n uniforms in [0,1); writes indices, importance weights
 * (may be NULL) and the gathered transitions */
int mpg_replay_sample(mpg_replay* rb, int n, const float* u, int32_t* idx_out, float* weights_out, float* obs_out,
                      float* act_out, float* rew_out, float* obs_tp1_out, float* done_out, void* stream);
/* update_priorities (buffer.py:167-189); priorities must be > 0 (callers pass |td| + eps) */
int mpg_replay_update_priorities(mpg_replay* rb, int n, const int32_t* idx, const float* priorities, void* stream);
/* root of the sum / min trees and the running max priority (synchronises the stream) */
int mpg_replay_tree_stats(mpg_replay* rb, double* sum_out, double* min_out, double* max_priority_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPG_B200_H */
