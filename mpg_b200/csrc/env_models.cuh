// Environment models: per-row, register-resident forward step and hand-derived adjoint.
//   PathTracking      envs_and_models/path_tracking_env.py:58-138,181-199,245-297
//   InvertedPendulum  envs_and_models/inverted_pendulum_model.py:16-97
//   InvertedDoublePendulum envs_and_models/inverted_double_pendulum_model.py:14-53,89-144
// Adjoint derivations: SURVEY.md 8(a) "Adjoint the kernel must implement" + Appendix A.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace mpg {

template <int ENV>
struct Env;

// =============================================================================================
// PathTracking: state (v_x, v_y, r, delta_y, delta_phi, x); obs = (v_x-20, v_y, r, dy, dphi, x, [dy]*nfd)
// =============================================================================================
template <>
struct Env<MPG_ENV_PATH_TRACKING> {
  static constexpr int S = 6, A = 2;
  static constexpr float NOISE_MEAN = 0.5f, NOISE_STD = 0.01f;
  static constexpr bool HAS_NOISE = true;
  // vehicle_params (path_tracking_env.py:60-67)
  static constexpr float Cf = -128915.5f, Cr = -85943.6f, a = 1.06f, b = 1.85f, m = 1412.f, Iz = 1536.7f;
  static constexpr float TAU = 0.1f;
  static constexpr float K = a * Cf - b * Cr;              // a C_f - b C_r
  static constexpr float CfCr = Cf + Cr;
  static constexpr float A2 = a * a * Cf + b * b * Cr;      // a^2 C_f + b^2 C_r
  static constexpr float STEER_SCALE = (float)(1.2 * 3.14159265358979323846 / 9.0), ACC_SCALE = 3.0f;
  static constexpr float PI_F = 3.14159265358979323846f;

  __device__ static void reset(const float* o, float* s) {  // _get_state (:273-277)
    s[0] = o[0] + 20.f; s[1] = o[1]; s[2] = o[2]; s[3] = o[3]; s[4] = o[4]; s[5] = o[5];
  }
  __device__ static void get_obs(const float* s, float* o, int nfd) {  // _get_obs (:265-271)
    o[0] = s[0] - 20.f; o[1] = s[1]; o[2] = s[2]; o[3] = s[3]; o[4] = s[4]; o[5] = s[5];
#pragma unroll
    for (int i = 0; i < MPG_MAX_OBS - 6; ++i)      // fixed trip count + predicate: o[] stays in registers
      if (i < nfd) o[6 + i] = s[3];
  }
  // d obs -> d state (E of SURVEY 8(a)); go already multiplied by obs_scale
  __device__ static void obs_grad_to_state(const float*, const float* go, int nfd, float* gs) {
    gs[0] += go[0]; gs[1] += go[1]; gs[2] += go[2]; gs[3] += go[3]; gs[4] += go[4]; gs[5] += go[5];
#pragma unroll
    for (int i = 0; i < MPG_MAX_OBS - 6; ++i)
      if (i < nfd) gs[3] += go[6 + i];
  }
  __device__ static float reward_pre(const float* s, float steer, float ax) {  // compute_rewards (:181-199)
    float dv = s[0] - 20.f;
    return -(0.01f * dv * dv + 0.04f * s[3] * s[3] + 0.1f * s[4] * s[4] + 0.02f * s[2] * s[2]
             + 5.f * steer * steer + 0.05f * ax * ax);
  }
  // rollout_out (:279-297): returns RAW reward (on the pre-step state), advances s in place
  __device__ static float step(float* s, const float* act, float eps, bool noisy) {
    float steer = act[0] * STEER_SCALE, ax = act[1] * ACC_SCALE;
    float rew = reward_pre(s, steer, ax);
    float vx = s[0], vy = s[1], r = s[2], dy = s[3], phi = s[4], x = s[5];
    float sn, cs;
    sincosf(phi, &sn, &cs);
    float D1 = m * vx - TAU * CfCr;
    float N1 = m * vy * vx + TAU * K * r - TAU * Cf * steer * vx - TAU * m * vx * vx * r;
    float D2 = TAU * A2 - Iz * vx;
    float N2 = -Iz * r * vx - TAU * K * vy + TAU * a * Cf * steer * vx;
    float vx1 = vx + TAU * (ax + vy * r);
    float dy1 = dy + TAU * (vx * sn + vy * cs);
    if (noisy) dy1 += NOISE_MEAN + NOISE_STD * eps;
    float phi1 = phi + TAU * r;
    s[0] = fminf(fmaxf(vx1, 1.f), 35.f);            // tf.clip_by_value(v_xs, 1, 35)
    s[1] = N1 / D1;
    s[2] = N2 / D2;
    s[3] = dy1;
    if (phi1 > PI_F) phi1 -= 2.f * PI_F;             // wrap (:290-291)
    if (phi1 <= -PI_F) phi1 += 2.f * PI_F;
    s[4] = phi1;
    s[5] = x + TAU * (vx * cs - vy * sn);
    return rew;
  }
  // adjoint of one step. lam = d L / d s_{t+1}; rc = coefficient on the RAW reward r_t.
  // gs += (df/ds)^T lam + rc dr/ds ; ga += scale * ((df/du)^T lam + rc dr/du)
  // FAST: MUFU sin / cos / reciprocal (|phi| <= pi: absolute error ~5e-7, far inside the 1e-4 gradient tolerance);
  // used by the tensor-core kernel, where this per-row chain sits on the critical path of every BPTT step
  template <bool FAST = false>
  __device__ static void step_bwd(const float* s, const float* act, const float* lam, float rc, float* gs, float* ga) {
    float steer = act[0] * STEER_SCALE, ax = act[1] * ACC_SCALE;
    float vx = s[0], vy = s[1], r = s[2], phi = s[4];
    float sn, cs;
    if (FAST) __sincosf(phi, &sn, &cs); else sincosf(phi, &sn, &cs);
    float vx1 = vx + TAU * (ax + vy * r);
    float Lvx = (vx1 >= 1.f && vx1 <= 35.f) ? lam[0] : 0.f;  // ClipByValue grad: inclusive pass-through
    float Lvy = lam[1], Lr = lam[2], Ldy = lam[3], Lphi = lam[4], Lx = lam[5];
    float D1 = m * vx - TAU * CfCr;
    float N1 = m * vy * vx + TAU * K * r - TAU * Cf * steer * vx - TAU * m * vx * vx * r;
    float D2 = TAU * A2 - Iz * vx;
    float N2 = -Iz * r * vx - TAU * K * vy + TAU * a * Cf * steer * vx;
    float iD1 = FAST ? __fdividef(1.f, D1) : 1.f / D1, iD2 = FAST ? __fdividef(1.f, D2) : 1.f / D2;
    gs[0] += Lvx + Lvy * ((m * vy - TAU * Cf * steer - 2.f * TAU * m * vx * r) * iD1 - N1 * m * iD1 * iD1)
             + Lr * ((-Iz * r + TAU * a * Cf * steer) * iD2 + N2 * Iz * iD2 * iD2)
             + Ldy * TAU * sn + Lx * TAU * cs
             + rc * (-0.02f * (vx - 20.f));
    gs[1] += Lvx * TAU * r + Lvy * m * vx * iD1 - Lr * TAU * K * iD2 + Ldy * TAU * cs - Lx * TAU * sn;
    gs[2] += Lvx * TAU * vy + Lvy * (TAU * K - TAU * m * vx * vx) * iD1 - Lr * Iz * vx * iD2 + Lphi * TAU
             + rc * (-0.04f * r);
    gs[3] += Ldy + rc * (-0.08f * s[3]);
    gs[4] += Ldy * TAU * (vx * cs - vy * sn) + Lphi - Lx * TAU * (vx * sn + vy * cs) + rc * (-0.2f * phi);
    gs[5] += Lx;
    float g_steer = -Lvy * TAU * Cf * vx * iD1 + Lr * TAU * a * Cf * vx * iD2 + rc * (-10.f * steer);
    float g_ax = Lvx * TAU + rc * (-0.1f * ax);
    ga[0] += STEER_SCALE * g_steer;
    ga[1] += ACC_SCALE * g_ax;
  }
};

// =============================================================================================
// Inverted pendulum (cart-pole): state = obs = (p, theta, pdot, thetadot)
// =============================================================================================
template <>
struct Env<MPG_ENV_INVERTED_PENDULUM> {
  static constexpr int S = 4, A = 1;
  static constexpr float NOISE_MEAN = 0.1f, NOISE_STD = 0.5f;
  static constexpr bool HAS_NOISE = true;
  static constexpr float TAU = 0.04f, ACT_SCALE = 100.f;
  // inverted_pendulum_model.py:18-25,37-44
  static constexpr double mc = 9.42, m1 = 4.89, l1 = 0.6, g = 9.81;
  static constexpr float d1 = (float)(mc + m1);
  static constexpr float d2 = (float)(0.5 * m1 * l1);
  static constexpr float d4 = (float)(1. / 3 * m1 * l1 * l1);
  static constexpr float f1c = (float)(0.5 * m1 * l1 * g);

  __device__ static void reset(const float* o, float* s) { s[0] = o[0]; s[1] = o[1]; s[2] = o[2]; s[3] = o[3]; }
  __device__ static void get_obs(const float* s, float* o, int) { o[0] = s[0]; o[1] = s[1]; o[2] = s[2]; o[3] = s[3]; }
  __device__ static void obs_grad_to_state(const float*, const float* go, int, float* gs) {
    gs[0] += go[0]; gs[1] += go[1]; gs[2] += go[2]; gs[3] += go[3];
  }
  __device__ static float reward_post(const float* s) {  // compute_rewards (:66-74)
    return -(0.01f * s[0] * s[0] + s[1] * s[1]) - (1e-3f * s[2] * s[2] + 1e-3f * s[3] * s[3]);
  }
  __device__ static float step(float* s, const float* act, float eps, bool noisy) {
    float u = ACT_SCALE * act[0];
    float p = s[0], th = s[1], pd = s[2], thd = s[3];
    float sn, c;
    sincosf(th, &sn, &c);
    float f0 = d2 * sn * thd * thd + u, f1v = f1c * sn;
    float det = d1 * d4 - d2 * c * d2 * c;
    float pdd = (d4 * f0 - d2 * c * f1v) / det;
    float thdd = (-d2 * c * f0 + d1 * f1v) / det;
    s[0] = p + TAU * pd + (noisy ? (NOISE_MEAN + NOISE_STD * eps) : 0.f);
    s[1] = th + TAU * thd;
    s[2] = pd + TAU * pdd;
    s[3] = thd + TAU * thdd;
    return reward_post(s);  // reward on the POST-step state (:92-93)
  }
  // lam = dL/ds_{t+1} (without this step's reward); s1 = post-step state (for the reward term)
  template <bool FAST = false>
  __device__ static void step_bwd(const float* s, const float* act, const float* lam, float rc, float* gs, float* ga,
                                  const float* s1) {
    float L0 = lam[0] + rc * (-0.02f * s1[0]);
    float L1 = lam[1] + rc * (-2.f * s1[1]);
    float L2 = lam[2] + rc * (-2e-3f * s1[2]);
    float L3 = lam[3] + rc * (-2e-3f * s1[3]);
    float u = ACT_SCALE * act[0];
    float th = s[1], thd = s[3];
    float sn, c;
    sincosf(th, &sn, &c);          // theta is unbounded here: keep the accurate range reduction
    float f0 = d2 * sn * thd * thd + u, f1v = f1c * sn;
    float det = d1 * d4 - d2 * c * d2 * c;
    float N0 = d4 * f0 - d2 * c * f1v, N1 = -d2 * c * f0 + d1 * f1v;
    float idet = FAST ? __fdividef(1.f, det) : 1.f / det;
    float Aq = L2 * TAU, Bq = L3 * TAU;   // adjoints of pdd, thdd
    float aN0 = Aq * idet, aN1 = Bq * idet;
    float adet = -(Aq * N0 + Bq * N1) * idet * idet;
    float af0 = d4 * aN0 - d2 * c * aN1;
    float af1 = -d2 * c * aN0 + d1 * aN1;
    float ac = -d2 * f1v * aN0 - d2 * f0 * aN1 + adet * (-2.f * d2 * d2 * c);
    float as = af0 * d2 * thd * thd + af1 * f1c;
    gs[0] += L0;
    gs[1] += L1 + ac * (-sn) + as * c;
    gs[2] += L0 * TAU + L2;
    gs[3] += L1 * TAU + L3 + af0 * 2.f * d2 * sn * thd;
    ga[0] += ACT_SCALE * af0;
  }
};

// =============================================================================================
// Inverted double pendulum: state (p, t1, t2, pd, t1d, t2d); obs (p, sin t1, sin t2, cos t1, cos t2,
// pd, t1d, t2d, 0, 0, 0); one rollout_out = 5 sub-steps of f_xu_old at tau = 0.01.
// =============================================================================================
template <>
struct Env<MPG_ENV_INVERTED_DOUBLE_PENDULUM> {
  static constexpr int S = 6, A = 1;
  static constexpr float NOISE_MEAN = 0.f, NOISE_STD = 0.f;
  static constexpr bool HAS_NOISE = false;
  static constexpr float TAU = 0.01f, ACT_SCALE = 500.f;
  static constexpr int SUB = 5;
  static constexpr double mc = 9.42477796, m1 = 4.1033127, m2 = 4.1033127, l1 = 0.6, l2 = 0.6, g = 9.81;
  static constexpr float A11 = (float)(mc + m1 + m2);
  static constexpr float K12 = (float)(l1 * (m1 + m2));
  static constexpr float K13 = (float)(m2 * l2);
  static constexpr float A22 = (float)(l1 * l1 * (m1 + m2));
  static constexpr float K23 = (float)(l1 * l2 * m2);
  static constexpr float A33 = (float)(l2 * l2 * m2);
  static constexpr float G1 = (float)(g * (m1 + m2) * l1);
  static constexpr float G2 = (float)(g * l2 * m2);

  __device__ static void reset(const float* o, float* s) {  // _get_state (:126-132)
    s[0] = o[0]; s[1] = atan2f(o[1], o[3]); s[2] = atan2f(o[2], o[4]); s[3] = o[5]; s[4] = o[6]; s[5] = o[7];
  }
  __device__ static void get_obs(const float* s, float* o, int) {  // _get_obs (:118-124)
    float s1, c1, s2, c2;
    sincosf(s[1], &s1, &c1);
    sincosf(s[2], &s2, &c2);
    o[0] = s[0]; o[1] = s1; o[2] = s2; o[3] = c1; o[4] = c2; o[5] = s[3]; o[6] = s[4]; o[7] = s[5];
    o[8] = 0.f; o[9] = 0.f; o[10] = 0.f;
  }
  __device__ static void obs_grad_to_state(const float* s, const float* go, int, float* gs) {
    float s1, c1, s2, c2;
    sincosf(s[1], &s1, &c1);
    sincosf(s[2], &s2, &c2);
    gs[0] += go[0];
    gs[1] += go[1] * c1 - go[3] * s1;
    gs[2] += go[2] * c2 - go[4] * s2;
    gs[3] += go[5]; gs[4] += go[6]; gs[5] += go[7];
  }
  __device__ static float reward_post(const float* s) {  // compute_rewards (:89-100)
    float s1, c1, s2, c2;
    sincosf(s[1], &s1, &c1);
    sincosf(s[2], &s2, &c2);
    float tx = s[0] + 0.6f * s1 + 0.6f * s2, ty = 0.6f * c1 + 0.6f * c2;
    return -(0.01f * tx * tx + (ty - 2.f) * (ty - 2.f)) - (1e-3f * s[4] * s[4] + 5e-3f * s[5] * s[5]);
  }
  struct Sub {  // quantities of one sub-step shared by forward and adjoint
    float s1, c1, s2, c2, s12, c12, a12, a13, a23;
    float i11, i12, i13, i22, i23, i33;  // inverse of the symmetric mass matrix
    float q0, q1, q2;
  };
  __device__ static void substep_eval(const float* s, float u, Sub& w) {
    sincosf(s[1], &w.s1, &w.c1);
    sincosf(s[2], &w.s2, &w.c2);
    sincosf(s[1] - s[2], &w.s12, &w.c12);
    w.a12 = K12 * w.c1; w.a13 = K13 * w.c2; w.a23 = K23 * w.c12;
    float t1d = s[4], t2d = s[5];
    float f0 = K12 * t1d * t1d * w.s1 + K13 * t2d * t2d * w.s2 + u;
    float f1 = -K23 * t2d * t2d * w.s12 + G1 * w.s1;
    float f2 = K23 * t1d * t1d * w.s12 + G2 * w.s2;
    float c11 = A22 * A33 - w.a23 * w.a23;
    float c12 = w.a13 * w.a23 - w.a12 * A33;
    float c13 = w.a12 * w.a23 - w.a13 * A22;
    float c22 = A11 * A33 - w.a13 * w.a13;
    float c23 = w.a12 * w.a13 - A11 * w.a23;
    float c33 = A11 * A22 - w.a12 * w.a12;
    float idet = 1.f / (A11 * c11 + w.a12 * c12 + w.a13 * c13);
    w.i11 = c11 * idet; w.i12 = c12 * idet; w.i13 = c13 * idet;
    w.i22 = c22 * idet; w.i23 = c23 * idet; w.i33 = c33 * idet;
    w.q0 = w.i11 * f0 + w.i12 * f1 + w.i13 * f2;
    w.q1 = w.i12 * f0 + w.i22 * f1 + w.i23 * f2;
    w.q2 = w.i13 * f0 + w.i23 * f1 + w.i33 * f2;
  }
  __device__ static void substep(float* s, float u) {  // f_xu_old (:26-53)
    Sub w;
    substep_eval(s, u, w);
    float n0 = s[0] + TAU * s[3], n1 = s[1] + TAU * s[4], n2 = s[2] + TAU * s[5];
    s[3] += TAU * w.q0; s[4] += TAU * w.q1; s[5] += TAU * w.q2;
    s[0] = n0; s[1] = n1; s[2] = n2;
  }
  __device__ static float step(float* s, const float* act, float, bool) {  // rollout_out (:134-141)
    float u = ACT_SCALE * act[0];
#pragma unroll 1
    for (int i = 0; i < SUB; ++i) substep(s, u);
    return reward_post(s);
  }
  // L (in/out): adjoint of the sub-step output -> adjoint of its input; returns d/du
  __device__ static float substep_bwd(const float* s, float u, float* L) {
    Sub w;
    substep_eval(s, u, w);
    float aq0 = TAU * L[3], aq1 = TAU * L[4], aq2 = TAU * L[5];
    // adj_f = A^-1 adj_q (A symmetric)
    float af0 = w.i11 * aq0 + w.i12 * aq1 + w.i13 * aq2;
    float af1 = w.i12 * aq0 + w.i22 * aq1 + w.i23 * aq2;
    float af2 = w.i13 * aq0 + w.i23 * aq1 + w.i33 * aq2;
    // adj_A = -adj_f q^T ; symmetric off-diagonals appear twice
    float aa12 = -(af0 * w.q1 + af1 * w.q0);
    float aa13 = -(af0 * w.q2 + af2 * w.q0);
    float aa23 = -(af1 * w.q2 + af2 * w.q1);
    float t1d = s[4], t2d = s[5];
    float ac1 = K12 * aa12, ac2 = K13 * aa13, ac12 = K23 * aa23;
    float as1 = af0 * K12 * t1d * t1d + af1 * G1;
    float as2 = af0 * K13 * t2d * t2d + af2 * G2;
    float as12 = -af1 * K23 * t2d * t2d + af2 * K23 * t1d * t1d;
    float at1d = af0 * 2.f * K12 * t1d * w.s1 + af2 * 2.f * K23 * t1d * w.s12;
    float at2d = af0 * 2.f * K13 * t2d * w.s2 - af1 * 2.f * K23 * t2d * w.s12;
    float at1 = -w.s1 * ac1 + w.c1 * as1 - w.s12 * ac12 + w.c12 * as12;
    float at2 = -w.s2 * ac2 + w.c2 * as2 + w.s12 * ac12 - w.c12 * as12;
    float g0 = L[0], g1 = L[1] + at1, g2 = L[2] + at2;
    float g3 = L[3] + TAU * L[0], g4 = L[4] + TAU * L[1] + at1d, g5 = L[5] + TAU * L[2] + at2d;
    L[0] = g0; L[1] = g1; L[2] = g2; L[3] = g3; L[4] = g4; L[5] = g5;
    return af0;
  }
  __device__ static void step_bwd(const float* s, const float* act, const float* lam, float rc, float* gs, float* ga,
                                  const float* /*s1 unused: recomputed*/) {
    float u = ACT_SCALE * act[0];
    float st[SUB + 1][S];
#pragma unroll
    for (int j = 0; j < S; ++j) st[0][j] = s[j];
#pragma unroll
    for (int i = 0; i < SUB; ++i) {
#pragma unroll
      for (int j = 0; j < S; ++j) st[i + 1][j] = st[i][j];
      substep(st[i + 1], u);
    }
    const float* e = st[SUB];
    float s1, c1, s2, c2;
    sincosf(e[1], &s1, &c1);
    sincosf(e[2], &s2, &c2);
    float tx = e[0] + 0.6f * s1 + 0.6f * s2, ty = 0.6f * c1 + 0.6f * c2;
    float L[S];
    L[0] = lam[0] + rc * (-0.02f * tx);
    L[1] = lam[1] + rc * (-0.02f * tx * 0.6f * c1 + 2.f * (ty - 2.f) * 0.6f * s1);
    L[2] = lam[2] + rc * (-0.02f * tx * 0.6f * c2 + 2.f * (ty - 2.f) * 0.6f * s2);
    L[3] = lam[3];
    L[4] = lam[4] + rc * (-2e-3f * e[4]);
    L[5] = lam[5] + rc * (-1e-2f * e[5]);
    float gu = 0.f;
#pragma unroll
    for (int i = SUB - 1; i >= 0; --i) gu += substep_bwd(st[i], u, L);
#pragma unroll
    for (int j = 0; j < S; ++j) gs[j] += L[j];
    ga[0] += ACT_SCALE * gu;
  }
};

// =============================================================================================
// PathTracking REAL environment (the ground truth the model approximates; SURVEY.md 8(f) next #3):
// PathTrackingEnv.reset(init_obs)/step/_get_obs/judge_done (path_tracking_env.py:356-487), VehicleDynamics.simulation
// (:144-179: 20 sub-steps of the non-model f_xu at 200 Hz with v_x clip, semi-implicit pose integration, projection on
// the reference path, period / angle wraps) and ReferencePath (:202-242).  Forward only (it is used for targets and
// acting, never differentiated).  state = (v_x, v_y, r, delta_y, delta_phi, x, y, phi).
// =============================================================================================
constexpr int MPG_ENV_PT_REAL = MPG_ENV_PATH_TRACKING_REAL;
template <>
struct Env<MPG_ENV_PT_REAL> {
  using Mdl = Env<MPG_ENV_PATH_TRACKING>;
  static constexpr int S = 8, A = 2;
  static constexpr bool HAS_NOISE = false;
  static constexpr float PI_F = 3.14159265358979323846f;
  static constexpr float PERIOD = 1200.f, FREQ = 200.f;
  static constexpr int SUBSTEPS = 20;

  __device__ static float path_y(float x) {   // ReferencePath.compute_path_y (:207-212), fp32 in the reference's op order
    return 7.5f * sinf(x * 2.f * PI_F / 200.f) + 2.5f * sinf(x * 2.f * PI_F / 300.f) + (-5.f) * sinf(x * 2.f * PI_F / 400.f);
  }
  __device__ static float path_phi(float x) {  // compute_path_phi (:214-220)
    const float d = (float)(7.5 * 2 * 3.14159265358979323846 / 200.) * cosf(x * 2.f * PI_F / 200.f)
                    + (float)(2.5 * 2 * 3.14159265358979323846 / 300.) * cosf(x * 2.f * PI_F / 300.f)
                    + (float)(-5. * 2 * 3.14159265358979323846 / 400.) * cosf(x * 2.f * PI_F / 400.f);
    return atanf(d);
  }
  __device__ static void reset(const float* o, float* s) {   // reset(init_obs=...) (:410-420)
    Mdl::reset(o, s);
    s[6] = s[3] + path_y(s[5]);
    s[7] = s[4] + path_phi(s[5]);
  }
  __device__ static void get_obs(const float* s, float* o, int nfd) {   // _get_obs (:384-402)
    o[0] = s[0] - 20.f; o[1] = s[1]; o[2] = s[2]; o[3] = s[3]; o[4] = s[4]; o[5] = s[5];
    float x_ = s[5];
#pragma unroll 1
    for (int i = 0; i < nfd; ++i) {
      x_ += s[0] * 1.f / FREQ * (float)SUBSTEPS * 2.f;
      const float v = s[6] - path_y(x_);
#pragma unroll
      for (int k = 0; k < MPG_MAX_OBS - 6; ++k)
        if (k == i) o[6 + k] = v;
    }
  }
  // step (:456-472); returns the RAW reward (pre-step state, clipped scaled action); *done gets judge_done (:474-487)
  __device__ static float step_done(float* s, const float* act, int* done) {
    float steer = act[0] * 1.2f * PI_F / 9.f, ax = act[1] * 3.f;
    const float smax = 1.2f * PI_F / 9.f;
    steer = fminf(fmaxf(steer, -smax), smax);
    ax = fminf(fmaxf(ax, -3.f), 3.f);
    const float rew = Mdl::reward_pre(s, steer, ax);
    constexpr float tau = 1.f / 200.f;
    constexpr float Cf = Mdl::Cf, Cr = Mdl::Cr, a = Mdl::a, b = Mdl::b, m = Mdl::m, Iz = Mdl::Iz;
    float vx = s[0], vy = s[1], r = s[2], x = s[5], y = s[6], phi = s[7], dy = s[3], dphi = s[4];
    float alpha_f = 0.f, alpha_r = 0.f, vx_in = vx;
    for (int it = 0; it < SUBSTEPS; ++it) {
      vx_in = vx;
      alpha_f = atanf((vy + a * r) / vx) - steer;   // stability_related of THIS prediction call (:105-106)
      alpha_r = atanf((vy - b * r) / vx);
      const float vx1 = fminf(fmaxf(vx + tau * (ax + vy * r), 1.f), 35.f);
      const float vy1 = (m * vy * vx + tau * Mdl::K * r - tau * Cf * steer * vx - tau * m * vx * vx * r) / (m * vx - tau * Mdl::CfCr);
      const float r1 = (-Iz * r * vx - tau * Mdl::K * vy + tau * a * Cf * steer * vx) / (tau * Mdl::A2 - Iz * vx);
      // pose: phi first (numpy views make the following lines see the UPDATED phi), old v_x, v_y, r (:160-165)
      phi += r / FREQ;
      float sn, cs;
      sincosf(phi, &sn, &cs);
      y += (vx * sn + vy * cs) / FREQ;
      x += (vx * cs - vy * sn) / FREQ;
      vx = vx1; vy = vy1; r = r1;
      dphi = phi - path_phi(x);
      dy = y - path_y(x);
      if (phi > PI_F) phi -= 2.f * PI_F;
      if (phi <= -PI_F) phi += 2.f * PI_F;
      if (x > PERIOD) x -= PERIOD;
      if (x <= 0.f) x += PERIOD;
      if (dphi > PI_F) dphi -= 2.f * PI_F;
      if (dphi <= -PI_F) dphi += 2.f * PI_F;
    }
    s[0] = vx; s[1] = vy; s[2] = r; s[3] = dy; s[4] = dphi; s[5] = x; s[6] = y; s[7] = phi;
    if (done) {
      // bounds from the last prediction call (:97-104,135-137); g = 9.81, miu = 1
      const float g = 9.81f, F_zf = b * m * g / (a + b), F_zr = a * m * g / (a + b);
      const float F_xf = ax < 0.f ? m * ax / 2.f : 0.f, F_xr = ax < 0.f ? m * ax / 2.f : m * ax;
      const float miu_f = sqrtf(F_zf * F_zf - F_xf * F_xf) / F_zf, miu_r = sqrtf(F_zr * F_zr - F_xr * F_xr) / F_zr;
      const float af_b = 3.f * miu_f * F_zf / Cf, ar_b = 3.f * miu_r * F_zr / Cr;   // negative: C_f, C_r < 0
      const float r_b = miu_r * g / fabsf(vx_in);   // |v_x| entering the last sub-step, like the last prediction() call
      *done = (fabsf(dy) > 3.f) | (fabsf(dphi) > PI_F / 4.f) | (vx < 2.f) | (alpha_f < -af_b) | (alpha_f > af_b)
              | (alpha_r < -ar_b) | (alpha_r > ar_b) | (r < -r_b) | (r > r_b);
    }
    return rew;
  }
  __device__ static float step(float* s, const float* act, float, bool) { return step_done(s, act, nullptr); }
  __device__ static void obs_grad_to_state(const float*, const float*, int, float*) {}
};

// uniform wrapper so the rollout kernel does not care whether the reward is pre- or post-step
template <int ENV, bool FAST = false>
__device__ __forceinline__ void env_step_bwd(const float* s, const float* act, const float* lam, float rc, float* gs,
                                             float* ga, const float* s1) {
  if constexpr (ENV == MPG_ENV_PATH_TRACKING) Env<ENV>::template step_bwd<FAST>(s, act, lam, rc, gs, ga);
  else if constexpr (ENV == MPG_ENV_PT_REAL) { }   // the real environment is never differentiated
  else if constexpr (ENV == MPG_ENV_INVERTED_PENDULUM) Env<ENV>::template step_bwd<FAST>(s, act, lam, rc, gs, ga, s1);
  else Env<ENV>::step_bwd(s, act, lam, rc, gs, ga, s1);
}

// The one place a runtime environment id (MPG_ENV_*) and backward flag become the template arguments of a kernel: calls
// f(integral_constant<int, ENV>, integral_constant<bool, BWD>) and returns true.  The real environment is forward only: with
// bwd set it has no kernel, and with_env calls nothing and returns false.
template <typename F>
bool with_env(int env, bool bwd, F&& f) {
  auto fwd_or_bwd = [&](auto e) {
    if (bwd) f(e, std::true_type()); else f(e, std::false_type());
    return true;
  };
  switch (env) {
    case MPG_ENV_PATH_TRACKING: return fwd_or_bwd(std::integral_constant<int, MPG_ENV_PATH_TRACKING>());
    case MPG_ENV_INVERTED_PENDULUM: return fwd_or_bwd(std::integral_constant<int, MPG_ENV_INVERTED_PENDULUM>());
    case MPG_ENV_PATH_TRACKING_REAL:
      if (bwd) return false;
      f(std::integral_constant<int, MPG_ENV_PATH_TRACKING_REAL>(), std::false_type());
      return true;
    default: return fwd_or_bwd(std::integral_constant<int, MPG_ENV_INVERTED_DOUBLE_PENDULUM>());
  }
}
// f(ENV, BWD) for every variant with_env selects
template <typename F>
void for_each_env(F&& f) {
  for (int env = MPG_ENV_PATH_TRACKING; env <= MPG_ENV_PATH_TRACKING_REAL; ++env) {
    with_env(env, false, f);
    with_env(env, true, f);
  }
}

}  // namespace mpg
