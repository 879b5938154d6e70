"""Deterministic synthetic inputs shared by tests, golden-vector generation and bench.py.

Everything is numpy + `np.random.default_rng` (PCG64 streams are stable across numpy versions),
so the same seed gives the same states / weights / noise in the build container (where the
golden vectors are made) and on the GPU box.

Start-state laws follow the reference's env reset (SURVEY.md 8(d)):
  PathTracking  envs_and_models/path_tracking_env.py:426-439
  pendulums     envs_and_models/inverted_pendulum_conti.py:17 (done bounds) / mujoco qpos ranges
Weights follow model.py:23-36: Orthogonal(sqrt 2) hidden kernels, Orthogonal(1) output kernel.
Biases are drawn small-but-nonzero (the reference starts them at 0) so bias paths are exercised.
"""
import numpy as np

ENV_DIMS = {
    # env_id: (obs_dim without future data, act_dim, state_dim)
    'PathTracking-v0': (6, 2, 6),
    'InvertedPendulumConti-v0': (4, 1, 4),
    'InvertedDoublePendulum-v2': (11, 1, 6),
}


def orthogonal(rng, rows, cols, gain):
    """Keras-style Orthogonal initializer: QR of a normal matrix, sign-fixed, shape (rows, cols)."""
    n, m = max(rows, cols), min(rows, cols)
    a = rng.standard_normal((n, m))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    if rows < cols:
        q = q.T
    return (gain * q[:rows, :cols]).astype(np.float32)


def make_mlp_weights(rng, in_dim, hidden, out_dim, bias_scale=0.05, layers=2):
    """[W1,b1,W2,b2,..,WL,bL,Wout,bout] (L = layers hidden layers) with Keras (in,out) kernels, fp32 (model.py:20-43
    order).  The draws are made in list order, so at layers = 2 a seed gives the same weights it always gave."""
    g = np.sqrt(2.0)
    w = [orthogonal(rng, in_dim, hidden, g), (bias_scale * rng.standard_normal(hidden)).astype(np.float32)]
    for _ in range(layers - 1):
        w += [orthogonal(rng, hidden, hidden, g), (bias_scale * rng.standard_normal(hidden)).astype(np.float32)]
    return w + [orthogonal(rng, hidden, out_dim, 1.0), (bias_scale * rng.standard_normal(out_dim)).astype(np.float32)]


def make_policy_with_qs_weights(seed, obs_dim, act_dim, hidden=256, double_q=True, layers=2):
    """Weights in PolicyWithQs.get_weights() order: models + target_models (policy.py:72-89,112-121).
    double_q: [Q1,Q2,policy, Q1t,Q2t,policyt]; else [Q1,policy, Q1t,policyt]. Targets are
    independent draws (not copies) so that target-network paths are distinguishable in tests."""
    rng = np.random.default_rng(seed)
    def q():
        return make_mlp_weights(rng, obs_dim + act_dim, hidden, 1, layers=layers)
    def pi():
        return make_mlp_weights(rng, obs_dim, hidden, 2 * act_dim, layers=layers)
    if double_q:
        return [q(), q(), pi(), q(), q(), pi()]
    return [q(), pi(), q(), pi()]


def make_obs(rng, env_id, batch, num_future_data=0):
    """Start observations (B, obs_dim) fp32 from the env reset law."""
    if env_id == 'PathTracking-v0':
        x = rng.uniform(0.0, 600.0, batch)
        dy = rng.normal(0.0, 1.0, batch)
        dphi = rng.normal(0.0, np.pi / 9, batch)
        vx = rng.uniform(15.0, 25.0, batch)
        beta = rng.normal(0.0, 0.15, batch)
        vy = vx * np.tan(beta)
        r = rng.normal(0.0, 0.3, batch)
        cols = [vx - 20.0, vy, r, dy, dphi, x] + [dy] * num_future_data
        return np.stack(cols, 1).astype(np.float32)
    if env_id == 'InvertedPendulumConti-v0':
        p = rng.uniform(-1.0, 1.0, batch)
        th = rng.uniform(-0.2, 0.2, batch)
        pd = rng.normal(0.0, 0.5, batch)
        thd = rng.normal(0.0, 0.5, batch)
        return np.stack([p, th, pd, thd], 1).astype(np.float32)
    if env_id == 'InvertedDoublePendulum-v2':
        p = rng.uniform(-1.0, 1.0, batch)
        t1 = rng.uniform(-0.2, 0.2, batch)
        t2 = rng.uniform(-0.2, 0.2, batch)
        pd = rng.normal(0.0, 0.5, batch)
        t1d = rng.normal(0.0, 0.5, batch)
        t2d = rng.normal(0.0, 0.5, batch)
        z = np.zeros(batch)
        return np.stack([p, np.sin(t1), np.sin(t2), np.cos(t1), np.cos(t2), pd, t1d, t2d, z, z, z], 1).astype(np.float32)
    raise ValueError(env_id)


def make_noise(rng, n_steps, rows):
    """Standard-normal eps (n_steps, rows) fp32; the model applies mean/std (0.5,0.01)/(0.1,0.5)."""
    return rng.standard_normal((n_steps, rows)).astype(np.float32)


def default_obs_scale(env_id, num_future_data=0):
    """train_script.py:276-281 / train_script4mujoco.py:267. The reference ships no 11-long scale
    for the double pendulum; 1.0 is used and reported as such (SURVEY.md 8(d) config 3)."""
    if env_id == 'PathTracking-v0':
        return [1., 1., 2., 1., 2.4, 1 / 1200] + [1.] * num_future_data
    if env_id == 'InvertedPendulumConti-v0':
        return [0.001, 1 / 3, 0.1, 0.5]
    return [1.0] * 11


def philox_normal(seed, rows, n_steps, global_rows=None, row_offset=0, M=1):
    """numpy restatement of the in-kernel noise stream (csrc/common.cuh: philox4x32_10 + Box-Muller):
    eps[t, m*rows + i] keyed by (seed, m*global_rows + row_offset + i, t). Returns (n_steps, M*rows) fp32."""
    global_rows = rows if global_rows is None else global_rows
    m_idx, i_idx = np.divmod(np.arange(M * rows, dtype=np.uint64), np.uint64(rows))
    nrow = m_idx * np.uint64(global_rows) + np.uint64(row_offset) + i_idx
    t = np.arange(n_steps, dtype=np.uint64)[:, None]
    c0 = np.broadcast_to((nrow & np.uint64(0xFFFFFFFF))[None, :], (n_steps, M * rows)).copy()
    c1 = np.broadcast_to((nrow >> np.uint64(32))[None, :], (n_steps, M * rows)).copy()
    c2 = np.broadcast_to(t, (n_steps, M * rows)).copy()
    c3 = np.zeros_like(c0)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    M0, M1, W0, W1, MASK = (np.uint64(v) for v in (0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF))
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    f = np.float32
    u1 = (c0.astype(f) + f(0.5)) * f(2.3283064365386963e-10)
    u2 = (c1.astype(f) + f(0.5)) * f(2.3283064365386963e-10)
    u1 = np.clip(u1, f(1e-12), f(1.0))
    return (np.sqrt(f(-2.0) * np.log(u1)) * np.cos(np.float64(2.0 * np.pi) * u2.astype(np.float64))).astype(f)
