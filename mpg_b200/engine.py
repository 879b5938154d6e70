"""Engine: one opaque libmpg_b200 handle + torch tensors for device memory and streams.

PyTorch is plumbing here (allocation, H2D/D2H, streams, torch.distributed); all arithmetic of the
hot path happens in the hand-written sm_100a kernels behind the C ABI (include/mpg_b200.h).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import MpgConfig, RolloutParams, ENV_IDS

BACKEND_FFMA, BACKEND_TC = 0, 1


def _ptr(t):
    if t is None:
        return None
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), 'expected a contiguous fp32 CUDA tensor'
    return ctypes.c_void_p(t.data_ptr())


class Engine:
    """Owns an mpg_ctx. kwargs are the learner's `args` (mpg_learner.py:30-58 / nadp.py:29-47)."""

    def __init__(self, env_id, obs_dim, act_dim, obs_scale, rew_scale, rew_shift, gamma,
                 policy_out_activation='tanh', action_range=None, num_future_data=0, hidden=256,
                 max_rows=4096, max_horizon=25, device=None, debug_lib=False, hidden_activation='elu', **_unused):
        self.lib = _lib.load(debug=bool(debug_lib))   # debug_lib: the library with the development probes (tests / tools)
        if not torch.cuda.is_available():
            raise RuntimeError('mpg_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        if env_id not in ENV_IDS:
            raise ValueError(f'unknown env_id {env_id!r}')
        if hidden_activation not in _lib.ACTIVATIONS:
            raise ValueError(f'hidden_activation must be one of {sorted(_lib.ACTIVATIONS)} (got {hidden_activation!r})')
        self.hidden_activation = hidden_activation
        self.env_id, self.obs_dim, self.act_dim = env_id, int(obs_dim), int(act_dim)
        cfg = MpgConfig()
        cfg.env = ENV_IDS[env_id]
        cfg.num_future_data = int(num_future_data) if env_id.startswith('PathTracking-v0') else 0
        cfg.obs_dim, cfg.act_dim, cfg.hidden = int(obs_dim), int(act_dim), int(hidden)
        cfg.policy_out_tanh = 1 if policy_out_activation == 'tanh' else 0
        cfg.action_range = float(action_range) if action_range is not None else 0.0
        scale = list(obs_scale) if obs_scale is not None else [1.0] * obs_dim
        if len(scale) != obs_dim:
            raise ValueError('obs_scale length must equal obs_dim')
        for i in range(_lib.MAX_OBS):
            cfg.obs_scale[i] = float(scale[i]) if i < obs_dim else 1.0
        cfg.rew_scale = float(rew_scale) if rew_scale is not None else 1.0
        cfg.rew_shift = float(rew_shift) if rew_shift is not None else 0.0
        cfg.gamma = float(gamma)
        cfg.max_rows, cfg.max_horizon = int(max_rows), int(max_horizon)
        self.cfg = cfg
        self._weights = {}
        self.h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            rc = self.lib.mpg_create(ctypes.byref(cfg), ctypes.byref(self.h))
        if rc != 0:
            raise RuntimeError('mpg_create failed: ' + self.lib.mpg_last_error(None).decode())
        self._check(self.lib.mpg_set_activation(self.h, _lib.ACTIVATIONS[hidden_activation]))
        self.state_dim = self.lib.mpg_state_dim(self.h)
        self.num_sms = self.lib.mpg_num_sms(self.h)

    # ------------------------------------------------------------------ lifetime / capacity
    def close(self):
        if getattr(self, 'h', None) is not None and self.h.value:
            self.lib.mpg_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def ensure_capacity(self, rows, horizon):
        if rows <= self.cfg.max_rows and horizon <= self.cfg.max_horizon:
            return
        backend = self.backend
        saved = {net: self.get_net_weights(net) for net in self._weights}
        moments = {net: self.get_adam_state(net) for net in self._weights}   # the optimiser state moves to the new handle
        self.close()
        self.cfg.max_rows = max(int(rows), self.cfg.max_rows)
        self.cfg.max_horizon = max(int(horizon), self.cfg.max_horizon)
        with torch.cuda.device(self.device):
            rc = self.lib.mpg_create(ctypes.byref(self.cfg), ctypes.byref(self.h))
        if rc != 0:
            raise RuntimeError('mpg_create failed: ' + self.lib.mpg_last_error(None).decode())
        self._check(self.lib.mpg_set_activation(self.h, _lib.ACTIVATIONS[self.hidden_activation]))
        for net, w in saved.items():
            self.set_net_weights(net, w)
            m, v = moments[net]
            if m.any() or v.any():
                self.set_adam_state(net, m, v)
        self.set_backend(backend)

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(f'libmpg_b200 error {rc}: ' + self.lib.mpg_last_error(self.h).decode())

    @property
    def stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def backend(self):
        return self.lib.mpg_get_backend(self.h)

    def set_backend(self, backend):
        self._check(self.lib.mpg_set_backend(self.h, int(backend)))

    def tc_available(self):
        """True when the tensor-core backend covers this configuration (the current backend is left as it was)."""
        prev = self.backend
        ok = self.lib.mpg_set_backend(self.h, BACKEND_TC) == 0
        self.lib.mpg_set_backend(self.h, prev)
        return ok

    def tc_selftest(self, kind, X, W, repeats=1):
        """GEMM building-block self test: needs Engine(..., debug_lib=True)."""
        Z = self.empty(256 if kind == 5 else 128, 16 if kind == 2 else 256)
        self._check(self.lib.mpg_tc_selftest(self.h, kind, _ptr(X), _ptr(W), _ptr(Z), repeats, self.stream))
        return Z

    def set_timing(self, enabled):
        self._check(self.lib.mpg_set_timing(self.h, int(bool(enabled))))

    def kernel_ms(self):
        return float(self.lib.mpg_kernel_ms(self.h))

    @property
    def launch_count(self):
        return int(self.lib.mpg_launch_count(self.h))

    def param_count(self, net):
        return self.lib.mpg_param_count(self.h, net)

    def dev(self, x):
        """numpy / tensor -> contiguous fp32 CUDA tensor on this engine's device."""
        if isinstance(x, torch.Tensor):
            return x.to(self.device, torch.float32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(self.device, non_blocking=True)

    def empty(self, *shape):
        return torch.empty(*shape, dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ weights
    def net_shapes(self, net):
        """Keras shapes [W1,b1,W2,b2,W3,b3] of slot `net` (model.py:20-43: kernels are (in, out))."""
        is_pol = net in (_lib.NET_POLICY, _lib.NET_POLICY_TARGET)
        i, o, h = (self.obs_dim, 2 * self.act_dim, self.cfg.hidden) if is_pol else (self.obs_dim + self.act_dim, 1, self.cfg.hidden)
        return [(i, h), (h,), (h, h), (h,), (h, o), (o,)]

    def set_net_weights(self, net, weights):
        """weights: [W1,b1,W2,b2,W3,b3] numpy arrays or tensors in Keras layout (model.py:20-43).
        Like Keras' set_weights, a wrong count or shape raises ValueError (the C side copies fixed sizes)."""
        weights = list(weights)
        want = self.net_shapes(net)
        if len(weights) != 6:
            raise ValueError(f'net {net}: expected 6 weight arrays [W1,b1,W2,b2,W3,b3], got {len(weights)}')
        for k, (w, shp) in enumerate(zip(weights, want)):
            if tuple(np.shape(w)) != shp:
                raise ValueError(f'net {net}: weight {k} has shape {tuple(np.shape(w))}, expected {shp}')
        ts = [self.dev(w) for w in weights]
        arr = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in ts])
        self._check(self.lib.mpg_set_weights(self.h, net, arr, self.stream))
        self._weights[net] = ts

    def get_net_weights(self, net):
        """Current weights of `net` read back from the handle (they change under mpg_adam_step / polyak)."""
        ts = [torch.empty_like(t) for t in self._weights[net]]
        arr = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in ts])
        self._check(self.lib.mpg_get_weights(self.h, net, arr, self.stream))
        return [t.cpu().numpy() for t in ts]

    def adam_step(self, net, grad, lr, step, beta1=0.9, beta2=0.999, eps=1e-7):
        self._check(self.lib.mpg_adam_step(self.h, net, _ptr(grad), float(lr), int(step), beta1, beta2, eps, self.stream))

    def get_adam_state(self, net):
        n = self.param_count(net)
        m, v = torch.empty(n, device=self.device), torch.empty(n, device=self.device)
        self._check(self.lib.mpg_get_adam_state(self.h, net, _ptr(m), _ptr(v), self.stream))
        return m.cpu().numpy(), v.cpu().numpy()

    def set_adam_state(self, net, m, v):
        m, v = self.dev(m).contiguous(), self.dev(v).contiguous()
        if m.numel() != self.param_count(net) or v.numel() != m.numel():
            raise ValueError('adam state size does not match the net')
        self._check(self.lib.mpg_set_adam_state(self.h, net, _ptr(m), _ptr(v), self.stream))
        torch.cuda.current_stream(self.device).synchronize()

    def polyak_update(self, src_net, dst_net, tau):
        self._check(self.lib.mpg_polyak_update(self.h, src_net, dst_net, float(tau), self.stream))

    # ------------------------------------------------------------------ rollouts
    def _params(self, rows, M, horizon, rollout_list, list_w, full_bptt, q_net, policy_net, global_rows, row_offset,
                noise_seed, use_philox, real_env=False):
        p = RolloutParams()
        p.rows, p.M, p.horizon, p.n_list = int(rows), int(M), int(horizon), len(rollout_list)
        for i, k in enumerate(rollout_list):
            p.list[i] = int(k)
            p.list_w[i] = float(list_w[i])
        p.full_bptt, p.q_net, p.policy_net = int(full_bptt), int(q_net), int(policy_net)
        p.global_rows, p.row_offset = int(global_rows or rows), int(row_offset)
        p.noise_seed, p.use_philox, p.real_env = int(noise_seed), int(use_philox), int(bool(real_env))
        return p

    def policy_grad(self, obs, rollout_list, list_w, M=1, full_bptt=True, q_net=_lib.NET_Q1, policy_net=_lib.NET_POLICY,
                    noise=None, use_philox=False, noise_seed=0, global_rows=None, row_offset=0, want_returns=True):
        """-> (flat unclipped gradient (P,), returns (n_list, M*rows) or None)."""
        rows, horizon = obs.shape[0], max(rollout_list)
        if self.backend == BACKEND_TC and full_bptt and rows * M > self.MAX_TC_FULL_BPTT_ROWS:
            return self._policy_grad_chunked(obs, rollout_list, list_w, M, q_net, policy_net, noise, use_philox,
                                             noise_seed, global_rows, row_offset, want_returns)
        self.ensure_capacity(rows * M, horizon)
        p = self._params(rows, M, horizon, rollout_list, list_w, full_bptt, q_net, policy_net, global_rows, row_offset,
                         noise_seed, use_philox)
        grad = self.empty(self.param_count(policy_net))
        ret = self.empty(len(rollout_list), M * rows) if want_returns else None
        self._check(self.lib.mpg_policy_grad(self.h, ctypes.byref(p), _ptr(obs), _ptr(noise), _ptr(grad), _ptr(ret),
                                             self.stream))
        return grad, ret

    # The tensor-core full-BPTT path records 110 KB of dW operands per row (DESIGN.md 3): bound it per call.
    MAX_TC_FULL_BPTT_ROWS = 262144    # 53 KB of dW2 operand records per row at n = 25: 14 GB

    def _policy_grad_chunked(self, obs, rollout_list, list_w, M, q_net, policy_net, noise, use_philox, noise_seed,
                             global_rows, row_offset, want_returns):
        """Row chunks of one call: every chunk is scaled by 1/(M*global_rows) and keyed by its global row offset,
        so the chunk gradients simply add up (the same property the multi-GPU shards rely on)."""
        rows = obs.shape[0]
        per = self.MAX_TC_FULL_BPTT_ROWS // M
        grad, rets = None, []
        for lo in range(0, rows, per):
            hi = min(rows, lo + per)
            nz = None
            if noise is not None:   # (n, M*rows): columns m*rows + [lo, hi) of every tile
                nz = torch.cat([noise[:, m * rows + lo: m * rows + hi] for m in range(M)], 1).contiguous()
            g, r = self.policy_grad(obs[lo:hi].contiguous(), rollout_list, list_w, M=M, full_bptt=True, q_net=q_net,
                                    policy_net=policy_net, noise=nz, use_philox=use_philox, noise_seed=noise_seed,
                                    global_rows=global_rows or rows, row_offset=row_offset + lo, want_returns=want_returns)
            grad = g if grad is None else grad.add_(g)
            rets.append(r)
        ret = None
        if want_returns:   # back to the (n_list, M*rows) layout: tile m of all chunks, then tile m+1, ...
            ret = torch.cat([torch.cat([r[:, m * (r.shape[1] // M):(m + 1) * (r.shape[1] // M)] for r in rets], 1)
                             for m in range(M)], 1).contiguous()
        return grad, ret

    def rollout_forward(self, obs, rollout_list, M=1, q_net=_lib.NET_Q1, policy_net=_lib.NET_POLICY, start_actions=None,
                        noise=None, use_philox=False, noise_seed=0, global_rows=None, row_offset=0, want_traj=False,
                        horizon=None, real_env=False):
        rows = obs.shape[0]
        horizon = max(rollout_list) if horizon is None else horizon
        self.ensure_capacity(rows * M, horizon)
        p = self._params(rows, M, horizon, rollout_list, [1.0] * len(rollout_list), 0, q_net, policy_net, global_rows,
                         row_offset, noise_seed, use_philox, real_env)
        ret = self.empty(max(len(rollout_list), 1), M * rows)
        traj = (None, None, None)
        if want_traj:
            traj = (self.empty(horizon, M * rows, self.obs_dim), self.empty(horizon, M * rows),
                    self.empty(horizon + 1, M * rows, self.act_dim))
        self._check(self.lib.mpg_rollout_forward(self.h, ctypes.byref(p), _ptr(obs), _ptr(start_actions), _ptr(noise),
                                                 _ptr(ret), _ptr(traj[0]), _ptr(traj[1]), _ptr(traj[2]), self.stream))
        return (ret,) + traj if want_traj else ret

    def philox_noise(self, rows, M, horizon, noise_seed, global_rows=None, row_offset=0):
        p = self._params(rows, M, horizon, [], [], 0, -1, _lib.NET_POLICY, global_rows, row_offset, noise_seed, 1)
        out = self.empty(horizon, M * rows)
        self._check(self.lib.mpg_philox_noise(self.h, ctypes.byref(p), _ptr(out), self.stream))
        return out

    def returns_stats(self, returns, rows, M):
        n_list = returns.shape[0]
        out = self.empty(2 * n_list)
        self._check(self.lib.mpg_returns_stats(self.h, _ptr(returns), n_list, rows, M, _ptr(out), self.stream))
        return out

    def returns_tile_mean(self, returns, rows, M):
        n_list = returns.shape[0]
        out = self.empty(n_list, rows)
        self._check(self.lib.mpg_returns_tile_mean(self.h, _ptr(returns), n_list, rows, M, _ptr(out), self.stream))
        return out

    # ------------------------------------------------------------------ Q side
    def q_grad(self, net, obs, act, target, global_rows=None):
        rows = obs.shape[0]
        grad, loss = self.empty(self.param_count(net)), self.empty(1)
        self._check(self.lib.mpg_q_grad(self.h, net, rows, int(global_rows or rows), _ptr(obs), _ptr(act), _ptr(target),
                                        _ptr(grad), _ptr(loss), self.stream))
        return grad, loss

    def policy_forward(self, net, obs):
        out = self.empty(obs.shape[0], self.act_dim)
        self._check(self.lib.mpg_policy_forward(self.h, net, obs.shape[0], _ptr(obs), _ptr(out), self.stream))
        return out

    def q_forward(self, net, obs, act):
        out = self.empty(obs.shape[0])
        self._check(self.lib.mpg_q_forward(self.h, net, obs.shape[0], _ptr(obs), _ptr(act), _ptr(out), self.stream))
        return out

    def q_target(self, double_q, rew, obs_tp1):
        out = self.empty(obs_tp1.shape[0])
        self._check(self.lib.mpg_q_target(self.h, int(bool(double_q)), obs_tp1.shape[0], _ptr(rew), _ptr(obs_tp1),
                                          _ptr(out), self.stream))
        return out

    def q_bootstrap(self, base, coef, obs):
        """base + coef * Q1_target(sigma obs, pi_target(sigma obs)) (mpg_learner.py:153-169)."""
        out = self.empty(obs.shape[0])
        self._check(self.lib.mpg_q_bootstrap(self.h, obs.shape[0], _ptr(base), float(coef), _ptr(obs), _ptr(out), self.stream))
        return out

    def env_step(self, state, action):
        """One step of the real PathTracking env (handle created with env_id 'PathTracking-v0-real')."""
        rows = state.shape[0]
        s1, o1, r = self.empty(rows, self.state_dim), self.empty(rows, self.obs_dim), self.empty(rows)
        done = torch.empty(rows, dtype=torch.int32, device=self.device)
        self._check(self.lib.mpg_env_step(self.h, rows, _ptr(state), _ptr(action), _ptr(s1), _ptr(o1), _ptr(r),
                                          ctypes.c_void_p(done.data_ptr()), self.stream))
        return s1, o1, r, done

    def td_error(self, obs, act, rew, obs_tp1):
        out = self.empty(obs.shape[0])
        self._check(self.lib.mpg_td_error(self.h, obs.shape[0], _ptr(obs), _ptr(act), _ptr(rew), _ptr(obs_tp1),
                                          _ptr(out), self.stream))
        return out

    def clip_global_norm(self, grad, clip):
        """In place; returns the pre-clip norm as a 1-element tensor."""
        norm = self.empty(1)
        self._check(self.lib.mpg_clip_global_norm(self.h, _ptr(grad), grad.numel(), float(clip), _ptr(norm), self.stream))
        return norm

    # ------------------------------------------------------------------ single model step
    def env_sample(self, state, obs, reset_obs, explore_noise=None, explore_sigma=0.0, policy_net=_lib.NET_POLICY, steps=None):
        """Fused sampler (mpg_env_sample): reset_obs (steps, agents, obs_dim) or None (nobody restarts; give `steps`);
        state / obs are updated in place.  Returns (obs, act, rew, obs_tp1, done), each with steps * agents rows."""
        agents = state.shape[0]
        steps = reset_obs.shape[0] if reset_obs is not None else int(steps)
        n = steps * agents
        out = [self.empty(n, self.obs_dim), self.empty(n, self.act_dim), self.empty(n), self.empty(n, self.obs_dim), self.empty(n)]
        self._check(self.lib.mpg_env_sample(self.h, policy_net, agents, steps, float(explore_sigma),
                                            _ptr(explore_noise) if explore_noise is not None else None,
                                            _ptr(reset_obs) if reset_obs is not None else None,
                                            _ptr(state), _ptr(obs), *[_ptr(t) for t in out], self.stream))
        return out

    def model_reset(self, obs):
        state = self.empty(obs.shape[0], self.state_dim)
        self._check(self.lib.mpg_model_reset(self.h, obs.shape[0], _ptr(obs), _ptr(state), self.stream))
        return state

    def model_step(self, state, action, eps=None):
        rows = state.shape[0]
        s1, o1, r = self.empty(rows, self.state_dim), self.empty(rows, self.obs_dim), self.empty(rows)
        self._check(self.lib.mpg_model_step(self.h, rows, _ptr(state), _ptr(action), _ptr(eps), _ptr(s1), _ptr(o1),
                                            _ptr(r), self.stream))
        return s1, o1, r

    def model_step_bwd(self, state, action, eps, g_obs, g_rew, g_state):
        rows = state.shape[0]
        gs, ga = self.empty(rows, self.state_dim), self.empty(rows, self.act_dim)
        self._check(self.lib.mpg_model_step_bwd(self.h, rows, _ptr(state), _ptr(action), _ptr(eps), _ptr(g_obs),
                                                _ptr(g_rew), _ptr(g_state), _ptr(gs), _ptr(ga), self.stream))
        return gs, ga

    def compute_rewards(self, state, scaled_action=None):
        out = self.empty(state.shape[0])
        self._check(self.lib.mpg_compute_rewards(self.h, state.shape[0], _ptr(state), _ptr(scaled_action), _ptr(out),
                                                 self.stream))
        return out
