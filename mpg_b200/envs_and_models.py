"""Environment models with the reference's API (envs_and_models/__init__.py:13-15):
    model = NAME2MODELCLS[env_id](**vars(args)); model.reset(obses); obses, rewards = model.rollout_out(actions)
on torch CUDA tensors, stateful between calls and differentiable (torch.autograd.Function around the
single-step kernel and its hand-derived adjoint).  The learners do not go through this class: they
call the fused n-step kernels (mpg_policy_grad / mpg_rollout_forward) on the same device functions.

Noise: the reference draws tfd.Normal(0.5, 0.01) / Normal(0.1, 0.5) samples inside f_xu
(path_tracking_env.py:119, inverted_pendulum_model.py:61).  Here the standard-normal eps comes from
`set_noise(eps_iterable)` (tests), else from torch.randn on the model's generator.
"""
import torch

from .engine import Engine
from .synthetic import ENV_DIMS


class _StepFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, state, action, eps):
        state, action = state.contiguous(), action.contiguous()
        s1, o1, r = engine.model_step(state, action, eps)
        ctx.engine, ctx.eps = engine, eps
        ctx.save_for_backward(state, action)
        return s1, o1, r

    @staticmethod
    def backward(ctx, g_s1, g_o1, g_r):
        state, action = ctx.saved_tensors
        z = lambda g, ref: None if g is None else g.contiguous()
        gs, ga = ctx.engine.model_step_bwd(state, action, ctx.eps, z(g_o1, None), z(g_r, None), z(g_s1, None))
        return None, gs, ga, None


class _RewardHolder(object):
    """model.vehicle_dynamics.compute_rewards(states, actions) / model.dynamics.compute_rewards(states)."""

    def __init__(self, engine, needs_action):
        self.engine, self.needs_action = engine, needs_action

    def compute_rewards(self, states, actions=None):
        e = self.engine
        return e.compute_rewards(e.dev(states), e.dev(actions) if self.needs_action else None)


class _ModelBase(object):
    env_id = None

    def __init__(self, num_future_data=0, **kwargs):
        obs_dim, act_dim, _ = ENV_DIMS[self.env_id]
        nfd = num_future_data if self.env_id == 'PathTracking-v0' else 0
        self.num_future_data = nfd
        self.engine = Engine(env_id=self.env_id, obs_dim=obs_dim + nfd, act_dim=act_dim, obs_scale=None,
                             rew_scale=1.0, rew_shift=0.0, gamma=1.0, num_future_data=nfd,
                             max_rows=64, max_horizon=0, device=kwargs.get('device'))
        self.obses = self.actions = self.states = None
        self._noise = None
        self.generator = torch.Generator(device=self.engine.device)
        self.generator.manual_seed(int(kwargs.get('seed', 0)))
        self.noisy = self.env_id != 'InvertedDoublePendulum-v2'

    def set_noise(self, eps_iterable):
        self._noise = iter(eps_iterable) if eps_iterable is not None else None

    def reset(self, obses):
        self.obses = self.engine.dev(obses)
        self.actions = None
        self.states = self.engine.model_reset(self.obses.detach())
        if self.obses.requires_grad:  # reset is linear in obs for PathTracking / cart-pole: keep the graph
            self.states = self._state_from_obs(self.obses)

    def _state_from_obs(self, o):
        if self.env_id == 'PathTracking-v0':
            shift = torch.zeros(6, device=o.device)
            shift[0] = 20.0
            return o[:, :6] + shift
        if self.env_id == 'InvertedPendulumConti-v0':
            return o
        return torch.stack([o[:, 0], torch.atan2(o[:, 1], o[:, 3]), torch.atan2(o[:, 2], o[:, 4]),
                            o[:, 5], o[:, 6], o[:, 7]], 1)

    def rollout_out(self, actions):
        actions = self.engine.dev(actions) if not isinstance(actions, torch.Tensor) else actions.to(self.engine.device)
        eps = None
        if self.noisy:
            if self._noise is not None:
                eps = self.engine.dev(next(self._noise))
            else:
                eps = torch.randn(actions.shape[0], device=self.engine.device, generator=self.generator)
        self.actions = actions
        self.states, self.obses, rewards = _StepFn.apply(self.engine, self.states, actions, eps)
        return self.obses, rewards


class PathTrackingModel(_ModelBase):
    env_id = 'PathTracking-v0'

    def __init__(self, num_future_data=0, **kwargs):
        super().__init__(num_future_data=num_future_data, **kwargs)
        self.vehicle_dynamics = _RewardHolder(self.engine, True)
        self.base_frequency, self.expected_vs = 10., 20.

    @property
    def veh_states(self):
        return self.states


class InvertedPendulumModel(_ModelBase):
    env_id = 'InvertedPendulumConti-v0'

    def __init__(self, **kwargs):
        super().__init__(**kwargs)
        self.dynamics = _RewardHolder(self.engine, False)
        self.tau = 0.04


class InvertedDoublePendulumModel(_ModelBase):
    env_id = 'InvertedDoublePendulum-v2'

    def __init__(self, **kwargs):
        super().__init__(**kwargs)
        self.dynamics = _RewardHolder(self.engine, False)
        self.tau = 0.01


class PathTrackingEnv(object):
    """The REAL PathTracking environment (path_tracking_env.py:356-487) batched on the GPU: reset(init_obs=obs) and
    step(action) -> (obs, reward, done, info) with the reference's 200 Hz x 20 sub-step simulation, reference-path
    projection and judge_done.  Used by the MPG-v1 n-step targets (through the fused rollout) and available to
    workers / evaluators.  Random resets (`reset()` without init_obs) draw the pose from the reset law in
    mpg_b200.synthetic and observe it as the environment does, future columns against the reference path included."""

    def __init__(self, num_future_data=0, num_agent=1, **kwargs):
        self.num_future_data, self.num_agent = num_future_data, num_agent
        self.engine = Engine(env_id='PathTracking-v0-real', obs_dim=6 + num_future_data, act_dim=2, obs_scale=None,
                             rew_scale=1.0, rew_shift=0.0, gamma=1.0, num_future_data=num_future_data, max_rows=64,
                             max_horizon=0, device=kwargs.get('device'))
        self.obs = self.state = self.done = self.action = None
        self._rng = __import__('numpy').random.default_rng(int(kwargs.get('seed', 0)))
        self._gen = None

    def reset(self, **kwargs):
        if 'init_obs' in kwargs:
            self.obs = self.engine.dev(kwargs['init_obs'])
        else:
            from .synthetic import make_obs
            base = self.engine.dev(make_obs(self._rng, 'PathTracking-v0', self.num_agent))
            # the future columns of the drawn pose, as the environment's own observation of it (not copies of delta_y)
            fut = self._future_columns(base[:, 0] + 20.0, base[:, 3], base[:, 5])
            self.obs = torch.stack([base[:, i] for i in range(6)] + fut, 1).contiguous()
        self.state = self.engine.model_reset(self.obs)
        return self.obs

    def _future_columns(self, vx, dy, x):
        """The future columns of _get_obs (path_tracking_env.py:384-402) at a reset pose: delta_y of the pose against the
        reference path at x + k * v_x / 200 * 20 * 2, k = 1..num_future_data; at reset y = delta_y + path_y(x)."""
        import math
        path_y = lambda xs: (7.5 * torch.sin(xs * 2.0 * math.pi / 200.0) + 2.5 * torch.sin(xs * 2.0 * math.pi / 300.0)
                             - 5.0 * torch.sin(xs * 2.0 * math.pi / 400.0))
        y, xf, cols = dy + path_y(x), x.clone(), []
        for _ in range(self.num_future_data):
            xf = xf + vx * 1.0 / 200.0 * 20.0 * 2.0
            cols.append(y - path_y(xf))
        return cols

    def step(self, action):
        self.action = self.engine.dev(action)
        self.state, self.obs, reward, self.done = self.engine.env_step(self.state, self.action)
        return self.obs, reward, self.done, {}

    def _draw_on_device(self, sets=1):
        """`sets` x num_agent observations from the reset law of path_tracking_env.py:426-437, drawn with a device
        generator (no host round trip): x ~ U(0,600), dy ~ N(0,1), dphi ~ N(0,pi/9), v_x ~ U(15,25), beta ~ N(0,0.15),
        v_y = v_x tan(beta), r ~ N(0,0.3)."""
        import math
        import torch
        if self._gen is None:
            self._gen = torch.Generator(device=self.engine.device)
            self._gen.manual_seed(int(self._rng.integers(1 << 31)))
        n, g, dev = self.num_agent * sets, self._gen, self.engine.device
        u = torch.rand(2, n, device=dev, generator=g)
        z = torch.randn(4, n, device=dev, generator=g)
        vx = 15.0 + 10.0 * u[1]
        dy = z[0]
        x = 600.0 * u[0]
        cols = [vx - 20.0, vx * torch.tan(0.15 * z[2]), 0.3 * z[3], dy, (math.pi / 9) * z[1], x]
        return torch.stack(cols + self._future_columns(vx, dy, x), 1).contiguous()

    def reset_done(self, fresh=None):
        """reset() of the reference without init_obs (path_tracking_env.py:422-454): agents whose `done` flag is set
        are re-drawn from the reset law (or take the rows of `fresh`), the others keep their state.  Everything stays
        on the device."""
        import torch
        if self.done is None:
            return self.reset()
        if fresh is None:
            fresh = self._draw_on_device()
        fresh_state = self.engine.model_reset(fresh)
        m = (self.done != 0).unsqueeze(1)
        self.state = torch.where(m, fresh_state, self.state)
        self.obs = torch.where(m, fresh, self.obs)
        return self.obs


NAME2MODELCLS = dict([('PathTracking-v0', PathTrackingModel),
                      ('InvertedDoublePendulum-v2', InvertedDoublePendulumModel),
                      ('InvertedPendulumConti-v0', InvertedPendulumModel)])
