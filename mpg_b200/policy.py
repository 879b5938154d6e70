"""PolicyWithQs: the reference's network container (policy.py:19-241) backed by device-resident
weights inside a libmpg_b200 handle.

Kept: constructor keywords, get_weights / set_weights nested-list format
(models + target_models, each [W1,b1,W2,b2,W3,b3] with Keras (in,out) kernels, policy.py:112-121),
compute_action / compute_mode / compute_target_action / compute_Q1 / compute_Q2 / compute_Q1_target /
compute_Q2_target on RAW-scaled ("processed") observations exactly like the reference.
apply_gradients (policy.py:123-171) runs on the device-resident weights: Keras-Adam with PolynomialDecay
learning rates, delayed policy update and Polyak targets (SURVEY.md 8(f) next #2).  save_weights / load_weights
(policy.py:98-110) write one .npz per iteration: weights, target weights, Adam moments and step counters.
"""
import numpy as np
import torch

from . import _lib
from .engine import Engine
from .synthetic import make_mlp_weights


HIDDEN_WIDTHS = (64, 128, 256)   # hidden widths the fp32 (FFMA) kernels are built for; tensor cores: 256 only
HIDDEN_ACTIVATIONS = ('elu', 'relu', 'tanh')   # hidden activations both backends are built for


class PolicyWithQs(object):
    def __init__(self, obs_dim, act_dim, value_num_hidden_layers=2, value_num_hidden_units=256,
                 value_hidden_activation='elu', policy_num_hidden_layers=2, policy_num_hidden_units=256,
                 policy_hidden_activation='elu', policy_out_activation='tanh', policy_only=False, double_Q=False,
                 target=True, tau=0.005, delay_update=1, deterministic_policy=True, action_range=None, seed=0,
                 **kwargs):
        if value_num_hidden_layers != 2 or policy_num_hidden_layers != 2:
            raise NotImplementedError('the sm_100a kernels are built for 2 hidden layers (reference default)')
        if value_num_hidden_units != policy_num_hidden_units:
            raise NotImplementedError('value_num_hidden_units and policy_num_hidden_units must be equal: one hidden '
                                      'width per handle (got %r and %r)' % (value_num_hidden_units, policy_num_hidden_units))
        if policy_num_hidden_units not in HIDDEN_WIDTHS:
            raise NotImplementedError('the sm_100a kernels are built for %s hidden units (got %r)'
                                      % (' / '.join(map(str, HIDDEN_WIDTHS)), policy_num_hidden_units))
        if value_hidden_activation != policy_hidden_activation:
            raise NotImplementedError('value_hidden_activation and policy_hidden_activation must be equal: one hidden '
                                      'activation per handle (got %r and %r)' % (value_hidden_activation,
                                                                                 policy_hidden_activation))
        if policy_hidden_activation not in HIDDEN_ACTIVATIONS:
            raise NotImplementedError('the sm_100a kernels are built for the hidden activations %s (got %r)'
                                      % (' / '.join(HIDDEN_ACTIVATIONS), policy_hidden_activation))
        if not deterministic_policy:
            raise NotImplementedError('the model-based learners use deterministic_policy=True (train_script.py:273)')
        self.obs_dim, self.act_dim, self.hidden = obs_dim, act_dim, int(policy_num_hidden_units)
        self.hidden_activation = policy_hidden_activation
        self.policy_only, self.double_Q, self.target = policy_only, double_Q, target
        self.tau, self.delay_update, self.action_range = tau, delay_update, action_range
        self.deterministic_policy = True
        self.value_lr_schedule = kwargs.get('value_lr_schedule') or [8e-5, 100000, 8e-6]
        self.policy_lr_schedule = kwargs.get('policy_lr_schedule') or [3e-5, 100000, 3e-6]
        self.opt_iterations = {}   # per-optimizer step counters (keras optimizer.iterations)
        rows = int(kwargs.get('replay_batch_size', 256)) * int(kwargs.get('M', 1))
        lists = list(kwargs.get('num_rollout_list_for_policy_update') or [25]) + \
            list(kwargs.get('num_rollout_list_for_q_estimation') or [])
        self.engine = Engine(env_id=kwargs.get('env_id', 'PathTracking-v0'), obs_dim=obs_dim, act_dim=act_dim,
                             obs_scale=kwargs.get('obs_scale'), rew_scale=kwargs.get('rew_scale', 1.0),
                             rew_shift=kwargs.get('rew_shift', 0.0), gamma=kwargs.get('gamma', 0.99),
                             policy_out_activation=policy_out_activation, action_range=action_range,
                             num_future_data=kwargs.get('num_future_data', 0), hidden=self.hidden,
                             hidden_activation=self.hidden_activation, max_rows=max(rows, 64),
                             max_horizon=max(lists + [1]), device=kwargs.get('device'), debug_lib=kwargs.get('debug_lib', False))
        # slot order == get_weights() order (policy.py:72-89)
        if policy_only:
            self.model_slots, self.target_slots = [_lib.NET_POLICY], []
        elif double_Q:
            self.model_slots = [_lib.NET_Q1, _lib.NET_Q2, _lib.NET_POLICY]
            self.target_slots = [_lib.NET_Q1_TARGET, _lib.NET_Q2_TARGET, _lib.NET_POLICY_TARGET]
        else:
            self.model_slots = [_lib.NET_Q1, _lib.NET_POLICY]
            self.target_slots = [_lib.NET_Q1_TARGET, _lib.NET_POLICY_TARGET] if target else []
        rng = np.random.default_rng(seed)
        for slot in self.model_slots:
            self.engine.set_net_weights(slot, self._init(rng, slot))
        for slot, src in zip(self.target_slots, self.model_slots):
            # Q targets start as copies (policy.py:61,68); policy_target is an independent init there
            w = self.engine.get_net_weights(src) if src != _lib.NET_POLICY else self._init(rng, slot)
            self.engine.set_net_weights(slot, w)

    def _init(self, rng, slot):
        if slot in (_lib.NET_POLICY, _lib.NET_POLICY_TARGET):
            return make_mlp_weights(rng, self.obs_dim, self.hidden, 2 * self.act_dim, bias_scale=0.0)
        return make_mlp_weights(rng, self.obs_dim + self.act_dim, self.hidden, 1, bias_scale=0.0)

    # -- weights --------------------------------------------------------------------------------
    def get_weights(self):
        return [self.engine.get_net_weights(s) for s in self.model_slots + self.target_slots]

    def set_weights(self, weights):
        slots = self.model_slots + self.target_slots
        for i, w in enumerate(weights):
            self.engine.set_net_weights(slots[i], w)

    def save_weights(self, save_dir, iteration):
        """policy.py:98-103: models + target models + optimizers of one iteration -> save_dir/ckpt_ite<iteration>.npz"""
        import os
        os.makedirs(save_dir, exist_ok=True)
        blob = {}
        for s in self.model_slots + self.target_slots:
            for i, w in enumerate(self.engine.get_net_weights(s)):
                blob['net%d_w%d' % (s, i)] = w
        for s in self.model_slots:
            blob['net%d_adam_m' % s], blob['net%d_adam_v' % s] = self.engine.get_adam_state(s)
            blob['net%d_opt_iterations' % s] = np.int64(self.opt_iterations.get(s, 0))
        np.savez(os.path.join(save_dir, 'ckpt_ite%d.npz' % iteration), **blob)

    def load_weights(self, load_dir, iteration):
        """policy.py:105-110"""
        import os
        with np.load(os.path.join(load_dir, 'ckpt_ite%d.npz' % iteration)) as blob:
            for s in self.model_slots + self.target_slots:
                self.engine.set_net_weights(s, [blob['net%d_w%d' % (s, i)] for i in range(6)])
            for s in self.model_slots:
                self.engine.set_adam_state(s, blob['net%d_adam_m' % s], blob['net%d_adam_v' % s])
                self.opt_iterations[s] = int(blob['net%d_opt_iterations' % s])

    @staticmethod
    def polynomial_decay(schedule, step):
        """keras PolynomialDecay(initial, decay_steps, end), power 1, no cycle."""
        init, decay_steps, end = schedule
        frac = min(float(step), float(decay_steps)) / float(decay_steps)
        return (init - end) * (1.0 - frac) + end

    def _adam(self, slot, schedule, flat_grad):
        it = self.opt_iterations.get(slot, 0)
        self.engine.adam_step(slot, flat_grad, self.polynomial_decay(schedule, it), it + 1)
        self.opt_iterations[slot] = it + 1

    def apply_gradients(self, iteration, grads):
        """PolicyWithQs.apply_gradients (policy.py:123-156). `grads`: the list compute_gradient returns (numpy,
        Q1[,Q2],policy x [W1,b1,W2,b2,W3,b3]) or one flat device tensor in the same order (no host round trip)."""
        e = self.engine
        if isinstance(grads, torch.Tensor):
            flat = grads.to(e.device, torch.float32).contiguous()
        else:
            flat = e.dev(np.concatenate([np.asarray(g, np.float32).ravel() for g in grads]))
        q_slots = [s for s in self.model_slots if s != _lib.NET_POLICY]
        pos = 0
        for s in q_slots:                              # Q nets: every call
            n = e.param_count(s)
            self._adam(s, self.value_lr_schedule, flat[pos:pos + n])
            pos += n
        npol = e.param_count(_lib.NET_POLICY)
        if self.policy_only or iteration % self.delay_update == 0:
            self._adam(_lib.NET_POLICY, self.policy_lr_schedule, flat[pos:pos + npol])
            if self.target_slots and not self.policy_only:
                for src, dst in zip(self.model_slots, self.target_slots):   # update_*_target (policy.py:158-171)
                    e.polyak_update(src, dst, self.tau)

    # -- forward passes (policy.py:173-241) --------------------------------------------------------
    def _raw(self, processed_obs):
        # the kernels apply obs_scale themselves, so undo it on the way in: obs_raw * scale == processed
        e = self.engine
        t = e.dev(processed_obs)
        scale = torch.tensor([e.cfg.obs_scale[i] for i in range(self.obs_dim)], device=t.device)
        return (t / scale).contiguous()

    def compute_action(self, obs):
        return self.engine.policy_forward(_lib.NET_POLICY, self._raw(obs)), 0.

    def compute_mode(self, obs):
        return self.engine.policy_forward(_lib.NET_POLICY, self._raw(obs))

    def compute_target_action(self, obs):
        return self.engine.policy_forward(_lib.NET_POLICY_TARGET, self._raw(obs)), 0.

    def _q(self, slot, obs, act):
        return self.engine.q_forward(slot, self._raw(obs), self.engine.dev(act))

    def compute_Q1(self, obs, act):
        return self._q(_lib.NET_Q1, obs, act)

    def compute_Q2(self, obs, act):
        return self._q(_lib.NET_Q2, obs, act)

    def compute_Q1_target(self, obs, act):
        return self._q(_lib.NET_Q1_TARGET, obs, act)

    def compute_Q2_target(self, obs, act):
        return self._q(_lib.NET_Q2_TARGET, obs, act)
