"""MPGLearner with the reference's interface (learners/mpg_learner.py:23-455); arithmetic in libmpg_b200.

compute_gradient(batch_data, rb, indexes, iteration) -> list of numpy arrays
q_gradient1 [+ q_gradient2] + policy_gradient, each net clipped by global norm (mpg_learner.py:401-455).
"""
import numpy as np
import torch

from .. import _lib
from .base import LearnerBase, rule_based_weights


class MPGLearner(LearnerBase):
    def __init__(self, policy_cls, args):
        lst = list(args.num_rollout_list_for_policy_update)
        n_run = len(lst) + (0 not in lst)   # policy_forward_and_backward adds step 0
        if n_run > _lib.MAX_LIST_LONG:
            raise ValueError(f'num_rollout_list_for_policy_update has {len(lst)} entries ({n_run} with the step 0 every '
                             f'update adds for value_mean); at most {_lib.MAX_LIST_LONG} are supported')
        super().__init__(policy_cls, args)
        self.sample_num_in_learner = self.args.sample_num_in_learner
        n = len(self.num_rollout_list_for_policy_update)
        self.ws_old = np.array([0.] + [1. / (n - 1)] * (n - 1), dtype=np.float32) if n > 1 else np.ones(1, np.float32)
        if self.args.learner_version not in ('MPG-v1', 'MPG-v2'):
            raise ValueError(self.args.learner_version)

    # -- batch intake (mpg_learner.py:66-85) ----------------------------------------------------------
    def get_batch_data(self, batch_data, rb, indexes):
        self._upload_batch(batch_data)
        with self.target_timer:
            if self.args.learner_version == 'MPG-v1':
                target = self.compute_n_step_target()
            elif self.args.learner_version == 'MPG-v2':
                target = self.compute_clipped_double_q_target()
            else:
                raise ValueError
        self._dev['batch_targets'] = target
        self.batch_data.update(dict(batch_targets=target))
        if self.args.buffer_type != 'normal':
            self.info_for_buffer.update(dict(td_error=self.compute_td_error(), rb=rb, indexes=indexes))

    def compute_clipped_double_q_target(self):  # mpg_learner.py:126-134
        return self.engine.q_target(True, self._dev['batch_rewards'], self._dev['batch_obs_tp1'])

    def compute_n_step_target(self):  # mpg_learner.py:146-169
        d = self._dev
        if self.sample_num_in_learner is None:
            return self.engine.q_target(False, d['batch_rewards'], d['batch_obs_tp1'])
        # MPG-v1: sample_num_in_learner steps of the REAL environment from the replay (obs, action) with the online
        # policy (sample(), mpg_learner.py:87-124), then the Q1_target / policy_target bootstrap on the last obs
        if self.args.env_id != 'PathTracking-v0':
            raise NotImplementedError('the real-env n-step sampler is built for PathTracking-v0; the pendulum ground truth '
                                      'is a mujoco simulation (inverted_pendulum_conti.py) that is not part of this build')
        T = int(self.sample_num_in_learner)
        ret, t_obs, _, _ = self.engine.rollout_forward(d['batch_obs'], [T], q_net=-1, start_actions=d['batch_actions'],
                                                      want_traj=True, real_env=True)
        return self.engine.q_bootstrap(ret[0].contiguous(), float(self.args.gamma) ** T, t_obs[T - 1].contiguous())

    def compute_td_error(self):  # mpg_learner.py:136-144
        d = self._dev
        td = self.engine.td_error(d['batch_obs'], d['batch_actions'], d['batch_rewards'], d['batch_obs_tp1'])
        return td if isinstance(self.batch_data['batch_obs'], torch.Tensor) else td.cpu().numpy()

    def rule_based_weights(self, ite, total_ite, eta):
        return rule_based_weights(ite, total_ite, eta, self.num_rollout_list_for_policy_update)

    # -- gradients ----------------------------------------------------------------------------------
    def q_forward_and_backward(self, mb_obs, mb_actions, mb_targets):  # mpg_learner.py:326-354
        nets = [_lib.NET_Q1] + ([_lib.NET_Q2] if self.args.learner_version == 'MPG-v2' else [])
        return [self.engine.q_grad(n, mb_obs, mb_actions, mb_targets, global_rows=self.global_rows) for n in nets]

    def policy_forward_and_backward(self, mb_obs, ite):  # mpg_learner.py:356-365 + 226-286
        e = self.engine
        lst = list(self.num_rollout_list_for_policy_update)
        ws = self.rule_based_weights(ite, self.args.rule_based_bias_total_ite, self.args.eta)
        klist, kw = lst, [float(w) for w in ws]
        if 0 not in klist:  # value_mean = mean Q1(p_0, a_0) is a statistic of every update (mpg_learner.py:285)
            klist, kw = [0] + klist, [0.0] + kw
        grad, ret = e.policy_grad(mb_obs, klist, kw, M=self.M, full_bptt=bool(self.args.deriv_interval_policy),
                                  q_net=_lib.NET_Q1, noise=self._noise_p, use_philox=self._noise_p is None,
                                  noise_seed=self.noise_seed + 1, global_rows=self.global_rows,
                                  row_offset=self.row_offset)
        sums = e.returns_stats(ret, mb_obs.shape[0], self.M)
        return grad, sums, ws, klist

    def compute_gradient(self, batch_data, rb, indexes, iteration):
        if self.counter % self.num_batch_reuse == 0:
            self.get_batch_data(batch_data, rb, indexes)
        self.counter += 1
        if self.args.buffer_type != 'normal':
            self.info_for_buffer.update(dict(td_error=self.compute_td_error()))
        d = self._dev
        e, clip = self.engine, self.args.gradient_clip_norm
        v2 = self.args.learner_version == 'MPG-v2'

        with self.q_gradient_timer:
            q_res = self.q_forward_and_backward(d['batch_obs'], d['batch_actions'], d['batch_targets'])
        with self.policy_gradient_timer:
            p_grad, sums, ws, klist = self.policy_forward_and_backward(d['batch_obs'], iteration)
            self.ws_old = ws

        flat = torch.cat([g for g, _ in q_res] + [p_grad] + [l for _, l in q_res] + [sums])
        self._allreduce(flat)
        nq = q_res[0][0].numel()
        norms, pos = [], 0
        for n in [nq] * len(q_res) + [p_grad.numel()]:
            norms.append(e.clip_global_norm(flat[pos:pos + n], clip))
            pos += n
        ng = pos
        self._finish_upload()
        host = self._to_host(torch.cat([flat] + norms))
        B = float(self.global_rows)
        nql = len(q_res)
        n_list = len(klist)
        ret_sums = host[ng + nql: ng + nql + n_list]
        ret_sq = host[ng + nql + n_list: ng + nql + 2 * n_list]
        lst = self.num_rollout_list_for_policy_update
        all_losses = np.array([-ret_sums[klist.index(k)] / B for k in lst], dtype=np.float32)
        norm_vals = host[-(nql + 1):]
        self.stats.update(dict(
            iteration=iteration,
            q_timer=self.q_gradient_timer.mean,
            pg_time=self.policy_gradient_timer.mean,
            target_time=self.target_timer.mean,
            value_mean=np.float32(ret_sums[klist.index(0)] / B),
            policy_total_loss=np.float32(np.sum(ws * all_losses)),
            policy_gradient_norm=np.float32(norm_vals[-1]),
            q_loss1=np.float32(host[ng] / B),
            q_gradient_norm1=np.float32(norm_vals[0]),
            num_rollout_list=self.num_rollout_list_for_policy_update,
            w_list_new=list(ws),
            w_list=list(ws),
            all_losses=list(all_losses),
            returns_var=[float(ret_sq[klist.index(k)] / B - (ret_sums[klist.index(k)] / B) ** 2) for k in lst],
        ))
        if self.world_size > 1:
            self.stats.update(allreduce_time=self.allreduce_timer.mean)
        if v2:
            self.stats.update(dict(q_loss2=np.float32(host[ng + 1] / B), q_gradient_norm2=np.float32(norm_vals[1])))
        self.flat_grad_device = flat[:ng]     # the same clipped gradients, still on the device (apply_gradients takes it)
        return self._split_to_numpy(host[:ng], ['q'] * nql + ['pi'])
