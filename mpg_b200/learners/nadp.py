"""NADPLearner with the reference's interface (learners/nadp.py:22-241); arithmetic in libmpg_b200.

compute_gradient(batch_data, rb, indexes, iteration) -> list of 12 numpy arrays
(Q1 [W1,b1,W2,b2,W3,b3] + policy [...]), each net clipped by global norm, like nadp.py:209-241.
"""
import numpy as np
import torch

from .. import _lib
from .base import LearnerBase


class NADPLearner(LearnerBase):
    def __init__(self, policy_cls, args):
        super().__init__(policy_cls, args)
        if len(self.num_rollout_list_for_q_estimation) != 1:
            raise ValueError('NADP regresses Q1 on ONE n-step target per sample (nadp.py:120-126 concatenates the '
                             'selected returns, which only matches q_pred for a single rollout length)')

    def get_batch_data(self, batch_data, rb, indexes):
        self._upload_batch(batch_data)
        if self.args.buffer_type != 'normal':
            self.info_for_buffer.update(dict(td_error=self.compute_td_error(), rb=rb, indexes=indexes))

    def compute_td_error(self):  # nadp.py:67-76
        d = self._dev
        td = self.engine.td_error(d['batch_obs'], d['batch_actions'], d['batch_rewards'], d['batch_obs_tp1'])
        return td if isinstance(self.batch_data['batch_obs'], torch.Tensor) else td.cpu().numpy()

    def model_rollout_for_q_estimation(self, mb_obs, mb_actions):
        """nadp.py:87-126: forward-only rollout from the replay (obs, action) with the online policy and
        the Q1_target bootstrap; returns the (stop-gradient) targets as a device tensor (B,)."""
        e = self.engine
        lst = self.num_rollout_list_for_q_estimation
        ret = e.rollout_forward(mb_obs, lst, M=self.M, q_net=_lib.NET_Q1_TARGET, start_actions=mb_actions,
                                noise=self._noise_q, use_philox=self._noise_q is None, noise_seed=self.noise_seed,
                                global_rows=self.global_rows, row_offset=self.row_offset)
        return e.returns_tile_mean(ret, mb_obs.shape[0], self.M).reshape(-1)

    def q_forward_and_backward(self, mb_obs, mb_actions):  # nadp.py:173-184
        targets = self.model_rollout_for_q_estimation(mb_obs, mb_actions)
        grad, loss_sum = self.engine.q_grad(_lib.NET_Q1, mb_obs, mb_actions, targets, global_rows=self.global_rows)
        return loss_sum, grad

    def policy_forward_and_backward(self, mb_obs):  # nadp.py:186-194
        e = self.engine
        k = self.num_rollout_list_for_policy_update[0]
        lst, w = ([0], [1.0]) if k == 0 else ([0, k], [0.0, 1.0])  # R_0 only feeds the value_mean statistic
        n = max(self.num_rollout_list_for_policy_update)
        if n not in lst:
            lst, w = lst + [n], w + [0.0]
        grad, ret = e.policy_grad(mb_obs, lst, w, M=self.M, full_bptt=True, q_net=_lib.NET_Q1,
                                  noise=self._noise_p, use_philox=self._noise_p is None,
                                  noise_seed=self.noise_seed + 1, global_rows=self.global_rows,
                                  row_offset=self.row_offset)
        sums = e.returns_stats(ret, mb_obs.shape[0], self.M)  # [sum R_k ..., sum R_k^2 ...]
        return grad, sums, lst.index(k)

    def compute_gradient(self, batch_data, rb, indexes, iteration):
        if self.counter % self.num_batch_reuse == 0:
            self.get_batch_data(batch_data, rb, indexes)
        self.counter += 1
        if self.args.buffer_type != 'normal':
            self.info_for_buffer.update(dict(td_error=self.compute_td_error()))
        mb_obs, mb_actions = self._dev['batch_obs'], self._dev['batch_actions']
        e, clip = self.engine, self.args.gradient_clip_norm

        with self.q_gradient_timer:
            q_loss_sum, q_grad = self.q_forward_and_backward(mb_obs, mb_actions)
        with self.policy_gradient_timer:
            p_grad, sums, kpos = self.policy_forward_and_backward(mb_obs)

        # one flat buffer: [q grad | policy grad | scalar sums]  ->  one all-reduce  ->  clip per net
        nq = q_grad.numel()
        flat = torch.cat([q_grad, p_grad, q_loss_sum, sums])
        self._allreduce(flat)
        q_norm = e.clip_global_norm(flat[:nq], clip)
        p_norm = e.clip_global_norm(flat[nq:nq + p_grad.numel()], clip)
        self._finish_upload()                                     # deferred H2D (rewards / obs_tp1) has overlapped the kernels
        host = self._to_host(torch.cat([flat, q_norm, p_norm]))   # the only device->host copy of the update
        ng = nq + p_grad.numel()
        B = float(self.global_rows)
        n_list = (host.size - ng - 3) // 2
        ret_sums = host[ng + 1: ng + 1 + n_list]
        self.stats.update(dict(
            iteration=iteration,
            q_timer=self.q_gradient_timer.mean,
            pg_time=self.policy_gradient_timer.mean,
            q_loss=np.float32(host[ng] / B),
            policy_loss=np.float32(-ret_sums[kpos] / B),
            value_mean=np.float32(ret_sums[0] / B),
            q_gradient_norm=np.float32(host[-2]),
            policy_gradient_norm=np.float32(host[-1]),
            num_rollout_list_for_policy=self.num_rollout_list_for_policy_update,
            num_rollout_list_for_q=self.num_rollout_list_for_q_estimation,
        ))
        if self.world_size > 1:
            self.stats.update(allreduce_time=self.allreduce_timer.mean)
        self.flat_grad_device = flat[:ng]     # the same clipped gradients, still on the device (apply_gradients takes it)
        return self._split_to_numpy(host[:ng], ['q', 'pi'])
