"""SingleProcessOffPolicyOptimizer with the reference's interface (optimizer.py:286-397): the synchronous
sample -> replay -> learn -> apply loop.  The asynchronous Ray variant (optimizer.py:127-280) is replaced by
synchronous data parallelism inside the learner (one NCCL all-reduce of the flat gradient).

Under a process group every rank runs this loop on its own worker and replay buffer.  Every branch of step() is
taken alike on every rank (the NaN check looks at the all-reduced gradient), so the replicas stay identical;
the optimizer.jsonl log and the checkpoints are rank 0's, and the replicas are compared at every evaluation
iteration and in stop()."""
import json
import logging
import os

import numpy as np

from . import parallel
from .utils.misc import TimerStat

logger = logging.getLogger(__name__)


class SingleProcessOffPolicyOptimizer(object):
    def __init__(self, worker, learner, replay_buffer, evaluator, args):
        self.args, self.worker, self.learner, self.replay_buffer, self.evaluator = args, worker, learner, replay_buffer, evaluator
        self.num_sampled_steps = self.iteration = 0
        self.timers = {k: TimerStat() for k in ['sampling_timer', 'replay_timer', 'learning_timer', 'grad_apply_timer']}
        self.stats, self.eval_history = {}, []
        self.log_dir = getattr(args, 'log_dir', None)
        self.shared = getattr(learner, 'policy_with_value', None) is getattr(worker, 'policy_with_value', object())
        self.world_size, self.rank = parallel.dist_info()
        logger.info('start filling the replay')
        while not len(self.replay_buffer) >= self.args.replay_starts:
            self._sample()
        logger.info('end filling the replay')
        self.get_stats()

    def _sample(self):
        batch = self.worker.sample_arrays()
        # every rank samples as many steps on the same schedule: the count over all ranks
        self.num_sampled_steps += batch[0].shape[0] * self.world_size
        self.replay_buffer.add_arrays(*batch)

    def get_stats(self):
        self.stats.update(dict(num_sampled_steps=self.num_sampled_steps, iteration=self.iteration,
                               sampling_time=self.timers['sampling_timer'].mean, replay_time=self.timers['replay_timer'].mean,
                               learning_time=self.timers['learning_timer'].mean,
                               grad_apply_timer=self.timers['grad_apply_timer'].mean))
        return self.stats

    def step(self):
        if self.iteration % 10 == 0:                                   # sampling_interval (optimizer.py:334-339)
            with self.timers['sampling_timer']:
                self._sample()
        with self.timers['replay_timer']:
            samples = self.replay_buffer.replay_device()
        with self.timers['learning_timer']:
            if not self.shared:
                self.learner.set_weights(self.worker.get_weights())
            grads = self.learner.compute_gradient(samples[:5], self.replay_buffer, samples[-1], self.iteration)
            learner_stats = self.learner.get_stats()
            if self.args.buffer_type == 'priority':
                info = self.learner.get_info_for_buffer()
                info['rb'].update_priorities(info['indexes'], info['td_error'])
        with self.timers['grad_apply_timer']:
            if not all(np.isfinite(g).all() for g in grads):            # judge_is_nan -> zero the gradient (optimizer.py:357-361)
                grads = [np.zeros_like(g) for g in grads]
                if getattr(self.learner, 'flat_grad_device', None) is not None:
                    self.learner.flat_grad_device = None
                logger.info('Grad is nan!, zero it')
            # one shared PolicyWithQs: hand over the flat device gradient, no host -> device copy of what just came back
            dev_grads = getattr(self.learner, 'flat_grad_device', None) if self.shared else None
            self.worker.apply_gradients(self.iteration, grads if dev_grads is None else dev_grads)
        if self.log_dir and self.rank == 0 and self.iteration % getattr(self.args, 'log_interval', 100) == 0:
            os.makedirs(self.log_dir, exist_ok=True)
            rec = {k: (v if not isinstance(v, (list, np.ndarray)) else [float(x) for x in v]) for k, v in learner_stats.items()}
            rec = {k: (float(v) if isinstance(v, (np.floating, np.integer)) else v) for k, v in rec.items()}
            with open(os.path.join(self.log_dir, 'optimizer.jsonl'), 'a') as f:
                f.write(json.dumps(dict(rec, **self.get_stats())) + '\n')
        if self.world_size > 1 and self.iteration % self.args.eval_interval == 0:
            parallel.check_replicas(self.worker.policy_with_value, self.iteration)
        if self.evaluator is not None and self.iteration % self.args.eval_interval == 0:
            if not getattr(self.evaluator, 'policy_with_value', None) is self.worker.policy_with_value:
                self.evaluator.set_weights(self.worker.get_weights())
            self.eval_history.append((self.iteration, self.evaluator.run_evaluation(self.iteration)))
        model_dir = getattr(self.args, 'model_dir', None)
        if model_dir and self.rank == 0 and self.iteration % getattr(self.args, 'save_interval', 3000) == 0:   # optimizer.py:389-391
            self.worker.save_weights(model_dir, self.iteration)
            self.worker.save_ppc_params(model_dir)
        self.get_stats()
        self.iteration += 1

    def stop(self):
        parallel.check_replicas(self.worker.policy_with_value, self.iteration)
