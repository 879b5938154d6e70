"""Trainer (trainer.py:18-80) for the single-process topology: one worker, one replay buffer, one learner and one
evaluator on one GPU, sharing ONE PolicyWithQs so that no weight ever crosses the host.
    python -m mpg_b200.trainer --alg MPG-v2 --iters 2000 [--hidden 64|128|256] [--activation elu|relu|tanh]"""
import argparse
import json
import logging

from .buffer import PrioritizedReplayBuffer, ReplayBuffer
from .config import default_args
from .evaluator import Evaluator
from .learners import MPGLearner, NADPLearner
from .optimizer import SingleProcessOffPolicyOptimizer
from .policy import PolicyWithQs
from .worker import OffPolicyWorker

NAME2LEARNERCLS = dict([('MPG', MPGLearner), ('NADP', NADPLearner)])
NAME2BUFFERCLS = dict([('normal', ReplayBuffer), ('priority', PrioritizedReplayBuffer)])


class Trainer(object):
    def __init__(self, args, share_policy=True):
        self.args = args
        self.worker = OffPolicyWorker(PolicyWithQs, args.env_id, args, 0)
        shared = self.worker.policy_with_value if share_policy else None
        self.learner = NAME2LEARNERCLS[args.alg_name](PolicyWithQs, args) if not share_policy else \
            self._learner_with_policy(NAME2LEARNERCLS[args.alg_name], args, shared)
        self.buffer = NAME2BUFFERCLS[args.buffer_type](args, 0)
        self.evaluator = Evaluator(PolicyWithQs, args.env_id, args, policy=shared)
        self.optimizer = SingleProcessOffPolicyOptimizer(self.worker, self.learner, self.buffer, self.evaluator, args)

    @staticmethod
    def _learner_with_policy(cls, args, policy):
        learner = cls(lambda **kw: policy, args)   # the learner's policy_cls(**vars(args)) returns the shared object
        return learner

    def train(self, iters=None):
        iters = self.args.max_iter if iters is None else iters
        while self.optimizer.iteration < iters:
            self.optimizer.step()
        self.optimizer.stop()
        return self.optimizer.eval_history


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--alg', default='MPG-v2')
    ap.add_argument('--iters', type=int, default=2000)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--hidden', type=int, default=256, help='hidden units of the policy and Q nets: 64, 128 or 256')
    ap.add_argument('--activation', default='elu', choices=('elu', 'relu', 'tanh'),
                    help='hidden activation of the policy and Q nets')
    ap.add_argument('--log_dir', default=None)
    o = ap.parse_args()
    logging.basicConfig(level=logging.INFO)
    args = default_args(o.alg, 'PathTracking-v0', replay_batch_size=o.batch, batch_size=512, num_agent=8, explore_sigma=0.1,
                        max_buffer_size=500000, replay_starts=3000, buffer_log_interval=10 ** 9, num_eval_agent=64,
                        num_eval_episode=1, fixed_steps=100, eval_interval=max(o.iters // 10, 1), log_interval=100,
                        max_iter=o.iters, log_dir=o.log_dir, value_num_hidden_units=o.hidden,
                        policy_num_hidden_units=o.hidden, value_hidden_activation=o.activation,
                        policy_hidden_activation=o.activation)
    import time
    trainer = Trainer(args)
    t0 = time.perf_counter()
    hist = trainer.train(o.iters)
    wall = time.perf_counter() - t0
    for it, m in hist:
        print(json.dumps(dict(iteration=it, **m)))
    st = trainer.optimizer.get_stats()
    print(json.dumps(dict(iterations=o.iters, wall_s=wall, ms_per_iteration=1e3 * wall / max(o.iters, 1),
                          sampling_ms=1e3 * st['sampling_time'], replay_ms=1e3 * st['replay_time'],
                          learning_ms=1e3 * st['learning_time'], grad_apply_ms=1e3 * st['grad_apply_timer'],
                          eval_ms=1e3 * trainer.evaluator.get_stats()['eval_time'])))


if __name__ == '__main__':
    main()
