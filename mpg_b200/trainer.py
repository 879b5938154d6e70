"""Trainer (trainer.py:18-80) for the single-process topology: one worker, one replay buffer, one learner and one
evaluator on one GPU, sharing ONE PolicyWithQs so that no weight ever crosses the host.
    python -m mpg_b200.trainer --alg MPG-v2 --iters 2000 [--hidden 64|128|256] [--activation elu|relu|tanh]
    [--layers 1|2|3] [--rollout_list 1-25 | 0,25 | ...]

Data parallel over the GPUs of one box, one synchronous rank per GPU:
    torchrun --nproc_per_node N -m mpg_b200.trainer --alg MPG-v2 ...
Every rank runs its own worker (env seed and exploration noise keyed by the rank) and its own replay buffer, and
draws --batch rows from it per iteration, so one update learns from N x batch rows.  Rank 0's weights are broadcast
once at the start; after that every rank applies the same all-reduced gradient.  The evaluator, the logs, the
checkpoints and the printed summary are rank 0's."""
import argparse
import json
import logging
import os

import torch

from . import parallel
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
    """Under a process group: this rank's share of a data-parallel run (see the module docstring)."""

    def __init__(self, args, share_policy=True):
        self.args = args
        self.world_size, self.rank = parallel.dist_info()
        self.worker = OffPolicyWorker(PolicyWithQs, args.env_id, args, self.rank)
        shared = self.worker.policy_with_value if share_policy else None
        self.learner = NAME2LEARNERCLS[args.alg_name](PolicyWithQs, args) if not share_policy else \
            self._learner_with_policy(NAME2LEARNERCLS[args.alg_name], args, shared)
        self.buffer = NAME2BUFFERCLS[args.buffer_type](args, self.rank)
        self.evaluator = Evaluator(PolicyWithQs, args.env_id, args, policy=shared) if self.rank == 0 else None
        if self.world_size > 1:
            parallel.broadcast_weights(self.worker.policy_with_value)   # before the replay fill samples with them
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


def parse_rollout_list(text):
    """'1-25' -> [1, .., 25]; '0,5,10-12' -> [0, 5, 10, 11, 12]"""
    out = []
    for part in text.split(','):
        lo, _, hi = part.strip().partition('-')
        out += list(range(int(lo), int(hi) + 1)) if hi else [int(lo)]
    return out


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description='Train on the PathTracking environment; under torchrun --nproc_per_node N, '
                                             'one synchronous data-parallel rank per GPU.')
    ap.add_argument('--alg', default='MPG-v2')
    ap.add_argument('--iters', type=int, default=2000)
    ap.add_argument('--batch', type=int, default=256,
                    help='replay rows each rank draws per iteration: one update learns from N x batch rows on N GPUs')
    ap.add_argument('--hidden', type=int, default=256, help='hidden units of the policy and Q nets: 64, 128 or 256')
    ap.add_argument('--activation', default='elu', choices=('elu', 'relu', 'tanh'),
                    help='hidden activation of the policy and Q nets')
    ap.add_argument('--layers', type=int, default=2, choices=(1, 2, 3), help='hidden layers of the policy and Q nets')
    ap.add_argument('--rollout_list', default=None, type=parse_rollout_list,
                    help='num_rollout_list_for_policy_update of MPG: comma-separated steps and ranges a-b, e.g. 1-25; '
                         'up to 64 entries counting the step 0 MPG adds (default: the reference list)')
    ap.add_argument('--log_dir', default=None)
    return ap.parse_args(argv)


def trainer_args(o):
    """The learner / worker / buffer / evaluator arguments of a command line parsed by parse_args."""
    return default_args(o.alg, 'PathTracking-v0', replay_batch_size=o.batch, batch_size=512, num_agent=8, explore_sigma=0.1,
                        max_buffer_size=500000, replay_starts=3000, buffer_log_interval=10 ** 9, num_eval_agent=64,
                        num_eval_episode=1, fixed_steps=100, eval_interval=max(o.iters // 10, 1), log_interval=100,
                        max_iter=o.iters, log_dir=o.log_dir, value_num_hidden_units=o.hidden,
                        policy_num_hidden_units=o.hidden, value_hidden_activation=o.activation,
                        policy_hidden_activation=o.activation, value_num_hidden_layers=o.layers,
                        policy_num_hidden_layers=o.layers,
                        **({} if o.rollout_list is None else dict(num_rollout_list_for_policy_update=o.rollout_list)))


def run(o):
    import time
    trainer = Trainer(trainer_args(o))
    t0 = time.perf_counter()
    hist = trainer.train(o.iters)
    wall = time.perf_counter() - t0
    if trainer.rank != 0:
        return
    for it, m in hist:
        print(json.dumps(dict(iteration=it, **m)))
    st = trainer.optimizer.get_stats()
    n = max(o.iters, 1)
    print(json.dumps(dict(iterations=o.iters, wall_s=wall, ms_per_iteration=1e3 * wall / n,
                          sampling_ms=1e3 * st['sampling_time'], replay_ms=1e3 * st['replay_time'],
                          learning_ms=1e3 * st['learning_time'], grad_apply_ms=1e3 * st['grad_apply_timer'],
                          eval_ms=1e3 * trainer.evaluator.get_stats()['eval_time'],
                          world_size=trainer.world_size, global_batch=o.batch * trainer.world_size,
                          sampling_ms_per_iteration=1e3 * trainer.optimizer.timers['sampling_timer'].total / n,
                          allreduce_ms_per_iteration=1e3 * trainer.learner.allreduce_timer.total / n)))


def main():
    o = parse_args()
    logging.basicConfig(level=logging.INFO)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world == 1:
        run(o)
        return
    local_rank = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local_rank)
    torch.distributed.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    try:
        run(o)
    finally:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
