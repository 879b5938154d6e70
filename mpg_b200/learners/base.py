"""Shared host logic of the model-based learners: batch intake, sharded data parallelism, the
flat gradient buffer, clipping, conversion back to the reference's list-of-numpy format."""
import numpy as np
import torch

from ..engine import Engine  # noqa: F401  (documentation of the dependency)
from .. import parallel
from ..preprocessor import Preprocessor
from ..utils.misc import CudaTimerStat


def rule_based_weights(ite, total_ite, eta, rollout_list):
    """MPGLearner.rule_based_weights (mpg_learner.py:384-399), evaluated in float32 like the TF graph.
    Host-side: a handful of scalars per update, not device work."""
    f = np.float32
    lam = f(1. - eta) + f(2. * eta / total_ite) * f(ite)
    lam = f(min(max(lam, f(0.)), f(1.5)))
    if lam < 1.:
        biases = np.array([np.power(lam, f(i), dtype=f) for i in rollout_list], dtype=f)
    else:
        mx = max(rollout_list)
        biases = np.array([np.power(f(2.) - lam, f(mx - i), dtype=f) for i in rollout_list], dtype=f)
    inv = f(1.) / (biases + f(1e-8))
    e = np.exp(inv - inv.max(), dtype=f)
    return (e / e.sum(dtype=f)).astype(f)


class _LazyDev(dict):
    """Device copies of the batch; a key whose upload was deferred is uploaded on first access."""

    def __init__(self, owner):
        super().__init__()
        self._owner = owner

    def __missing__(self, k):
        self._owner._finish_upload(consumer_waits=True)
        return dict.__getitem__(self, k)


class LearnerBase(object):
    """What MPGLearner and NADPLearner share (mpg_learner.py:30-64,171-178; nadp.py:29-53,78-85)."""

    def __init__(self, policy_cls, args):
        self.args = args
        self.batch_size = self.args.replay_batch_size
        self.policy_with_value = policy_cls(**vars(self.args))
        self.engine = self.policy_with_value.engine
        self.batch_data = {}
        self.counter = 0
        self.num_batch_reuse = self.args.num_batch_reuse
        self.M = self.args.M
        self.num_rollout_list_for_policy_update = list(self.args.num_rollout_list_for_policy_update)
        self.num_rollout_list_for_q_estimation = list(self.args.num_rollout_list_for_q_estimation or [])
        self.preprocessor = Preprocessor(self.args.obs_dim, self.args.obs_ptype, self.args.rew_ptype,
                                         self.args.obs_scale, self.args.rew_scale, self.args.rew_shift,
                                         gamma=self.args.gamma)
        # device time of each section (CUDA events), read after the update's single D2H copy
        self.policy_gradient_timer = CudaTimerStat()
        self.q_gradient_timer = CudaTimerStat()
        self.target_timer = CudaTimerStat()
        self.stats = {}
        self.info_for_buffer = {}
        # noise of the model rollout: None -> in-kernel Philox keyed by (seed, global row, step);
        # tests install explicit eps tensors with set_rollout_noise
        self.noise_seed = int(getattr(self.args, 'noise_seed', 7))
        self._noise_q = self._noise_p = None
        self._dev, self._pinned, self.h2d_bytes = {}, {}, 0
        self._pending, self._copy_stream, self._copy_pending = [], None, False
        # data parallel: each rank holds a contiguous shard of the global batch (SURVEY.md 8(e))
        self.world_size, self.rank = parallel.dist_info()

    # -- reference interface ------------------------------------------------------------------------
    def get_stats(self):
        return self.stats

    def get_info_for_buffer(self):
        return self.info_for_buffer

    def get_weights(self):
        return self.policy_with_value.get_weights()

    def set_weights(self, weights):
        return self.policy_with_value.set_weights(weights)

    def set_ppc_params(self, params):
        self.preprocessor.set_params(params)

    # -- helpers ------------------------------------------------------------------------------------
    def set_rollout_noise(self, noise_q=None, noise_p=None):
        """Explicit standard-normal eps, shape (n, M*B), for the Q-target / policy rollouts."""
        self._noise_q = None if noise_q is None else self.engine.dev(noise_q)
        self._noise_p = None if noise_p is None else self.engine.dev(noise_p)

    def _upload_batch(self, batch_data):
        # mpg_learner.py:66-72: cast to fp32; here additionally host -> device (pinned when possible)
        names = ('batch_obs', 'batch_actions', 'batch_rewards', 'batch_obs_tp1', 'batch_dones')
        if isinstance(batch_data[0], torch.Tensor):
            # device-resident replay (mpg_b200.buffer.*.replay_device): no host round trip
            self.batch_data = {k: v for k, v in zip(names, batch_data)}
            self._dev = {k: self.engine.dev(v) for k, v in self.batch_data.items() if k != 'batch_dones'}
            self.h2d_bytes = 0
            self._pending = []
            return
        self.batch_data = {k: np.asarray(v, dtype=np.float32) for k, v in zip(names, batch_data)}   # mpg_learner.py:66-72
        # obs and actions feed the first kernels: staged and enqueued now.  rewards / obs_tp1 are needed later (targets,
        # TD errors) or not at all (NADP with a uniform buffer): their staging copy and H2D transfer run on a side
        # stream while the GPU is already busy -- on first use, at the latest before compute_gradient returns.
        self._dev = _LazyDev(self)
        self._pending = [k for k in ('batch_rewards', 'batch_obs_tp1')]
        for k in ('batch_obs', 'batch_actions'):
            self._dev[k] = self._stage(k).to(self.engine.device, non_blocking=True)
        self.h2d_bytes = sum(v.size * 4 for k, v in self.batch_data.items() if k != 'batch_dones')   # batch_dones: ignored (mpg_learner.py:71)

    def _stage(self, k):
        v = self.batch_data[k]
        pin = self._pinned.get(k)
        if pin is None or pin.shape != v.shape:
            pin = self._pinned[k] = torch.empty(v.shape, dtype=torch.float32, pin_memory=True)
        pin.copy_(torch.from_numpy(v))      # multi-threaded for MB-sized batches (a numpy slice assignment is one thread)
        return pin

    def _finish_upload(self, consumer_waits=True):
        """Upload what _upload_batch deferred.  consumer_waits: the current stream is about to read the tensors."""
        pending = getattr(self, '_pending', None)
        if pending:
            self._pending = []
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=self.engine.device)
            with torch.cuda.stream(self._copy_stream):
                for k in pending:
                    dict.__setitem__(self._dev, k, self._stage(k).to(self.engine.device, non_blocking=True))
            self._copy_pending = True
        if consumer_waits and getattr(self, '_copy_pending', False):
            torch.cuda.current_stream(self.engine.device).wait_stream(self._copy_stream)
            for k in ('batch_rewards', 'batch_obs_tp1'):
                self._dev[k].record_stream(torch.cuda.current_stream(self.engine.device))
            self._copy_pending = False

    @property
    def global_rows(self):
        return parallel.shard_rows(self._dev['batch_obs'].shape[0], self.world_size, self.rank)[0]

    @property
    def row_offset(self):
        return parallel.shard_rows(self._dev['batch_obs'].shape[0], self.world_size, self.rank)[1]

    def _allreduce(self, flat):
        return parallel.allreduce_flat(flat, self.world_size)

    def _to_host(self, dev):
        """The update's single device -> host copy: into a pinned staging buffer (a pageable destination makes the
        driver bounce the copy through its own staging area), then one stream synchronise.  Returns a fresh numpy
        array -- the caller hands views of it out as the gradient list."""
        n = dev.numel()
        pin = self._pinned.get('_d2h')
        if pin is None or pin.numel() < n:
            pin = self._pinned['_d2h'] = torch.empty(n, dtype=torch.float32, pin_memory=True)
        pin[:n].copy_(dev, non_blocking=True)
        torch.cuda.current_stream(self.engine.device).synchronize()
        return pin[:n].numpy().copy()

    def _split_to_numpy(self, flat_host, nets):
        return parallel.split_flat(flat_host, self.args.obs_dim, self.args.act_dim, nets, self.engine.cfg.hidden,
                                   self.engine.hidden_layers)
