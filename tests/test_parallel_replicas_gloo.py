"""CPU, world_size 2, gloo: the replica plumbing of the data-parallel trainer.  broadcast_weights makes every rank
hold rank 0's nets whatever each rank was initialised with, and check_replicas passes on equal replicas and raises
on EVERY rank (not only the odd one out, which would leave the others waiting in a collective) when one weight of
one rank differs in its last bit."""
import os
import socket
import sys

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Nets(object):
    """get_weights / set_weights of PolicyWithQs: a list of nets, each a list of arrays."""

    def __init__(self, seed):
        rng = np.random.default_rng(seed)
        self.nets = [[rng.standard_normal(s).astype(np.float32) for s in ((7, 5), (5,), (5, 1), (1,))] for _ in range(3)]

    def get_weights(self):
        return [[w.copy() for w in net] for net in self.nets]

    def set_weights(self, weights):
        self.nets = [[np.array(w, np.float32) for w in net] for net in weights]


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from mpg_b200 import parallel
        nets = _Nets(seed=100 + rank)
        parallel.broadcast_weights(nets)
        ref = _Nets(seed=100).nets
        same = all(np.array_equal(a, b) for na, nb in zip(nets.nets, ref) for a, b in zip(na, nb))
        parallel.check_replicas(nets, 0)
        if rank == 1:
            w = nets.get_weights()
            w[2][0][3, 1] = np.nextafter(w[2][0][3, 1], np.float32(np.inf))
            nets.set_weights(w)
        try:
            parallel.check_replicas(nets, 7)
            raised = ''
        except RuntimeError as e:
            raised = str(e)
        with open(os.path.join(out_dir, f'rank{rank}.txt'), 'w') as f:
            f.write(f'{int(same)}\n{raised}')
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def test_broadcast_and_replica_guard_world2(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        same, raised = open(tmp_path / f'rank{r}.txt').read().split('\n', 1)
        assert same == '1', r
        assert 'diverged at iteration 7' in raised and 'ranks [1]' in raised, (r, raised)
