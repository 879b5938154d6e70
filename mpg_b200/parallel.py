"""Data parallelism of the learner (SURVEY.md 8(e)): the state batch shards over ranks (contiguous row
blocks), every rank produces SUMS already scaled by 1/B_global, and ONE all-reduce (sum, fp32) of a single
flat buffer [grads of every net | scalar sums] makes all ranks hold the global-batch gradient; the per-net
global-norm clip and the statistics are then computed redundantly on every rank.

The data-parallel trainer keeps one replica of every net per rank: rank 0's weights are broadcast once at the
start (broadcast_weights), after which every rank applies the same all-reduced gradient, and check_replicas
compares a checksum of every rank's weights.

Plumbing only (torch.distributed: NCCL over NVLink on GPUs, gloo in the CPU tests) -- no arithmetic of
the hot path lives here."""
import hashlib

import numpy as np
import torch

from .engine import mlp_shapes


def dist_info():
    """(world_size, rank) of the default process group, (1, 0) when not initialised."""
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        return torch.distributed.get_world_size(), torch.distributed.get_rank()
    return 1, 0


def shard_rows(local_rows, world_size, rank):
    """Contiguous sharding with equal shards: -> (global_rows, row_offset of this rank)."""
    return local_rows * world_size, local_rows * rank


def allreduce_flat(flat, world_size):
    """In-place sum over ranks of the flat fp32 buffer (no-op for a single rank)."""
    if world_size > 1:
        torch.distributed.all_reduce(flat, op=torch.distributed.ReduceOp.SUM)
    return flat


def _collective_device():
    """Where tensors of a collective live: the current GPU under NCCL, the host under gloo."""
    if torch.distributed.get_backend() == 'nccl':
        return torch.device('cuda', torch.cuda.current_device())
    return torch.device('cpu')


def broadcast_weights(policy, src=0):
    """Overwrite every rank's nets (get_weights order: models, then targets) with those of rank `src`: one flat
    fp32 broadcast.  The replicas start equal whatever seed each rank's nets were initialised with."""
    nets = policy.get_weights()
    flat = torch.from_numpy(np.concatenate([np.asarray(w, np.float32).ravel() for net in nets for w in net]))
    flat = flat.to(_collective_device())
    torch.distributed.broadcast(flat, src=src)
    flat, pos, out = flat.cpu().numpy(), 0, []
    for net in nets:
        out.append([])
        for w in net:
            out[-1].append(flat[pos:pos + w.size].reshape(w.shape))
            pos += w.size
    policy.set_weights(out)


def weights_checksum(nets):
    """SHA-256 of the bytes of every weight array (get_weights order) -> 4 int64 words."""
    h = hashlib.sha256()
    for net in nets:
        for w in net:
            h.update(np.ascontiguousarray(w, np.float32).tobytes())
    return torch.from_numpy(np.frombuffer(h.digest(), dtype=np.int64).copy())


def check_replicas(policy, iteration):
    """Fault detector of the data-parallel trainer: every rank all-gathers the checksum of every rank's weights and
    raises if any differ.  Every rank sees the same gathered checksums, so every rank raises together and none is
    left waiting in a later collective."""
    world_size, rank = dist_info()
    if world_size == 1:
        return
    mine = weights_checksum(policy.get_weights()).to(_collective_device())
    every = [torch.empty_like(mine) for _ in range(world_size)]
    torch.distributed.all_gather(every, mine)
    every = [t.cpu() for t in every]
    differ = [r for r in range(world_size) if not torch.equal(every[r], every[0])]
    if differ:
        raise RuntimeError(f'replica weights diverged at iteration {iteration}: ranks {differ} differ from rank 0 '
                           f'(seen on rank {rank})')


def net_shapes(obs_dim, act_dim, kind, hidden=256, layers=2):
    """Shapes of one net's [W1,b1,..,WL,bL,Wout,bout] (Keras (in,out) kernels, L = layers); kind 'q' or 'pi'."""
    in_dim = obs_dim + (act_dim if kind == 'q' else 0)
    out_dim = 1 if kind == 'q' else 2 * act_dim
    return mlp_shapes(in_dim, hidden, out_dim, layers)


def split_flat(flat_host, obs_dim, act_dim, nets, hidden=256, layers=2):
    """flat fp32 host vector (concatenated nets) -> list of arrays in the reference's gradient-list order."""
    out, pos = [], 0
    for kind in nets:
        for shape in net_shapes(obs_dim, act_dim, kind, hidden, layers):
            n = int(np.prod(shape))
            out.append(flat_host[pos:pos + n].reshape(shape))
            pos += n
    assert pos == flat_host.size, (pos, flat_host.size)
    return out
