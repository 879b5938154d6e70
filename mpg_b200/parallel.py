"""Data parallelism of the learner (SURVEY.md 8(e)): the state batch shards over ranks (contiguous row
blocks), every rank produces SUMS already scaled by 1/B_global, and ONE all-reduce (sum, fp32) of a single
flat buffer [grads of every net | scalar sums] makes all ranks hold the global-batch gradient; the per-net
global-norm clip and the statistics are then computed redundantly on every rank.

Plumbing only (torch.distributed: NCCL over NVLink on GPUs, gloo in the CPU tests) -- no arithmetic of
the hot path lives here."""
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
