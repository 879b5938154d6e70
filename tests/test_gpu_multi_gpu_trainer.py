"""The data-parallel trainer on two GPUs of one box: one rank per GPU over NCCL, each with its own worker and replay
buffer, one all-reduced gradient per update.  Checked: the replicas stay bit-identical (uniform and prioritized
replay), one update equals the single-process update on the concatenated batch, each rank samples and prioritizes
its own rows, only rank 0 writes logs / evaluations / checkpoints, the replica guard raises on every rank, a
one-rank run is the single-process trainer, and a short 2-rank run learns.

With two or more GPUs the ranks run one per GPU over NCCL, as under torchrun.  On a box with one GPU both ranks share
it and talk over gloo: the trainer, learner and replica code under test is the same, only the transport differs."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORLD = 2

pytestmark = pytest.mark.gpu
BACKEND = 'nccl' if torch.cuda.device_count() >= WORLD else 'gloo'
TIMER_STATS = ('q_timer', 'pg_time', 'target_time', 'allreduce_time', 'iteration')


def _args(alg, **kw):
    from mpg_b200.config import default_args
    base = dict(replay_batch_size=256, batch_size=512, num_agent=8, explore_sigma=0.1, max_buffer_size=100000,
                replay_starts=2048, buffer_log_interval=10 ** 9, num_eval_agent=64, num_eval_episode=1, fixed_steps=60,
                eval_interval=10 ** 9, log_interval=10 ** 9, max_iter=400, log_dir=None,
                policy_lr_schedule=[3e-4, 100000, 3e-5], value_lr_schedule=[8e-4, 100000, 8e-5])
    base.update(kw)
    return default_args(alg, 'PathTracking-v0', **base)


def _flat(nets):
    return np.concatenate([np.asarray(w, np.float32).ravel() for net in nets for w in net])


def _gather(t):
    """all_gather -> list of per-rank tensors on t's device (through the host under gloo)"""
    src = t.contiguous() if BACKEND == 'nccl' else t.cpu()
    every = [torch.empty_like(src) for _ in range(dist.get_world_size())]
    dist.all_gather(every, src)
    return [x.to(t.device) for x in every]


def _replicas_identical(tr):
    every = _gather(torch.from_numpy(_flat(tr.worker.get_weights())).cuda())
    return all(torch.equal(x, every[0]) for x in every)


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ---- what each rank runs ------------------------------------------------------------------------------------------
def _steps(rank, out, alg, buffer_type, iters):
    """`iters` optimizer steps with per-rank init seeds and per-rank output directories."""
    from mpg_b200.trainer import Trainer
    d = os.path.join(out, f'rank{rank}')
    args = _args(alg, buffer_type=buffer_type, seed=rank, replay_batch_size=128, replay_starts=1024, max_buffer_size=20000,
                 fixed_steps=20, log_dir=os.path.join(d, 'log'), model_dir=os.path.join(d, 'model'), log_interval=5,
                 eval_interval=10, save_interval=10)
    tr = Trainer(args)
    identical = [_replicas_identical(tr)]           # after the start broadcast
    cap = {}
    if buffer_type == 'priority':
        compute_gradient = tr.learner.compute_gradient

        def capture(batch, rb, indexes, iteration):   # TD errors of this rank's rows under the weights of the update
            cap['td'] = tr.learner.engine.td_error(*batch[:4]).clone()
            cap['idx'] = indexes.clone()
            return compute_gradient(batch, rb, indexes, iteration)
        tr.learner.compute_gradient = capture
    for _ in range(iters):
        tr.optimizer.step()
        identical.append(_replicas_identical(tr))
    tr.optimizer.stop()
    res = dict(identical=identical, num_sample=tr.worker.num_sample)
    # replay contents: the same uniforms draw different transitions on each rank
    u = torch.linspace(0.0005, 0.9995, 512, device='cuda')
    obs = _gather(tr.buffer.dev.sample(512, u)[0])
    res['replay_same_as_rank0'] = bool(torch.equal(obs[rank], obs[0]))
    if buffer_type == 'priority':
        # leaf priority of every drawn index from its importance weight: w = (p / p_min)^-beta
        _, p_min, _ = tr.buffer.dev.tree_stats()
        beta, alpha = args.replay_beta, args.replay_alpha
        _, _, _, _, _, w, idx = tr.buffer.dev.sample(65536)
        leaf = p_min * w.double().cpu().numpy() ** (-1.0 / beta)
        want = np.full(len(tr.buffer), np.nan)
        td = cap['td'].cpu().numpy()
        want[cap['idx'].cpu().numpy()] = (np.abs(td) + np.float32(1e-6)).astype(np.float32).astype(np.float64) ** alpha
        hit = ~np.isnan(want[idx.cpu().numpy()])
        res['priority_rel_err'] = float(np.max(np.abs(leaf[hit] / want[idx.cpu().numpy()][hit] - 1.0)))
        res['priority_checked'] = int(hit.sum())
    res['files'] = sorted(os.path.relpath(os.path.join(r, f), d) for r, _, fs in os.walk(d) for f in fs)
    log = os.path.join(d, 'log', 'optimizer.jsonl')
    if os.path.exists(log):
        res['logged_num_sampled_steps'] = json.loads(open(log).read().splitlines()[-1])['num_sampled_steps']
    return res


def _one_update(rank, out, alg):
    """One optimizer step; then, on rank 0 outside the group, one single-process update on the concatenated batch."""
    import copy
    from mpg_b200.policy import PolicyWithQs
    from mpg_b200.trainer import NAME2LEARNERCLS, Trainer
    args = _args(alg, seed=rank, replay_batch_size=256)
    tr = Trainer(args)
    start = tr.worker.get_weights()
    cap = {}
    replay_device, compute_gradient = tr.buffer.replay_device, tr.learner.compute_gradient

    def capture_batch(*a, **k):
        s = replay_device(*a, **k)
        cap['batch'] = [t.clone() for t in s[:5]]
        return s

    def capture_grads(*a):
        g = compute_gradient(*a)
        cap['grads'] = np.concatenate([x.ravel() for x in g])
        return g
    tr.buffer.replay_device, tr.learner.compute_gradient = capture_batch, capture_grads
    tr.optimizer.step()
    stats = {k: v for k, v in tr.learner.get_stats().items() if k not in TIMER_STATS}
    after = _flat(tr.worker.get_weights())
    identical = _replicas_identical(tr)
    batch = [torch.cat(_gather(t)) for t in cap['batch']]      # rank order == global row order
    dist.destroy_process_group()
    if rank != 0:
        return dict(identical=identical)
    from mpg_b200 import parallel
    assert parallel.dist_info() == (1, 0)
    sargs = copy.copy(args)
    sargs.replay_batch_size = args.replay_batch_size * WORLD
    single = NAME2LEARNERCLS[args.alg_name](PolicyWithQs, sargs)
    single.set_weights(start)
    g = np.concatenate([x.ravel() for x in single.compute_gradient(batch, None, None, 0)])
    ref = single.get_stats()
    stat_err = {}
    for k, v in stats.items():
        if isinstance(v, (list, np.ndarray, float, np.floating)) and not isinstance(v, str):
            a, b = np.asarray(v, np.float64), np.asarray(ref[k], np.float64)
            if k == 'returns_var':     # E[R^2] - E[R]^2: the error is relative to E[R^2]
                scale = b + np.asarray(ref['all_losses'], np.float64) ** 2
            else:
                scale = np.maximum(np.abs(b), 1e-12)
            stat_err[k] = float(np.max(np.abs(a - b) / scale))
    single.policy_with_value.apply_gradients(0, single.flat_grad_device)
    return dict(identical=identical, grad_rel_l2=_rel(cap['grads'], g), stat_err=stat_err,
                weight_rel_l2=_rel(after, _flat(single.get_weights())), weights_moved=_rel(after, _flat(start)))


def _guard(rank, out):
    from mpg_b200.trainer import Trainer
    tr = Trainer(_args('MPG-v2', replay_batch_size=64, replay_starts=1024, eval_interval=2))
    tr.train(2)                                     # the guard passes at iteration 0 and in stop()
    if rank == 1:
        w = tr.worker.get_weights()
        w[1][0] = np.array(w[1][0])
        w[1][0][0, 0] = np.nextafter(w[1][0][0, 0], np.float32(np.inf))
        tr.worker.set_weights(w)
    try:
        tr.train(4)
        return dict(raised='')
    except RuntimeError as e:
        return dict(raised=str(e))


def _learn(rank, out):
    from mpg_b200.trainer import Trainer
    args = _args('MPG-v2')
    tr = Trainer(args)
    before = tr.evaluator.run_evaluation(0) if rank == 0 else None
    tr.train(args.max_iter)
    after = tr.evaluator.run_evaluation(args.max_iter) if rank == 0 else None
    return dict(before=before, after=after, has_evaluator=tr.evaluator is not None)


SCENARIOS = dict(steps=_steps, one_update=_one_update, guard=_guard, learn=_learn)


def _rank_main(rank, port, out, scenario, kw):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    if BACKEND == 'nccl':
        torch.cuda.set_device(rank)
        dist.init_process_group('nccl', rank=rank, world_size=WORLD, device_id=torch.device('cuda', rank))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group('gloo', rank=rank, world_size=WORLD)
    try:
        res = SCENARIOS[scenario](rank, out, **kw)
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()
    with open(os.path.join(out, f'result{rank}.json'), 'w') as f:
        json.dump(res, f)


def _spawn(tmp_path, scenario, **kw):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mp.spawn(_rank_main, args=(port, str(tmp_path), scenario, kw), nprocs=WORLD, join=True)
    return [json.load(open(tmp_path / f'result{r}.json')) for r in range(WORLD)]


# ---- tests --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module', params=[('MPG-v2', 'normal'), ('NADP', 'priority')], ids=['MPG-v2-normal', 'NADP-priority'])
def twenty_steps(request, tmp_path_factory):
    alg, buffer_type = request.param
    return buffer_type, _spawn(tmp_path_factory.mktemp('steps'), 'steps', alg=alg, buffer_type=buffer_type, iters=20)


def test_replicas_stay_bit_identical(twenty_steps):
    """Ranks start from different init seeds; after the broadcast and after every update the weights are equal."""
    _, res = twenty_steps
    for r in res:
        assert len(r['identical']) == 21 and all(r['identical']), r['identical']


def test_ranks_sample_their_own_replay(twenty_steps):
    buffer_type, res = twenty_steps
    assert not res[1]['replay_same_as_rank0']
    if buffer_type == 'priority':   # each rank's tree holds |TD error| + eps of the rows that rank learned from
        for r in res:
            assert r['priority_checked'] > 100 and r['priority_rel_err'] < 1e-5, r


def test_rank0_alone_writes_log_evaluations_and_checkpoints(twenty_steps):
    _, res = twenty_steps
    files = res[0]['files']
    assert 'log/optimizer.jsonl' in files and 'log/evaluator.jsonl' in files, files
    assert 'model/ckpt_ite0.npz' in files and 'model/ckpt_ite10.npz' in files, files
    assert res[1]['files'] == []
    # the log's sample count covers every rank (logged at iteration 15, after the last sampling at iteration 10)
    assert res[0]['logged_num_sampled_steps'] == sum(r['num_sample'] for r in res)


@pytest.mark.parametrize('alg', ['MPG-v2', 'NADP'])
def test_one_update_equals_single_process_update_on_concatenated_batch(tmp_path, alg):
    res = _spawn(tmp_path, 'one_update', alg=alg)
    assert all(r['identical'] for r in res)
    r = res[0]
    assert r['weights_moved'] > 0
    assert r['grad_rel_l2'] <= 1e-5, r
    assert max(r['stat_err'].values()) <= 2e-5, r['stat_err']
    assert r['weight_rel_l2'] <= 1e-5, r


def test_replica_guard_raises_on_every_rank(tmp_path):
    """One ulp of one weight on rank 1: every rank raises at the next evaluation iteration, and every rank exits
    (mp.spawn joins them all before the results are read)."""
    res = _spawn(tmp_path, 'guard')
    for r in res:
        assert 'diverged at iteration 2' in r['raised'] and 'ranks [1]' in r['raised'], r


def test_two_rank_training_improves_evaluation_return(tmp_path):
    res = _spawn(tmp_path, 'learn')
    assert res[0]['has_evaluator'] and not res[1]['has_evaluator']
    before, after = res[0]['before'], res[0]['after']
    assert after['episode_return'] > before['episode_return'], (before, after)


def test_single_rank_run_is_the_single_process_trainer():
    """`WORLD_SIZE=1` (what torchrun --nproc_per_node 1 sets) runs the single-process trainer: the same evaluation
    history, bit for bit, as Trainer(args).train() in this process."""
    from mpg_b200.trainer import Trainer, parse_args, trainer_args
    argv = ['--alg', 'MPG-v2', '--iters', '30', '--batch', '64', '--hidden', '64']
    env = dict(os.environ, WORLD_SIZE='1', RANK='0', LOCAL_RANK='0')
    p = subprocess.run([sys.executable, '-m', 'mpg_b200.trainer'] + argv, cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [json.loads(x) for x in p.stdout.splitlines() if x.startswith('{')]
    got = [x for x in lines if 'episode_return' in x]
    o = parse_args(argv)
    want = [dict(iteration=it, **m) for it, m in Trainer(trainer_args(o)).train(o.iters)]
    assert len(want) == 10 and got == want
