#!/usr/bin/env python3
"""Scaling of the data-parallel trainer over the GPUs of one box: `torchrun --nproc_per_node N -m mpg_b200.trainer`
with MPG-v2 at --rows rows per rank (weak scaling: one update learns from N x rows rows), for N = 1 / 2 / 4 / 8 (those
the box has).  One JSON line per N, appended to --out:
    iterations_per_s             iterations over the wall clock of train() (sampling, learning, apply, evaluation)
    state_steps_per_s            N x rows x 25 model state-steps of the policy rollout per iteration, over that clock
    learner_state_steps_per_s    the same state-steps over the learner section alone (compute_gradient incl. all-reduce)
    sampling_ms_per_iteration    worker sampling (every 10th iteration) per iteration
    allreduce_ms_per_iteration   the gradient all-reduce per iteration (device time, 0 on one rank)
with the card's name and power limit read in the same run.  bench.py --gpus N measures the learner's kernels alone.
    python tools/train_scaling.py [--gpus 1,2,4,8] [--rows 65536] [--iters 1000] [--out profiles/r6_train_scaling.jsonl]"""
import argparse
import json
import os
import socket
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HORIZON = 25   # the longest rollout of MPG-v2's default list [0, 25]


def card():
    """name and power limit of GPU 0: part of every number measured on it"""
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader,nounits', '-i', '0'],
                         capture_output=True, text=True, timeout=60, check=True).stdout
    name, limit = [x.strip() for x in out.strip().split(',')]
    return dict(gpu=name, power_limit_w=float(limit))


def run(n, rows, iters):
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={n}', '--master-addr=127.0.0.1',
           f'--master-port={port}', '-m', 'mpg_b200.trainer', '--alg', 'MPG-v2', '--batch', str(rows), '--iters', str(iters)]
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    if p.returncode != 0:
        raise RuntimeError(f'{n} GPUs: exit code {p.returncode}\n{p.stderr[-4000:]}')
    summary = [json.loads(x) for x in p.stdout.splitlines() if x.startswith('{') and '"wall_s"' in x][-1]
    its = iters / summary['wall_s']
    steps = summary['global_batch'] * HORIZON
    return dict(alg='MPG-v2', gpus=n, rows_per_rank=rows, global_batch=summary['global_batch'], iterations=iters,
                iterations_per_s=its, state_steps_per_s=steps * its,
                learner_state_steps_per_s=steps / (summary['learning_ms'] * 1e-3),
                ms_per_iteration=summary['ms_per_iteration'], learning_ms=summary['learning_ms'],
                sampling_ms_per_iteration=summary['sampling_ms_per_iteration'],
                allreduce_ms_per_iteration=summary['allreduce_ms_per_iteration'],
                grad_apply_ms=summary['grad_apply_ms'], eval_ms=summary['eval_ms'])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', default='1,2,4,8')
    ap.add_argument('--rows', type=int, default=65536)
    ap.add_argument('--iters', type=int, default=1000)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r6_train_scaling.jsonl'))
    o = ap.parse_args()
    have = torch.cuda.device_count()
    if have == 0:
        raise SystemExit('no CUDA device')
    info = card()
    lines = []
    for n in [int(x) for x in o.gpus.split(',')]:
        if n > have:
            print(f'skipping {n} GPUs: the box has {have}', file=sys.stderr)
            continue
        line = dict(run(n, o.rows, o.iters), **info)
        lines.append(line)
        print(json.dumps(line), flush=True)
    base = next((x for x in lines if x['gpus'] == 1), None)
    with open(o.out, 'a') as f:
        for line in lines:
            if base is not None:
                line['weak_scaling_efficiency'] = line['iterations_per_s'] / base['iterations_per_s']
            f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
