#!/usr/bin/env python3
"""Throughput of the policy forward+backward rollout (mpg_policy_grad) for the BASELINE.json configs that
are parity-test cases rather than bench lines: env x learner mode x batch sweep, both kernel backends.
Prints one JSON line per case (device time by CUDA events, 3 warm-ups, median of 5).
    python tools/sweep.py > profiles/rNN_sweep.jsonl
--hidden H (64, 128, 256; default 256) sets the width of the policy and Q nets; the lines of H != 256 carry `hidden`
and `flop_per_state_step`.  The algorithmic FLOP per state-step at that width (SURVEY.md 8(a)) is printed to stderr.
--activation (elu, relu, tanh; default elu) sets the hidden activation of the policy and Q nets; the lines of a
non-default activation carry `activation`.
--env / --mode / --rows / --backend restrict the sweep to the matching cases."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpg_b200 import synthetic  # noqa: E402
from mpg_b200.config import default_args  # noqa: E402
from mpg_b200.policy import PolicyWithQs  # noqa: E402

N = 25


def flop_per_state_step(mode, H, d_o, d_a, n=N):
    """SURVEY.md 8(a) algorithmic work of one policy-gradient update per state-step (row x horizon step).
    nadp: full BPTT, (n+1) F_pi fwd + n 2F_pi bwd + (2F_pi - 2 d_o H) at t=0 + 3 F_Q;
    mpg: default MPG, (n+1) F_pi + n F_pi + (2F_pi - 2 d_o H) + 4 F_Q."""
    f_pi = 2 * (d_o * H + H * H + H * 2 * d_a)
    f_q = 2 * ((d_o + d_a) * H + H * H + H)
    if mode == 'nadp':
        total = (n + 1) * f_pi + n * 2 * f_pi + (2 * f_pi - 2 * d_o * H) + 3 * f_q
    else:
        total = (n + 1) * f_pi + n * f_pi + (2 * f_pi - 2 * d_o * H) + 4 * f_q
    return total / n


def run(env_id, mode, B, backend, H=256, act='elu'):
    args = default_args('NADP' if mode == 'nadp' else 'MPG-v2', env_id, replay_batch_size=B,
                        value_num_hidden_units=H, policy_num_hidden_units=H,
                        value_hidden_activation=act, policy_hidden_activation=act)
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(synthetic.make_policy_with_qs_weights(1, args.obs_dim, args.act_dim, H, double_q=(mode != 'nadp')))
    e = pol.engine
    if backend == 'tc':
        if not e.tc_available():
            return None
        e.set_backend(1)
    else:
        e.set_backend(0)   # the handle defaults to the tensor-core backend wherever it covers the configuration
    obs = e.dev(synthetic.make_obs(np.random.default_rng(2), env_id, B))
    lst, w, full = ([0, N], [0.0, 1.0], True) if mode == 'nadp' else ([0, N], [0.42, 0.58], False)
    ts = []
    for i in range(8):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e.policy_grad(obs, lst, w, full_bptt=full, use_philox=True, noise_seed=3, want_returns=False)
        b.record()
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(a.elapsed_time(b))
    ms = float(np.median(ts))
    r = dict(env=env_id, mode=mode, rows=B, backend=backend, ms=ms, state_steps_per_s=B * N / (ms * 1e-3))
    if H != 256:
        r.update(hidden=H, flop_per_state_step=flop_per_state_step(mode, H, args.obs_dim, args.act_dim))
    if act != 'elu':
        r.update(activation=act)
    return r


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--hidden', type=int, default=256, choices=(64, 128, 256))
    ap.add_argument('--activation', default='elu', choices=('elu', 'relu', 'tanh'))
    ap.add_argument('--env', default=None)
    ap.add_argument('--mode', default=None, choices=('nadp', 'mpg'))
    ap.add_argument('--rows', type=int, default=None)
    ap.add_argument('--backend', default=None, choices=('ffma', 'tc'))
    o = ap.parse_args()
    for env in ('PathTracking-v0', 'InvertedPendulumConti-v0', 'InvertedDoublePendulum-v2'):
        a = default_args('NADP', env)
        print(json.dumps(dict(hidden=o.hidden, env=env, flop_per_state_step={
            m: flop_per_state_step(m, o.hidden, a.obs_dim, a.act_dim) for m in ('nadp', 'mpg')})), file=sys.stderr)
    cases = [('PathTracking-v0', 'nadp', b) for b in (256, 4096, 65536, 262144)]
    cases += [('PathTracking-v0', 'mpg', b) for b in (256, 65536, 262144)]
    for env in ('InvertedPendulumConti-v0', 'InvertedDoublePendulum-v2'):
        cases += [(env, 'nadp', b) for b in (1024, 16384, 131072, 1048576)]
    cases = [c for c in cases if (o.env is None or c[0] == o.env) and (o.mode is None or c[1] == o.mode)
             and (o.rows is None or c[2] == o.rows)]
    for env, mode, B in cases:
        for backend in ('ffma', 'tc'):
            if o.backend is not None and backend != o.backend:
                continue
            if backend == 'tc' and mode == 'nadp' and B > 262144:
                continue  # full-BPTT dW2 operand store is 53 KB per row: call in <= 256K-row chunks
            if backend == 'ffma' and B > 262144:
                continue
            r = run(env, mode, B, backend, o.hidden, o.activation)
            if r:
                print(json.dumps(r), flush=True)
            torch.cuda.empty_cache()
