#!/usr/bin/env python3
"""bench.py -- model state-steps/s (fwd+bwd, n = 25) of the MPG model-based learner hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--backend auto|ffma|tc]
                    [--config 1..5] [--rows R] [--scaling weak|strong] [--global-rows G] [--mode nadp|mpg] [--env pt|ip|idp]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Default workload = BASELINE.json configs[1] (the configuration the metric is quoted on): PathTrackingModel, NADP (pure
n-step ADP gradient, full BPTT), n = 25, B = 65536 rows per GPU, H = 256, synthetic seeded states / weights, in-kernel
Philox noise; N > 1: weak scaling (65536 rows per GPU, one NCCL all-reduce of the flat gradient inside the step).
  value : rows*n*N / (device time of ONE policy forward+backward rollout, mpg_policy_grad, inputs resident in HBM)
  e2e   : the same unit through the reference-facing call <Learner>.compute_gradient(batch, rb, idx, it) with HOST numpy
          buffers: H2D of the replay batch, Q side (target rollout / targets, Q gradient), policy rollout fwd+bwd, clip,
          D2H of the gradient arrays + stats inside the timed region.  Median of three blocks of K updates.
  --impl reference : the restated reference learner (oracle, PyTorch CPU fp32 -- TensorFlow is not installable in this
          image) timed on the host cores for the same compute_gradient on the SAME rows.
The other BASELINE.json configs (parity-test cases and the config matrix of profiles/r2_configs.jsonl):
  --config 1 : PathTracking MPG-v2 learner (first-action gradient, lists [0, 25]), B = 256 (the reference's default run)
  --config 3 : --env ip|idp, NADP n-step rollout at --rows R in [2^10, 2^20]
  --config 4 : PathTracking MPG-v2, 1,048,576 states sharded over N GPUs (strong scaling) + NCCL gradient all-reduce
  --config 5 : PathTracking MPG-v2 + prioritized replay at B = 262,144: sum-tree sample -> compute_gradient ->
               update_priorities on the device, reported as updates/s (e2e) next to the policy-gradient value
One JSON line is printed by rank 0.
--dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned, so that two builds can be
          compared output for output on the same seeded inputs:
            DIR/policy_grad.npy       flat policy gradient of the last device step (fp32; all-reduced when N > 1)
            DIR/compute_gradient.npy  the arrays of the last e2e compute_gradient, flattened and concatenated in the
                                      order it returns them (clipped [Q1 | Q2 | policy]; --impl reference: the oracle's)
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line: everything else that writes to fd 1 (NCCL's version banner, library chatter)
# is sent to stderr; the JSON line goes to a private duplicate of the original stdout.
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_JSON_FD, (json.dumps(line) + '\n').encode())


from mpg_b200 import synthetic  # noqa: E402
from mpg_b200.config import default_args  # noqa: E402

N_STEPS, ROWS_PER_GPU, HID = 25, 65536, 256
ENVS = {'pt': 'PathTracking-v0', 'ip': 'InvertedPendulumConti-v0', 'idp': 'InvertedDoublePendulum-v2'}


def flop_per_state_step(env_id, full_bptt):
    """Algorithmic FLOP per state-step (SURVEY.md 8(a)/(d)): full BPTT (n+1)F_pi + n 2F_pi + (2F_pi - 2 d_o H) + 3F_Q,
    default MPG (n+1)F_pi + n F_pi + (2F_pi - 2 d_o H) + 4F_Q, per trajectory, / n."""
    d_o, d_a, _ = synthetic.ENV_DIMS[env_id]
    f_pi = 2 * (d_o * HID + HID * HID + HID * 2 * d_a)
    f_q = 2 * ((d_o + d_a) * HID + HID * HID + HID)
    n = N_STEPS
    if full_bptt:
        traj = (n + 1) * f_pi + n * 2 * f_pi + (2 * f_pi - 2 * d_o * HID) + 3 * f_q
    else:
        traj = (n + 1) * f_pi + n * f_pi + (2 * f_pi - 2 * d_o * HID) + 4 * f_q
    return traj / n


def dump_outputs(out_dir, arrays):
    """{name: array} -> out_dir/<name>.npy; fp32 is kept, every other dtype is written as fp64."""
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        np.save(os.path.join(out_dir, name + '.npy'), a if a.dtype == np.float32 else a.astype(np.float64))


def make_inputs(env_id, rows, seed=1234):
    rng = np.random.default_rng(seed)
    act_dim = synthetic.ENV_DIMS[env_id][1]
    obs = synthetic.make_obs(rng, env_id, rows)
    act = np.clip(rng.normal(0.0, 0.5, (rows, act_dim)), -1, 1).astype(np.float32)
    rew = (-np.abs(rng.standard_normal(rows))).astype(np.float32)
    obs_tp1 = synthetic.make_obs(rng, env_id, rows)
    done = np.zeros(rows, np.float32)
    return [obs, act, rew, obs_tp1, done]


def resolve(opts):
    """-> dict(alg, env_id, rows (per rank), full_bptt, lists, workload, scaling, global_rows)."""
    world = int(os.environ.get('WORLD_SIZE', '1'))
    c = dict(alg='NADP', env_id=ENVS['pt'], rows=ROWS_PER_GPU, scaling='weak', replay=False)
    if opts.config == 1:
        c.update(alg='MPG-v2', rows=256)
    elif opts.config == 3:
        c.update(env_id=ENVS[opts.env if opts.env != 'pt' else 'ip'], rows=131072)
    elif opts.config == 4:
        c.update(alg='MPG-v2', scaling='strong', rows=1048576 // max(world, 1))
    elif opts.config == 5:
        c.update(alg='MPG-v2', rows=262144, replay=True)
    if opts.mode:
        c['alg'] = {'nadp': 'NADP', 'mpg': 'MPG-v2'}[opts.mode]
    if opts.env and opts.config != 3:
        c['env_id'] = ENVS[opts.env]
    if opts.scaling:
        c['scaling'] = opts.scaling
    if opts.global_rows:
        c['scaling'] = 'strong'
        c['rows'] = opts.global_rows // max(world, 1)
    elif opts.rows:
        c['rows'] = opts.rows
    c['full_bptt'] = c['alg'] == 'NADP'
    c['global_rows'] = c['rows'] * max(world, 1)
    names = {'NADP': 'NADP (pure n-step ADP gradient, full BPTT)', 'MPG-v2': 'MPG-v2 (first-action gradient, lists [0, 25])'}
    model = {'PathTracking-v0': 'PathTrackingModel', 'InvertedPendulumConti-v0': 'InvertedPendulumModel',
             'InvertedDoublePendulum-v2': 'InvertedDoublePendulumModel'}[c['env_id']]
    cfg_idx = opts.config if opts.config else 2
    c['workload'] = (f"{model} {names[c['alg']]}, n=25, H=256, B={c['rows']} rows per GPU"
                     f"{' + prioritized replay (sum-tree sampling, priority feedback)' if c['replay'] else ''}"
                     f" (BASELINE.json configs[{cfg_idx - 1}])")
    return c


def learner_args(c, rows):
    kw = dict(replay_batch_size=rows)
    if c['replay']:
        kw.update(buffer_type='priority', max_buffer_size=500000, replay_starts=1, buffer_log_interval=10 ** 9)
    return default_args(c['alg'], c['env_id'], **kw)


def cpu_reference_update(c, args, weights, batch, threads, repeats):
    """Time the restated reference learner (oracle, fp32) for one compute_gradient. Returns seconds (median)."""
    from oracle import mpg_oracle as O
    torch.set_num_threads(threads)
    rows = batch[0].shape[0]
    rng = np.random.default_rng(7)
    nq, npol = synthetic.make_noise(rng, N_STEPS, rows), synthetic.make_noise(rng, N_STEPS, rows)
    times = []
    for i in range(repeats + 1):
        t0 = time.perf_counter()
        if c['alg'] == 'NADP':
            O.nadp_compute_gradient(args, weights, batch, nq, npol, torch.float32)
        else:
            O.mpg_compute_gradient(args, weights, batch, npol, 4000, torch.float32)
        if i:
            times.append(time.perf_counter() - t0)
    return float(np.median(times))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                       '-lms', '100', '-i', str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)    # a run that fails before stop() must not leave the sampler behind
        except Exception:
            self.p = None

    def wait_first_sample(self, timeout=5.0):
        """nvidia-smi needs up to a second to start on an 8-GPU box: do not begin before it is sampling."""
        t0 = time.time()
        while self.p is not None and time.time() - t0 < timeout:
            try:
                if os.path.getsize(self.f.name) > 0:
                    return
            except OSError:
                return
            time.sleep(0.05)

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, power, reasons = [], [], [], set()
        for line in self.f.read().strip().splitlines():
            c = [x.strip() for x in line.split(',')]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), c[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            busy = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
            out.update(sm_mhz=float(np.median(busy)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       power_w_max=float(max(power)), samples=len(sm))
        return out


def run_reference(opts, c, rank):
    """Reference arm: the restated TF2 learner on the host cores, on the SAME rows as our arm (one rank's shard)."""
    if rank != 0:
        return
    rows = c['rows']
    args = learner_args(dict(c, replay=False), rows)
    dq = c['alg'] == 'MPG-v2'
    weights = synthetic.make_policy_with_qs_weights(0, args.obs_dim, args.act_dim, HID, double_q=dq)
    batch = make_inputs(c['env_id'], rows)
    threads = os.cpu_count() or 1
    from oracle import mpg_oracle as O
    torch.set_num_threads(threads)
    rng = np.random.default_rng(7)
    nq, npol = synthetic.make_noise(rng, N_STEPS, rows), synthetic.make_noise(rng, N_STEPS, rows)

    def step():
        if c['alg'] == 'NADP':
            return O.nadp_compute_gradient(args, weights, batch, nq, npol, torch.float32)
        return O.mpg_compute_gradient(args, weights, batch, npol, 4000, torch.float32)
    for _ in range(opts.warmup):
        step()
    ts = []
    for _ in range(opts.steps):
        t0 = time.perf_counter()
        out = step()
        ts.append(time.perf_counter() - t0)
    if opts.dump_outputs:
        dump_outputs(opts.dump_outputs, {'compute_gradient': out['compute_gradient']})
    dt = float(np.mean(ts))
    value = rows * N_STEPS / dt
    sample = (f'all {rows} rows of one GPU\'s shard per step, full {c["alg"]} compute_gradient (Q side + policy rollout '
              f'fwd+bwd + clip), PyTorch-CPU fp32 restatement of the TF2 learner, {threads} threads')
    emit({
        'impl': 'reference', 'metric': 'model state-steps/s (fwd+bwd, n=25)', 'value': value,
        'unit': 'state-steps/s', 'n_gpus': opts.gpus, 'steps': opts.steps, 'warmup': opts.warmup,
        'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': c['scaling'], 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'updates_per_s': 1.0 / dt,
        'config': {'workload': c['workload'], 'global_batch': c['global_rows'], 'horizon': N_STEPS,
                   'host_cores': threads, 'sample': f'{rows} rows per step on the host cores (same rows as one GPU)'},
        'cpu_baseline': {'value': value, 'unit': 'state-steps/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'state-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    })


def mgpu_check(dist, world, rank, e, lists, list_w, full_bptt):
    """Outside the timed region: the all-reduced gradient of the row shards equals the gradient of the global batch
    computed on one rank, and every rank holds bit-identical bytes after the all-reduce."""
    from mpg_b200 import _lib
    rows = 384
    gobs = e.dev(synthetic.make_obs(np.random.default_rng(99), e.env_id, rows * world))
    kw = dict(full_bptt=full_bptt, q_net=_lib.NET_Q1, use_philox=True, noise_seed=3, want_returns=False)
    g, _ = e.policy_grad(gobs[rank * rows:(rank + 1) * rows].contiguous(), lists, list_w, global_rows=rows * world,
                         row_offset=rank * rows, **kw)
    dist.all_reduce(g)
    g_full, _ = e.policy_grad(gobs, lists, list_w, **kw)
    err = float((g - g_full).norm() / g_full.norm())
    digest = g.view(torch.int32).to(torch.int64).sum().reshape(1)
    all_d = [torch.zeros_like(digest) for _ in range(world)]
    dist.all_gather(all_d, digest)
    same = all(int(d.item()) == int(all_d[0].item()) for d in all_d)
    ok = torch.tensor([1.0 if (err <= 1e-5 and same) else 0.0], device=g.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return dict(status='ok' if ok.item() == 1.0 else 'FAILED', rel_l2_vs_single_rank_global_batch=err,
                bit_identical_across_ranks=bool(same), rows_per_rank=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--backend', default='auto', choices=['auto', 'ffma', 'tc'])
    ap.add_argument('--config', type=int, default=0, choices=[0, 1, 2, 3, 4, 5])
    ap.add_argument('--rows', type=int, default=0, help='rows per GPU (overrides the config)')
    ap.add_argument('--scaling', default='', choices=['', 'weak', 'strong'])
    ap.add_argument('--global-rows', type=int, default=0, help='strong scaling: total rows, split evenly over the ranks')
    ap.add_argument('--mode', default='', choices=['', 'nadp', 'mpg'])
    ap.add_argument('--env', default='', choices=['', 'pt', 'ip', 'idp'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)')
    opts = ap.parse_args()
    opts.warmup = max(opts.warmup, 3) if opts.impl == 'ours' else opts.warmup
    if opts.steps < 1:
        raise SystemExit('--steps must be at least 1')
    if opts.dump_outputs:
        os.makedirs(opts.dump_outputs, exist_ok=True)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    c = resolve(opts)
    if opts.impl == 'reference':
        run_reference(opts, c, rank)
        return
    if world != opts.gpus:
        if opts.gpus != 1:
            raise SystemExit(f'--gpus {opts.gpus} needs torchrun with {opts.gpus} processes (WORLD_SIZE={world})')
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    from mpg_b200 import _lib
    from mpg_b200.learners import MPGLearner, NADPLearner
    from mpg_b200.policy import PolicyWithQs

    rows, env_id, full_bptt = c['rows'], c['env_id'], c['full_bptt']
    dq = c['alg'] == 'MPG-v2'
    args = learner_args(c, rows)
    weights = synthetic.make_policy_with_qs_weights(0, args.obs_dim, args.act_dim, HID, double_q=dq)
    learner = (MPGLearner if dq else NADPLearner)(PolicyWithQs, args)
    learner.set_weights(weights)
    e = learner.engine
    backend = 'ffma'
    if opts.backend in ('auto', 'tc') and e.tc_available():
        e.set_backend(1)
        backend = 'tc'
    elif opts.backend == 'tc':
        raise SystemExit('tensor-core backend unavailable for this configuration')
    else:
        e.set_backend(0)
    batch = make_inputs(env_id, rows, seed=1234 + rank)   # every rank owns different rows of the global batch
    obs_dev = e.dev(batch[0])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')   # > 126 MB L2
    global_rows, row_offset = rows * world, rows * rank
    if dq:   # default MPG: lists [0, 25] with the rule-based weights of iteration 4000 (mpg_learner.py:384-399)
        from mpg_b200.learners.base import rule_based_weights
        lists = [0, N_STEPS]
        list_w = [float(x) for x in rule_based_weights(4000, args.rule_based_bias_total_ite, args.eta, lists)]
    else:
        lists, list_w = [N_STEPS], [1.0]

    def device_step():
        g, _ = e.policy_grad(obs_dev, lists, list_w, full_bptt=full_bptt, q_net=_lib.NET_Q1, use_philox=True,
                             noise_seed=7, global_rows=global_rows, row_offset=row_offset, want_returns=False)
        if world > 1:
            dist.all_reduce(g)
        return g

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    check = mgpu_check(dist, world, rank, e, lists, list_w, full_bptt) if world > 1 else None

    # ---------------- device-resident metric ----------------
    sampler = ClockSampler(local_rank) if rank == 0 else None   # runs through warm-up, timed region and e2e loop
    if sampler:
        sampler.wait_first_sample()
    for _ in range(opts.warmup):
        device_step()
    e.set_timing(True)
    barrier()
    l0 = e.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(opts.steps)]
    for a, b in ev:
        flush.zero_()                       # evict L2 between timed iterations
        a.record()
        g_last = device_step()
        b.record()
    barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    launches = e.launch_count - l0
    # dominant-kernel duration of the last timed step (events recorded inside the library right around the rollout kernel)
    kernel_ms = e.kernel_ms()
    e.set_timing(False)
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    ms_per_step = total_ms / opts.steps
    value = rows * world * N_STEPS / (ms_per_step * 1e-3)

    # ---------------- end to end through the learner API with host buffers ----------------
    rb = None
    if c['replay']:
        # config 5: the transitions live in the device sum-tree buffer; an update = sample -> compute_gradient -> priorities
        from mpg_b200.buffer import PrioritizedReplayBuffer
        rb = PrioritizedReplayBuffer(args, 0)
        fill = make_inputs(env_id, args.max_buffer_size, seed=77)
        rb.add_arrays(*fill)

    def update(it):
        if rb is None:
            return learner.compute_gradient(batch, None, None, it)   # returns host numpy arrays (D2H inside)
        samples = rb.replay_device()
        g = learner.compute_gradient(samples[:5], rb, samples[-1], it)
        info = learner.get_info_for_buffer()
        rb.update_priorities(info['indexes'], info['td_error'])
        return g

    for it in range(2):
        update(it)
    e2e_steps = opts.steps
    block_s = []
    for _ in range(3):            # three blocks of K updates; the MEDIAN block is reported
        barrier()
        t0 = time.perf_counter()
        for it in range(e2e_steps):
            grads = update(it)
        torch.cuda.synchronize()
        block_s.append((time.perf_counter() - t0) / e2e_steps)
    e2e_s = torch.tensor([float(np.median(block_s))], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    d2h = int(sum(g.nbytes for g in grads)) + 4 * 8
    e2e_value = rows * world * N_STEPS / e2e_s
    clocks = sampler.stop() if sampler else None
    if opts.dump_outputs and rank == 0:
        dump_outputs(opts.dump_outputs, {'policy_grad': g_last,
                                         'compute_gradient': np.concatenate([x.ravel() for x in grads])})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    flop = flop_per_state_step(env_id, full_bptt)
    k_ms = kernel_ms if kernel_ms > 0 else ms_per_step
    if full_bptt and backend == 'tc' and rows > e.MAX_TC_FULL_BPTT_ROWS:
        k_ms = ms_per_step      # the call is split into row chunks (several launches): the whole step is the denominator
    achieved_tf = rows * N_STEPS * flop / (k_ms * 1e-3) / 1e12
    # a kernel timed alone over a sub-100 ms region at full clocks: the burst figure is the honest denominator
    peak_tf = float(peaks.get('bf16_tflops', 1655.0))
    sm_mhz = (clocks or {}).get('sm_mhz') or 1965.0
    ffma_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    traffic, traffic_src = None, None   # dram__bytes_read.sum + dram__bytes_write.sum of the same kernel (ncu --set full)
    for name in (('r2_tc_rollout_kernel_ncu_full.csv', 'r1c_tc_rollout_kernel_ncu_full.csv') if backend == 'tc'
                 else ('r1_ffma_rollout_kernel_ncu_full.csv',)):
        try:
            mult = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
            tot = 0.0
            for line in open(os.path.join(ROOT, 'profiles', name)):
                cc = line.strip().split(',')
                if cc[0] in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                    tot += float(cc[2]) * mult[cc[1]]
            if tot > 0 and env_id == ENVS['pt'] and full_bptt:
                traffic, traffic_src = tot * (rows / float(ROWS_PER_GPU)), name
                break
        except Exception:
            continue
    roofline = {
        'bound': 'tensor', 'achieved': achieved_tf, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved_tf / peak_tf,
        'traffic': traffic,
        'traffic_note': ('bytes per launch from profiles/%s (ncu --set full of the same kernel at B=65536, scaled by rows); '
                         'algorithmic bytes are 56 B/state-step; the tc path adds the h2 image store (1 KB/state-step written '
                         'by the forward pass, read back by BPTT) and the dW2 operand records (h1, delta2: 1 KB/state-step hi-only at this size, 2 KB below 262,144 row-steps)'
                         % traffic_src) if traffic_src else 'no ncu capture of this configuration',
        'kernel': 'rollout_kernel<%s,BWD> (fused forward rollout + BPTT, %s backend)' % (env_id, backend),
        'kernel_ms': k_ms, 'algorithmic_flop_per_state_step': flop,
        'peak_source': ('MEASURED_PEAKS.json bf16_tflops (burst, of measured)' if peaks else 'fallback 1.655 PFLOP/s (of fallback)'),
        'frac_of_sustained_bf16': achieved_tf / float(peaks.get('bf16_tflops_sustained', 1373.4)),
        'fp32_ffma_peak_tflops_at_run_clock': ffma_peak, 'frac_of_fp32_ffma_peak': achieved_tf / ffma_peak,
        'hbm_bytes_per_state_step_algorithmic': 56,
    }
    cpu_baseline = None
    if world == 1 and not opts.no_cpu_baseline:
        threads = os.cpu_count() or 1
        cpu_rows = min(rows, ROWS_PER_GPU)      # bounded: ~10-30 s of CPU work
        cpu_args = learner_args(dict(c, replay=False), cpu_rows)
        cpu_batch = [b[:cpu_rows] for b in batch]
        t_all = cpu_reference_update(c, cpu_args, weights, cpu_batch, threads, 2)
        b256 = [b[:256] for b in batch]
        t_one = cpu_reference_update(c, learner_args(dict(c, replay=False), 256), weights, b256, 1, 3)
        cpu_baseline = {
            'value': cpu_rows * N_STEPS / t_all, 'unit': 'state-steps/s', 'cores': threads, 'kind': 'port',
            'sample': ('%d of the %d rows of the workload, full %s compute_gradient, PyTorch-CPU fp32 restatement of the '
                       'TF2 learner (TensorFlow not installable here), median of 2 after 1 warm-up' % (cpu_rows, rows, c['alg'])),
            'single_thread_b256_value': 256 * N_STEPS / t_one,
            'single_thread_b256_note': 'reference default: 1 intra/inter-op thread per learner, batch 256',
        }
    line = {
        'metric': 'model state-steps/s (fwd+bwd, n=25)', 'value': value, 'unit': 'state-steps/s', 'n_gpus': world,
        'steps': opts.steps, 'warmup': opts.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
        'scaling': c['scaling'], 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': c['workload'],
                   'global_batch': rows * world, 'horizon': N_STEPS, 'backend': backend,
                   'noise': 'in-kernel Philox4x32-10 keyed (seed, global row, step)',
                   'cache': 'L2 flushed between timed iterations (256 MiB memset)',
                   'step': 'one policy forward+backward rollout (mpg_policy_grad)' + (
                       ' + NCCL all-reduce of the flat policy gradient' if world > 1 else ''),
                   'e2e_step': ('%s.compute_gradient with host numpy buffers' % type(learner).__name__ if rb is None else
                                'sum-tree sample (device) -> MPGLearner.compute_gradient -> update_priorities')
                               + ' (adds the Q side and the clip); wall clock, median of three blocks of %d updates' % e2e_steps,
                   'host_cores': os.cpu_count()},
        'updates_per_s': 1.0 / e2e_s,
        'e2e': {'value': e2e_value, 'unit': 'state-steps/s', 'h2d_bytes_per_step': int(learner.h2d_bytes),
                'd2h_bytes_per_step': d2h, 'ms_per_update': e2e_s * 1e3, 'blocks_ms': [b * 1e3 for b in block_s]},
        'gpu_launches': int(launches),
        'clocks': clocks,
        'roofline': roofline,
        'cpu_baseline': cpu_baseline,
        'target_state_steps_per_s_per_gpu': 1e8,
    }
    if check is not None:
        line['mgpu_check'] = check['status']
        line['mgpu_check_detail'] = check
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
