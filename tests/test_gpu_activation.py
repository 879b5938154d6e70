"""relu and tanh hidden activations (value_hidden_activation == policy_hidden_activation) on the fp32 FFMA kernels at
H = 64 / 128 / 256 and on the tensor-core kernels at H = 256.  The reference has golden vectors for 'elu' only, so the
truth here is the fp64 oracle with the same activation, held to the suite's bars: states / rewards / actions 1e-5 per
step, gradients 1e-4, scalars 2e-5.  The oracle's own relu / tanh gradients are first checked against central finite
differences (CPU).

The oracle (oracle/mpg_oracle.py) evaluates every MLP through its module-level mlp(); `oracle_activation` swaps that
function for the duration of a comparison, so every oracle routine (rollout, targets, TD errors, n-step targets) runs
the activation under test."""
import contextlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mpg_b200 import synthetic
from mpg_b200.config import default_args
from tests.util import make_batch, rel_l2

TOL_STATE, TOL_GRAD, TOL_SCALAR = 1e-5, 1e-4, 2e-5
PT, IP, IDP = 'PathTracking-v0', 'InvertedPendulumConti-v0', 'InvertedDoublePendulum-v2'
ACTS = ['relu', 'tanh']
CONFIGS = [('ffma', 64), ('ffma', 128), ('ffma', 256), ('tc', 256)]
CONFIG_IDS = ['ffma64', 'ffma128', 'ffma256', 'tc256']
HIDDEN_FN = {'elu': F.elu, 'relu': F.relu, 'tanh': torch.tanh}


@contextlib.contextmanager
def oracle_activation(act):
    """Run the oracle's MLPNet (model.py:39-43) with Dense(activation=act) hidden layers."""
    from oracle import mpg_oracle as O
    f = HIDDEN_FN[act]

    def mlp(w, x, out_act='linear'):
        h = f(x @ w[0] + w[1])
        h = f(h @ w[2] + w[3])
        y = h @ w[4] + w[5]
        return torch.tanh(y) if out_act == 'tanh' else y

    saved = O.mlp
    O.mlp = mlp
    try:
        yield O
    finally:
        O.mlp = saved


def _args(alg, env_id, H, act, **kw):
    return default_args(alg, env_id, value_num_hidden_units=H, policy_num_hidden_units=H,
                        value_hidden_activation=act, policy_hidden_activation=act, **kw)


def _flat(grads):
    return np.concatenate([np.asarray(g, np.float64).ravel() for g in grads])


def _unclip(g, norm, clip):
    return g * max(norm, clip) / clip


def _select(engine, backend):
    from mpg_b200.engine import BACKEND_FFMA, BACKEND_TC
    if backend == 'tc':
        assert engine.tc_available()
        engine.set_backend(BACKEND_TC)
    else:
        engine.set_backend(BACKEND_FFMA)


def _learner(kind, args, weights, backend):
    from mpg_b200.learners import MPGLearner, NADPLearner
    from mpg_b200.policy import PolicyWithQs
    learner = (NADPLearner if kind == 'nadp' else MPGLearner)(PolicyWithQs, args)
    learner.set_weights(weights)
    _select(learner.engine, backend)
    assert learner.engine.lib.mpg_get_activation(learner.engine.h) == {'relu': 1, 'tanh': 2}[args.policy_hidden_activation]
    return learner


def _policy(args, weights, backend):
    from mpg_b200.policy import PolicyWithQs
    pol = PolicyWithQs(**vars(args))
    if weights is not None:
        pol.set_weights(weights)
    _select(pol.engine, backend)
    return pol


# ------------------------------------------------------------------------------------------------
# CPU: the oracle's relu / tanh gradients against central finite differences; the activation check
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('act', ACTS)
def test_oracle_gradients_match_finite_differences(act):
    """Policy gradient of the model rollout (NADP loss -R_n) and Q regression gradient of the oracle with relu / tanh
    hidden layers against central differences in fp64.  For relu a sampled parameter is skipped when a hidden
    pre-activation changes sign between the two evaluations: across a kink a difference quotient is not a derivative."""
    from oracle import mpg_oracle as O
    H, B, n, h = 32, 6, 3, 1e-6
    args = _args('NADP', PT, H, act, replay_batch_size=B)
    w = synthetic.make_policy_with_qs_weights(3, args.obs_dim, args.act_dim, H, double_q=False)
    rng = np.random.default_rng(4)
    obs = O.to_t(synthetic.make_obs(rng, PT, B), torch.float64)
    noise = O.to_t(synthetic.make_noise(rng, n, B), torch.float64)
    act_in = O.to_t(rng.uniform(-1, 1, (B, args.act_dim)), torch.float64)
    target = O.to_t(rng.standard_normal(B), torch.float64)
    sigma = O.to_t(args.obs_scale, torch.float64)
    pre_acts = []
    f = HIDDEN_FN[act]

    def recording_mlp(wt, x, out_act='linear'):
        z1 = x @ wt[0] + wt[1]
        z2 = f(z1) @ wt[2] + wt[3]
        pre_acts.append(torch.cat([z1.detach().ravel(), z2.detach().ravel()]))
        y = f(z2) @ wt[4] + wt[5]
        return torch.tanh(y) if out_act == 'tanh' else y

    with oracle_activation(act):
        O.mlp = recording_mlp
        nets = O.Nets(w, False, torch.float64)

        def policy_loss(pw):
            return -O.rollout(args, torch.float64, pw, pw, nets.Q1, obs, noise, n)[n].mean()

        def q_loss(qw):
            return 0.5 * torch.mean((O.q_value(qw, obs * sigma, act_in) - target) ** 2)

        checked = 0
        for loss_fn, params in ((policy_loss, nets.policy), (q_loss, nets.Q1)):
            grads = torch.autograd.grad(loss_fn(params), params)
            sel = np.random.default_rng(5)
            for _ in range(24):
                i = int(sel.integers(len(params)))
                j = int(sel.integers(params[i].numel()))
                vals, signs = [], []
                for s in (h, -h):
                    pw = [p.detach().clone(memory_format=torch.contiguous_format) for p in params]
                    pw[i].view(-1)[j] += s
                    pre_acts.clear()
                    with torch.no_grad():
                        vals.append(float(loss_fn(pw)))
                    signs.append(torch.cat(pre_acts) > 0)
                if act == 'relu' and not torch.equal(signs[0], signs[1]):
                    continue                    # the two evaluations straddle a kink
                fd = (vals[0] - vals[1]) / (2 * h)
                an = float(grads[i].reshape(-1)[j])
                assert abs(fd - an) <= 1e-6 * max(abs(an), 1e-3), (i, j, fd, an)
                checked += 1
        assert checked >= 40, checked


def test_activation_check_precedes_the_device():
    from mpg_b200.policy import PolicyWithQs
    with pytest.raises(NotImplementedError, match='elu / relu / tanh'):
        PolicyWithQs(**vars(_args('NADP', PT, 256, 'gelu')))
    with pytest.raises(NotImplementedError, match='must be equal'):
        PolicyWithQs(**vars(default_args('NADP', PT, value_hidden_activation='relu', policy_hidden_activation='tanh')))
    if torch.cuda.is_available():
        return
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        PolicyWithQs(**vars(_args('NADP', PT, 64, 'relu')))


# ------------------------------------------------------------------------------------------------
# compute_gradient against the oracle
# ------------------------------------------------------------------------------------------------
def _nadp_vs_oracle(env_id, B, n, backend, H, act, seed=0, per_row=False):
    from tests.test_gpu_parity import _row_returns_vs_oracle
    args = _args('NADP', env_id, H, act, replay_batch_size=B, num_rollout_list_for_policy_update=[n],
                 num_rollout_list_for_q_estimation=[n])
    w = synthetic.make_policy_with_qs_weights(100 + seed, args.obs_dim, args.act_dim, H, double_q=False)
    batch = make_batch(200 + seed, env_id, B, 0)
    rng = np.random.default_rng(300 + seed)
    nq, npol = synthetic.make_noise(rng, n, B), synthetic.make_noise(rng, n, B)
    learner = _learner('nadp', args, w, backend)
    learner.set_rollout_noise(nq, npol)
    flat = _flat(learner.compute_gradient(batch, None, None, 0))
    st = learner.get_stats()
    with oracle_activation(act) as O:
        ref = O.nadp_compute_gradient(args, w, batch, nq, npol, torch.float64)
        row = _row_returns_vs_oracle(learner, args, w, batch, npol, n) if per_row else None
    nQ = ref['q_grad'].size
    clip = args.gradient_clip_norm
    errs = dict(q=rel_l2(_unclip(flat[:nQ], st['q_gradient_norm'], clip), ref['q_grad']),
                p=rel_l2(_unclip(flat[nQ:], st['policy_gradient_norm'], clip), ref['policy_grad']),
                clipped=rel_l2(flat, ref['compute_gradient']))
    if per_row:
        # means of per-row returns of both signs nearly cancel: rows to 1e-5, means to the matching absolute error
        errs['rows'], scale = row
        assert errs['rows'] <= TOL_STATE, errs
        for k in ('policy_loss', 'value_mean'):
            assert abs(st[k] - ref[k]) <= TOL_SCALAR * max(scale, abs(ref[k])), (k, st[k], ref[k], scale)
        target_scale = float(np.abs(ref['q_targets']).mean())
        assert abs(st['q_loss'] - ref['q_loss']) <= 2 * TOL_SCALAR * max(target_scale ** 2, abs(ref['q_loss']))
    else:
        for k in ('q_loss', 'policy_loss', 'value_mean'):
            errs[k] = rel_l2(st[k], ref[k])
            assert errs[k] <= TOL_SCALAR, errs
    print('NADP', env_id, B, n, backend, H, act, errs)
    assert errs['q'] <= TOL_GRAD and errs['p'] <= TOL_GRAD and errs['clipped'] <= TOL_GRAD, errs
    return learner


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize('B', [1, 300, 2048])
def test_nadp_pathtracking_vs_oracle(B, backend, H, act):
    # tensor cores + relu: the means over the rows land at ~3e-5 of the oracle's (measured 3.2e-5 at B = 300 and 2048),
    # so there the rows are held to 1e-5 each and the means to the matching absolute error, as for B = 1
    _nadp_vs_oracle(PT, B, 25, backend, H, act, per_row=(B < 16 or (backend == 'tc' and act == 'relu')))


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_nadp_multi_wave_vs_oracle(backend, H, act):
    """20,011 rows: more tiles than SMs on both backends (and the wave-tail split of the tensor-core path)."""
    learner = _nadp_vs_oracle(PT, 20011, 3, backend, H, act, seed=9, per_row=True)
    assert learner.engine.num_sms < 20011 // 128


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_nadp_cart_pole_vs_oracle(backend, H, act):
    _nadp_vs_oracle(IP, 200, 25, backend, H, act)


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_nadp_double_pendulum_short_horizon_vs_oracle(backend, H, act):
    # the falling double pendulum amplifies rounding beyond a few steps (tests/test_gpu_parity.py): n = 3
    _nadp_vs_oracle(IDP, 128, 3, backend, H, act)


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_mpg_v2_vs_oracle(backend, H, act):
    B, ite = 160, 4000
    args = _args('MPG-v2', PT, H, act, replay_batch_size=B, num_rollout_list_for_policy_update=[0, 25],
                 buffer_type='priority', sample_num_in_learner=None)
    w = synthetic.make_policy_with_qs_weights(7, args.obs_dim, args.act_dim, H, double_q=True)
    batch = make_batch(8, PT, B, 0)
    npol = synthetic.make_noise(np.random.default_rng(9), 25, B)
    learner = _learner('mpg', args, w, backend)
    learner.set_rollout_noise(None, npol)
    flat = _flat(learner.compute_gradient(batch, None, None, ite))
    st = learner.get_stats()
    with oracle_activation(act) as O:
        ref = O.mpg_compute_gradient(args, w, batch, npol, ite, torch.float64)
    nQ = ref['q_grad1'].size
    errs = dict(clipped=rel_l2(flat, ref['compute_gradient']),
                p=rel_l2(_unclip(flat[2 * nQ:], st['policy_gradient_norm'], args.gradient_clip_norm), ref['policy_grad']),
                targets=rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), ref['batch_targets']),
                td=rel_l2(learner.get_info_for_buffer()['td_error'], ref['td_error']),
                total_loss=rel_l2(st['policy_total_loss'], ref['total_loss']),
                value_mean=rel_l2(st['value_mean'], ref['value_mean']),
                q1=rel_l2(st['q_loss1'], ref['q_loss1']))
    print('MPG-v2', backend, H, act, errs)
    assert errs['clipped'] <= TOL_GRAD and errs['p'] <= TOL_GRAD, errs
    for k in ('targets', 'td', 'total_loss', 'value_mean', 'q1'):
        assert errs[k] <= TOL_SCALAR, errs


# ------------------------------------------------------------------------------------------------
# closed-loop trajectories (mpg_rollout_forward traj outputs), per step
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_closed_loop_trajectories_vs_oracle(backend, H, act):
    """Observations, rewards and actions of every step <= 1e-5 norm-relative; on the tensor-core path over 4 (weight,
    state, noise) seeds, whose fp16-pair forward is where an inexact tanh would show."""
    B, n = 512, 25
    args = _args('NADP', PT, H, act, replay_batch_size=B)
    pol = _policy(args, None, backend)
    e = pol.engine
    worst = dict(obs=0.0, rew=0.0, act=0.0)
    for seed in (range(4) if backend == 'tc' else range(1)):
        w = synthetic.make_policy_with_qs_weights(40 + seed, args.obs_dim, args.act_dim, H, double_q=False)
        rng = np.random.default_rng(60 + seed)
        obs0 = synthetic.make_obs(rng, PT, B)
        noise = synthetic.make_noise(rng, n, B)
        pol.set_weights(w)
        _, t_obs, t_rew, t_act = e.rollout_forward(e.dev(obs0), [n], noise=e.dev(noise), want_traj=True)
        with oracle_activation(act) as O:
            ro, rr, ra = O.closed_loop(args, w[1], obs0, noise, n, torch.float64)
        cur = dict(obs=max(rel_l2(t_obs[t].cpu().numpy(), ro[t]) for t in range(n)),
                   rew=max(rel_l2(t_rew[t].cpu().numpy(), rr[t]) for t in range(n)),
                   act=max(rel_l2(t_act[t].cpu().numpy(), ra[t]) for t in range(n + 1)))
        print('closed loop', backend, H, act, 'seed', seed, cur)
        for k in worst:
            worst[k] = max(worst[k], cur[k])
    assert max(worst.values()) <= TOL_STATE, worst


# ------------------------------------------------------------------------------------------------
# Q side
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_forward_entry_points_vs_oracle(backend, H, act):
    """compute_action / compute_Q1 (mpg_policy_forward / mpg_q_forward), mpg_q_target (double Q), mpg_td_error and
    mpg_q_bootstrap against the oracle's networks."""
    B = 1000
    args = _args('MPG-v2', PT, H, act, replay_batch_size=B)   # capacity B: the tensor-core handle evaluates on tensor cores
    w = synthetic.make_policy_with_qs_weights(3, args.obs_dim, args.act_dim, H, double_q=True)
    pol = _policy(args, w, backend)
    e = pol.engine
    assert e.cfg.max_rows >= B
    rng = np.random.default_rng(4)
    obs, obs1 = synthetic.make_obs(rng, PT, B), synthetic.make_obs(rng, PT, B)
    sigma = np.asarray(args.obs_scale, np.float32)
    act_in = rng.uniform(-1, 1, (B, args.act_dim)).astype(np.float32)
    rew = (-np.abs(rng.standard_normal(B))).astype(np.float32)
    got_a, _ = pol.compute_action(obs * sigma)
    got_q = pol.compute_Q1(obs * sigma, act_in)
    got_tgt = e.q_target(True, e.dev(rew), e.dev(obs1))
    got_td = e.td_error(e.dev(obs), e.dev(act_in), e.dev(rew), e.dev(obs1))
    got_bs = e.q_bootstrap(e.dev(rew), 0.7, e.dev(obs))
    with oracle_activation(act) as O, torch.no_grad():
        nets = O.Nets(w, True, torch.float64)
        t64 = lambda x: O.to_t(x, torch.float64)   # noqa: E731
        p, p1 = t64(obs) * t64(sigma), t64(obs1) * t64(sigma)
        prew = (t64(rew) + args.rew_shift) * args.rew_scale
        a1 = O.policy_action(nets.policy_t, p1, args.policy_out_activation, args.action_range)
        a0 = O.policy_action(nets.policy_t, p, args.policy_out_activation, args.action_range)
        ref = dict(
            act=O.policy_action(nets.policy, p, args.policy_out_activation, args.action_range),
            q=O.q_value(nets.Q1, p, t64(act_in)),
            tgt=prew + args.gamma * torch.minimum(O.q_value(nets.Q1_t, p1, a1), O.q_value(nets.Q2_t, p1, a1)),
            td=prew + args.gamma * O.q_value(nets.Q1_t, p1, a1) - O.q_value(nets.Q1, p, t64(act_in)),
            bs=t64(rew) + 0.7 * O.q_value(nets.Q1_t, p, a0))
    got = dict(act=got_a, q=got_q, tgt=got_tgt, td=got_td, bs=got_bs)
    errs = {k: rel_l2(got[k].cpu().numpy(), ref[k].numpy()) for k in ref}
    print('forward entry points', backend, H, act, errs)
    assert errs['act'] <= TOL_STATE and errs['q'] <= TOL_STATE, errs
    for k in ('tgt', 'td', 'bs'):
        assert errs[k] <= TOL_SCALAR, errs


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('residual', ['systematic', 'noise'])
def test_tc_q_grad_262144_rows_vs_oracle(residual, act):
    """Q regression on the tensor-core path at 262,144 rows; the two residual regimes and bars of
    tests/test_gpu_parity.py::test_tc_q_grad_262144_rows_vs_oracle ('noise' cancels to ~1/512 of its terms: 5e-4)."""
    from mpg_b200 import _lib
    rows, H = 262144, 256
    args = _args('NADP', PT, H, act, replay_batch_size=rows)
    w = synthetic.make_policy_with_qs_weights(11, args.obs_dim, args.act_dim, H, double_q=False)
    rng = np.random.default_rng(12)
    obs = synthetic.make_obs(rng, PT, rows)
    act_in = rng.uniform(-1, 1, (rows, args.act_dim)).astype(np.float32)
    with oracle_activation(act) as O:
        nets = O.Nets(w, False, torch.float64)
        q_pred = O.q_value(nets.Q1, O.to_t(obs, torch.float64) * O.to_t(args.obs_scale, torch.float64),
                           O.to_t(act_in, torch.float64))
        q0 = q_pred.detach().numpy()
        target = ((0.5 * q0 if residual == 'systematic' else q0) + rng.standard_normal(rows)).astype(np.float32)
        loss = 0.5 * torch.mean((q_pred - O.to_t(target, torch.float64)) ** 2)
        ref = np.concatenate([x.numpy().ravel() for x in torch.autograd.grad(loss, nets.Q1)])
    e = _policy(args, w, 'tc').engine
    g, loss_sum = e.q_grad(_lib.NET_Q1, e.dev(obs), e.dev(act_in), e.dev(target))
    err = rel_l2(g.cpu().numpy(), ref)
    print('tc q_grad 262144 rows', residual, act, err)
    assert abs(float(loss_sum.item()) / rows - float(loss.item())) <= TOL_SCALAR * abs(float(loss.item()))
    # relu, 'noise': the delta1 mask comes from the bf16-pair first-layer recompute, not from the forward's fp16-pair z1, so
    # rows whose |z1| is below the recompute's rounding can flip it; the cancellation of this regime magnifies each flip
    # ~512 x (measured 7.6e-4, ELU / tanh ~2e-4)
    noise_bar = 1e-3 if act == 'relu' else 5e-4
    assert err <= (TOL_GRAD if residual == 'systematic' else noise_bar), err


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_mpg_v1_real_env_n_step_target_vs_oracle(backend, H, act):
    """compute_n_step_target (mpg_learner.py:153-169): 25 steps of the real PathTracking environment under the policy,
    bootstrapped with Q1_target, against the oracle's n-step target."""
    B, T = 300, 25
    args = _args('MPG-v1', PT, H, act, replay_batch_size=B, sample_num_in_learner=T)
    w = synthetic.make_policy_with_qs_weights(5, args.obs_dim, args.act_dim, H, double_q=False)
    batch = make_batch(6, PT, B, 0)
    learner = _learner('mpg', args, w, backend)
    learner.get_batch_data(batch, None, None)
    with oracle_activation(act) as O:
        ref, _ = O.mpg_v1_n_step_target(args, w, batch, T, torch.float64)
    err = rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), ref)
    print('MPG-v1 n-step target', backend, H, act, err)
    assert err <= TOL_SCALAR, err


# ------------------------------------------------------------------------------------------------
# fused sampler (worker / evaluator): mpg_env_sample transitions against the oracle's policy + env step
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('H', [64, 128, 256])
def test_env_sample_vs_oracle(H, act):
    from mpg_b200.envs_and_models import PathTrackingEnv
    agents, steps, sig = 200, 12, 0.2
    args = _args('MPG-v2', PT, H, act)
    w = synthetic.make_policy_with_qs_weights(21, args.obs_dim, args.act_dim, H, double_q=True)
    pol = _policy(args, w, 'ffma')
    e = pol.engine
    rng = np.random.default_rng(22)
    obs0 = synthetic.make_obs(rng, PT, agents)
    eps = rng.standard_normal((steps, agents, args.act_dim)).astype(np.float32)
    env = PathTrackingEnv(num_future_data=0, num_agent=agents)
    env.reset(init_obs=obs0)
    o, a, r, o1, d = [t.cpu().numpy() for t in e.env_sample(env.state, env.obs, None, e.dev(eps), sig, steps=steps)]
    sigma = np.asarray(args.obs_scale, np.float64)
    worst = 0.0
    with oracle_activation(act) as O, torch.no_grad():
        nets = O.Nets(w, True, torch.float64)
        env_o = O.PathTrackingEnvOracle(0, np.float64)
        env_o.reset(obs0)
        for t in range(steps):
            ob = env_o.get_obs()
            at = O.policy_action(nets.policy, O.to_t(ob * sigma, torch.float64), args.policy_out_activation,
                                 args.action_range).numpy() + sig * eps[t]
            ob1, rew, _ = env_o.step(at)
            rows = slice(t * agents, (t + 1) * agents)
            worst = max(worst, rel_l2(o[rows], ob), rel_l2(a[rows], at), rel_l2(o1[rows], ob1), rel_l2(r[rows], rew))
    print('env_sample', H, act, 'worst per-step rel-L2', worst)
    assert worst <= TOL_STATE, worst


# ------------------------------------------------------------------------------------------------
# bench size: B = 65,536, n = 25
# ------------------------------------------------------------------------------------------------
_BENCH_ORACLE = {}


def _bench_path_oracle(args, w, obs, n, seed, H, act, chunk=8192):
    """fp64 oracle of the bench workload in row chunks: per-row returns R_n and the policy gradient, with the noise
    of the numpy restatement of the kernel's Philox stream (as tests/test_gpu_parity.py::_bench_path_oracle)."""
    if (H, act) in _BENCH_ORACLE:
        return _BENCH_ORACLE[(H, act)]
    B = obs.shape[0]
    grad, rows = None, []
    with oracle_activation(act) as O:
        nets = O.Nets(w, False, torch.float64)
        for lo in range(0, B, chunk):
            hi = min(B, lo + chunk)
            noise = synthetic.philox_normal(seed, hi - lo, n, global_rows=B, row_offset=lo)
            ret = O.rollout(args, torch.float64, nets.policy, nets.policy, nets.Q1, O.to_t(obs[lo:hi], torch.float64),
                            O.to_t(noise, torch.float64), n)
            g = np.concatenate([x.numpy().ravel() for x in torch.autograd.grad(-ret[n].sum() / B, nets.policy)])
            grad = g if grad is None else grad + g
            rows.append(ret[n].detach().numpy())
    _BENCH_ORACLE[(H, act)] = (np.concatenate(rows), grad)
    return _BENCH_ORACLE[(H, act)]


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('backend,H', CONFIGS, ids=CONFIG_IDS)
def test_bench_size_properties_and_oracle(backend, H, act):
    """Two identical calls are bit-identical; two half batches with global scaling add up to the full batch; the bench
    path (in-kernel Philox, full BPTT; on the tensor-core path with hi-only dW2 records) per-row returns <= 1e-5 and
    gradient <= 1e-4 against the fp64 oracle."""
    from mpg_b200 import _lib
    B, n, seed = 65536, 25, 7
    args = _args('NADP', PT, H, act, replay_batch_size=B)
    w = synthetic.make_policy_with_qs_weights(0, args.obs_dim, args.act_dim, H, double_q=False)
    obs = synthetic.make_obs(np.random.default_rng(1234), PT, B)
    e = _policy(args, w, backend).engine
    x = e.dev(obs)
    kw = dict(full_bptt=True, use_philox=True, noise_seed=11)
    g1, r1 = e.policy_grad(x, [0, n], [0.3, 0.7], **kw)
    g2, r2 = e.policy_grad(x, [0, n], [0.3, 0.7], **kw)
    assert torch.equal(g1, g2) and torch.equal(r1, r2), 'not bit-reproducible run to run'
    assert torch.isfinite(g1).all() and torch.isfinite(r1).all()
    h = B // 2
    gl, _ = e.policy_grad(x[:h].contiguous(), [0, n], [0.3, 0.7], global_rows=B, row_offset=0, **kw)
    gr, _ = e.policy_grad(x[h:].contiguous(), [0, n], [0.3, 0.7], global_rows=B, row_offset=h, **kw)
    shard = rel_l2((gl + gr).cpu().numpy(), g1.cpu().numpy())
    assert shard <= (1e-5 if backend == 'ffma' else 1e-4), shard
    g, ret = e.policy_grad(x, [n], [1.0], full_bptt=True, q_net=_lib.NET_Q1, use_philox=True, noise_seed=seed)
    rows_ref, grad_ref = _bench_path_oracle(args, w, obs, n, seed, H, act)
    errs = dict(rows=rel_l2(ret[0].cpu().numpy(), rows_ref), grad=rel_l2(g.cpu().numpy(), grad_ref), shard=shard)
    print('bench path', backend, H, act, errs)
    assert errs['rows'] <= TOL_STATE and errs['grad'] <= TOL_GRAD, errs


# ------------------------------------------------------------------------------------------------
# C ABI
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('backend,H', [('ffma', 64), ('tc', 256)], ids=['ffma64', 'tc256'])
def test_activation_abi(backend, H):
    """The default is ELU; set / get round trip; an unknown value is refused and changes nothing; switching the
    activation of a live handle gives the same bytes as a handle created with it (the weight images do not depend
    on the activation)."""
    from mpg_b200 import _lib
    B, n = 1000, 10
    w = synthetic.make_policy_with_qs_weights(2, 6, 2, H, double_q=False)
    fresh = _policy(_args('NADP', PT, H, 'tanh', replay_batch_size=B), w, backend).engine
    live = _policy(_args('NADP', PT, H, 'elu', replay_batch_size=B), w, backend).engine
    lib = live.lib
    assert lib.mpg_get_activation(live.h) == 0 and lib.mpg_get_activation(fresh.h) == _lib.ACTIVATIONS['tanh']
    for bad in (-1, 3, 99):
        assert lib.mpg_set_activation(live.h, bad) == -1             # MPG_ERR_ARG
        assert b'bad activation' in lib.mpg_last_error(live.h)
        assert lib.mpg_get_activation(live.h) == 0
    obs = live.dev(synthetic.make_obs(np.random.default_rng(3), PT, B))
    kw = dict(full_bptt=True, use_philox=True, noise_seed=5)
    g_elu, _ = live.policy_grad(obs, [0, n], [0.5, 0.5], **kw)
    for name in ('relu', 'tanh', 'elu'):
        assert lib.mpg_set_activation(live.h, _lib.ACTIVATIONS[name]) == 0
        assert lib.mpg_get_activation(live.h) == _lib.ACTIVATIONS[name]
        g, r = live.policy_grad(obs, [0, n], [0.5, 0.5], **kw)
        if name == 'tanh':
            g_ref, r_ref = fresh.policy_grad(obs, [0, n], [0.5, 0.5], **kw)
            assert torch.equal(g, g_ref) and torch.equal(r, r_ref)
            a_live = live.policy_forward(_lib.NET_POLICY, obs)
            assert torch.equal(a_live, fresh.policy_forward(_lib.NET_POLICY, obs))
        if name == 'elu':
            assert torch.equal(g, g_elu)
        else:
            assert not torch.equal(g, g_elu)


# ------------------------------------------------------------------------------------------------
# trainer smoke tests
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('H,act', [(64, 'relu'), (256, 'tanh')], ids=['relu64', 'tanh256'])
def test_trainer_smoke(H, act):
    from mpg_b200.engine import BACKEND_FFMA, BACKEND_TC
    from mpg_b200.trainer import Trainer
    args = _args('MPG-v2', PT, H, act, replay_batch_size=256, batch_size=512, num_agent=8, explore_sigma=0.1,
                 max_buffer_size=100000, replay_starts=1024, buffer_log_interval=10 ** 9, num_eval_agent=16,
                 num_eval_episode=1, fixed_steps=20, eval_interval=10 ** 9, log_interval=10 ** 9, max_iter=8, log_dir=None)
    tr = Trainer(args)
    assert tr.learner.engine.backend == (BACKEND_TC if H == 256 else BACKEND_FFMA)
    assert tr.learner.engine.hidden_activation == act
    tr.train(args.max_iter)
    st = tr.learner.get_stats()
    for k in ('policy_gradient_norm', 'q_gradient_norm1', 'q_loss1', 'policy_total_loss', 'value_mean'):
        assert np.isfinite(st[k]), (k, st[k])
    assert np.isfinite(tr.evaluator.run_evaluation(args.max_iter)['episode_return'])
