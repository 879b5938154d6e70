"""Both kernel families against the fp64 oracle across the configurations the reference defaults never reach:
num_future_data up to 10 (the tensor-core / FFMA boundary at 7 / 8), the four policy heads, reward shift / scale and
discount, no bootstrap (q_net = -1), unsorted / zero-weight / negative-weight / eight-entry / repeated rollout lists,
a 70-step horizon across the 64-bit list masks of the tensor-core kernel, M = 3 with ragged tiles over more than one
wave, the return statistics and the model adjoint at nfd > 0.

The bars are the suite's: per-row returns and per-step closed-loop obs / rewards / actions <= 1e-5 norm-relative,
gradients <= 1e-4 relative L2.  Every case prints its measured errors."""
import copy

import numpy as np
import pytest
import torch

from mpg_b200 import _lib, synthetic
from mpg_b200.config import default_args
from tests.util import make_batch, rel_l2

pytestmark = pytest.mark.gpu

TOL_STATE, TOL_GRAD = 1e-5, 1e-4
PT, IP = 'PathTracking-v0', 'InvertedPendulumConti-v0'
BACKENDS = ['ffma', 'tc']
Q_NETS = {_lib.NET_Q1: 'Q1', _lib.NET_Q1_TARGET: 'Q1_t'}


def _handle(args, w, backend):
    """PolicyWithQs handle with weights `w` on the requested backend (skips where tensor cores do not cover it)."""
    from mpg_b200.policy import PolicyWithQs
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(w)
    e = pol.engine
    if backend == 'tc':
        if not e.tc_available():
            pytest.skip('tensor-core backend does not cover this configuration')
        e.set_backend(1)
    else:
        e.set_backend(0)
    return pol, e


def oracle_policy_grad(args, w, obs, noise, lst, list_w, M, full_bptt, q_net, dtype=torch.float64):
    """Reference of one mpg_policy_grad call: the oracle rollout over the M tiles of `obs`, then the per-row returns
    R_k (n_list, M*rows) of every list entry, in list order, and the autograd gradient of sum_k w_k (-mean R_k) with
    respect to the policy.  full_bptt = 0: a_1..a_n come from a detached copy of the policy (policy_for_rollout,
    mpg_learner.py:422); q_net = -1: no bootstrap (AMPC)."""
    from oracle import mpg_oracle as O
    nets = O.Nets(w, len(w) == 6, dtype)
    a1 = copy.copy(args)
    a1.M = 1                                  # the M tiles as rows: row m * rows + i starts from obs[i] with noise column m * rows + i
    obs_t = np.tile(np.asarray(obs), (M, 1))
    w_rest = nets.policy if full_bptt else [x.detach() for x in nets.policy]
    w_q = None if q_net < 0 else getattr(nets, Q_NETS[q_net])
    ret = O.rollout(a1, dtype, nets.policy, w_rest, w_q, O.to_t(obs_t, dtype),
                    None if noise is None else O.to_t(noise, dtype), max(lst))
    rows = torch.stack([ret[k] for k in lst])
    loss = sum(wk * -ret[k].mean() for k, wk in zip(lst, list_w))
    grad = torch.autograd.grad(loss, nets.policy)
    return rows.detach().numpy(), np.concatenate([g.numpy().ravel() for g in grad])


def _check_policy_grad(e, args, w, obs, noise, lst, list_w, label, M=1, full_bptt=True, q_net=_lib.NET_Q1,
                       tol_rows=TOL_STATE, tol_grad=TOL_GRAD):
    g, ret = e.policy_grad(e.dev(obs), lst, list_w, M=M, full_bptt=full_bptt, q_net=q_net,
                           noise=None if noise is None else e.dev(noise))
    rows_ref, g_ref = oracle_policy_grad(args, w, obs, noise, lst, list_w, M, full_bptt, q_net)
    got = ret.cpu().numpy()
    errs = dict(rows=max(rel_l2(got[k], rows_ref[k]) for k in range(len(lst))), grad=rel_l2(g.cpu().numpy(), g_ref))
    print(label, 'backend', e.backend, errs)
    assert np.isfinite(got).all(), 'a returns row was not written'
    assert errs['rows'] <= tol_rows, errs
    assert errs['grad'] <= tol_grad, errs
    return rows_ref, errs


def _check_closed_loop(e, args, w_pi, obs, noise, n, label, spread_k=None):
    """Worst per-step norm-relative error of the closed-loop obs / rewards / actions.  spread_k = (K_ffma, K_tc): a
    quantity may also stay within K x the oracle's own fp32-vs-fp64 distance on the same inputs (the sensitivity of
    the problem), for cases whose fp32 reference alone comes near the fixed bar."""
    from oracle import mpg_oracle as O
    _, t_obs, t_rew, t_act = e.rollout_forward(e.dev(obs), [n], noise=None if noise is None else e.dev(noise),
                                               want_traj=True)
    ref = O.closed_loop(args, w_pi, obs, noise, n, torch.float64)
    got = (t_obs.cpu().numpy(), t_rew.cpu().numpy(), t_act.cpu().numpy())
    worst = lambda xs, ys: max(rel_l2(x, y) for x, y in zip(xs, ys))
    errs = {k: worst(g, r) for k, g, r in zip(('obs', 'rew', 'act'), got, ref)}
    bar = dict.fromkeys(errs, TOL_STATE)
    if spread_k is not None:
        ref32 = O.closed_loop(args, w_pi, obs, noise, n, torch.float32)
        K = spread_k[e.backend]
        for k, r32, r64 in zip(('obs', 'rew', 'act'), ref32, ref):
            errs['spread_' + k] = worst(r32, r64)
            bar[k] = max(TOL_STATE, K * errs['spread_' + k])
    print(label, 'closed loop, backend', e.backend, errs)
    for k in bar:
        assert errs[k] <= bar[k], (k, errs)


def _inputs(args, B, n, M=1, seed=0, H=256, double_q=False):
    w = synthetic.make_policy_with_qs_weights(500 + seed, args.obs_dim, args.act_dim, H, double_q=double_q)
    rng = np.random.default_rng(600 + seed)
    obs = synthetic.make_obs(rng, args.env_id, B, args.num_future_data)
    noise = synthetic.make_noise(rng, n, B * M) if n else None
    return w, obs, noise


def _pt_args(alg, nfd=0, seed=0, **kw):
    """PathTracking args with non-unit random scales on the future columns (preprocessor 'scale' mode)."""
    args = default_args(alg, PT, num_future_data=nfd, **kw)
    rng = np.random.default_rng(700 + nfd + seed)
    args.obs_scale = list(args.obs_scale[:6]) + [float(x) for x in rng.uniform(0.3, 3.0, nfd)]
    return args


# ------------------------------------------------------------------------------------------------
# num_future_data sweep: the tensor-core first-layer image is full at nfd = 7 (13 + 2 Q inputs, bias at K = 15),
# nfd = 8 moves the handle to FFMA, nfd = 10 is the widest FFMA Q input (18 of MAX_IN = 20)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('nfd', [3, 7, 8, 10])
@pytest.mark.parametrize('alg', ['NADP', 'MPG-v2'])
def test_nfd_sweep_vs_oracle(alg, nfd, backend):
    B, n = 1024, 25
    args = _pt_args(alg, nfd, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=nfd, double_q=(alg == 'MPG-v2'))
    from mpg_b200.policy import PolicyWithQs
    assert PolicyWithQs(**vars(args)).engine.tc_available() == (nfd <= 7), 'the tensor-core path covers nfd <= 7'
    _, e = _handle(args, w, backend)
    if alg == 'NADP':
        _check_policy_grad(e, args, w, obs, noise, [n], [1.0], f'nfd={nfd} NADP')
        _check_closed_loop(e, args, w[1], obs, noise, n, f'nfd={nfd}')
    else:
        _check_policy_grad(e, args, w, obs, noise, [0, n], [0.3, 0.7], f'nfd={nfd} MPG-v2 first action', full_bptt=False)


def test_ffma_h64_nfd10_full_bptt_vs_oracle():
    """H = 64 with the widest FFMA Q input: its input-gradient partials are the largest user of the shared slab."""
    B, n, H = 1024, 25, 64
    args = _pt_args('NADP', 10, replay_batch_size=B, value_num_hidden_units=H, policy_num_hidden_units=H)
    w, obs, noise = _inputs(args, B, n, seed=64, H=H)
    _, e = _handle(args, w, 'ffma')
    assert not e.tc_available()
    _check_policy_grad(e, args, w, obs, noise, [0, 9, n], [0.2, 0.3, 0.5], 'H=64 nfd=10')
    _check_closed_loop(e, args, w[1], obs, noise, n, 'H=64 nfd=10')


# ------------------------------------------------------------------------------------------------
# policy heads: policy_out_activation x action_range (tanh / linear x None / range)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('out_act,action_range', [('tanh', None), ('tanh', 2.0), ('linear', None), ('linear', 1.5)])
@pytest.mark.parametrize('env_id', [PT, IP])
def test_policy_heads_vs_oracle(env_id, out_act, action_range, backend):
    """On the cart-pole these weights start with small actions (mean |a_0| ~ 0.01, the output layer's sum cancels):
    there the fp32 oracle itself is 3.7e-6 from fp64 on a_0, the FFMA path measures 2.8e-6 and the tensor-core path,
    whose forward contractions run on fp16 pairs (DESIGN 4.3), 1.13e-5 on every head.  The closed loop of that env is
    therefore held to max(1e-5, K x that spread) with K = 2 (FFMA) / 8 (tensor cores); PathTracking to 1e-5 itself."""
    B, n = 512, 25 if env_id == PT else 15
    args = default_args('NADP', env_id, replay_batch_size=B, policy_out_activation=out_act, action_range=action_range)
    w, obs, noise = _inputs(args, B, n, seed=11)
    _, e = _handle(args, w, backend)
    label = f'{env_id} head {out_act}/{action_range}'
    _check_closed_loop(e, args, w[1], obs, noise, n, label, spread_k=None if env_id == PT else (2.0, 8.0))
    _check_policy_grad(e, args, w, obs, noise, [0, n], [0.4, 0.6], label)


# ------------------------------------------------------------------------------------------------
# reward preprocessing and discount, in the rollout and in the evaluation entry points
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('gamma', [1.0, 0.9])
def test_reward_shift_scale_and_discount_vs_oracle(gamma, backend):
    """rew_shift != 0 enters every reward of a return (rho (r + shift)); a wrong placement would show in the rows."""
    from oracle import mpg_oracle as O
    B, n = 1000, 25
    args = default_args('MPG-v2', PT, replay_batch_size=B, rew_shift=0.37, rew_scale=0.05, gamma=gamma)
    w, obs, noise = _inputs(args, B, n, seed=21, double_q=True)
    pol, e = _handle(args, w, backend)
    label = f'shift/scale gamma={gamma}'
    _check_policy_grad(e, args, w, obs, noise, [0, 10, n], [0.2, 0.3, 0.5], label)
    _check_policy_grad(e, args, w, obs, noise, [0, n], [0.5, 0.5], label + ' first action', full_bptt=False)
    # evaluation entry points on a replay batch
    o, act, rew, o1, _ = make_batch(22, PT, B, 0)
    nets = O.Nets(w, True, torch.float64)
    t = lambda x: O.to_t(x, torch.float64)
    sigma = t(args.obs_scale)
    errs = {}
    with torch.no_grad():
        p, p1 = t(o) * sigma, t(o1) * sigma
        prew = (t(rew) + args.rew_shift) * args.rew_scale
        a1 = O.policy_action(nets.policy_t, p1, 'tanh', None)
        q1t, q2t = O.q_value(nets.Q1_t, p1, a1), O.q_value(nets.Q2_t, p1, a1)
        ref = dict(target_double=prew + gamma * torch.minimum(q1t, q2t), target_single=prew + gamma * q1t,
                   td=O.td_error(args, nets, [o, act, rew, o1], torch.float64),
                   act=O.policy_action(nets.policy, p, 'tanh', None),
                   act_target=O.policy_action(nets.policy_t, p, 'tanh', None))
        base = np.random.default_rng(23).standard_normal(B).astype(np.float32)
        a_t = O.policy_action(nets.policy_t, p, 'tanh', None)
        ref['bootstrap'] = t(base) + gamma ** 7 * O.q_value(nets.Q1_t, p, a_t)
    got = dict(target_double=e.q_target(True, e.dev(rew), e.dev(o1)), target_single=e.q_target(False, e.dev(rew), e.dev(o1)),
               td=e.td_error(e.dev(o), e.dev(act), e.dev(rew), e.dev(o1)),
               act=e.policy_forward(_lib.NET_POLICY, e.dev(o)), act_target=e.policy_forward(_lib.NET_POLICY_TARGET, e.dev(o)),
               bootstrap=e.q_bootstrap(e.dev(base), gamma ** 7, e.dev(o)))
    for k in ref:
        errs[k] = rel_l2(got[k].cpu().numpy(), ref[k].numpy())
    print(label, 'evaluations, backend', e.backend, errs)
    # the TD error is a difference of two Q values: held to the suite's 2e-5 bar for scalar results of that kind
    for k, v in errs.items():
        assert v <= (2e-5 if k == 'td' else TOL_STATE), errs


# ------------------------------------------------------------------------------------------------
# no bootstrap (q_net = -1, AMPC)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('full_bptt', [True, False])
def test_no_bootstrap_policy_grad_vs_oracle(full_bptt, backend):
    B, n = 1024, 25
    args = default_args('NADP', PT, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=31)
    _, e = _handle(args, w, backend)
    _check_policy_grad(e, args, w, obs, noise, [5, n], [0.4, 0.6], f'no bootstrap full_bptt={full_bptt}',
                       full_bptt=full_bptt, q_net=-1)


# ------------------------------------------------------------------------------------------------
# rollout lists: order, zero and negative weights, all eight entries, repeated entries
# ------------------------------------------------------------------------------------------------
LISTS = {
    'unsorted': ([25, 0, 7], [0.5, 0.2, 0.3]),
    'zero_weights': ([0, 7, 25], [0.0, 0.6, 0.0]),
    'negative_weights': ([0, 7, 25], [-0.3, 0.8, 0.5]),
    'eight_entries': ([0, 1, 3, 5, 8, 13, 21, 25], [0.05, 0.1, 0.1, 0.15, 0.1, 0.2, 0.1, 0.2]),
    'dup_half_half': ([25, 25], [0.5, 0.5]),
    'dup_half_zero': ([25, 25], [0.5, 0.0]),
    'dup_zero_half': ([25, 25], [0.0, 0.5]),
    'dup_inner': ([0, 7, 7], [0.2, 0.5, 0.3]),
    'dup_inner_half_zero': ([7, 7, 25], [0.5, 0.0, 0.5]),   # tensor cores: the h2 prefetch schedule of step 7 and 8
    'dup_first': ([0, 0, 25], [0.3, 0.3, 0.4]),
}


@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('full_bptt', [True, False])
@pytest.mark.parametrize('case', list(LISTS))
def test_rollout_lists_vs_oracle(case, full_bptt, backend):
    """Every returns row of the list, from the gradient kernel and from the forward-only kernel, and the gradient of
    sum_k w_k (-mean R_k): repeated entries are independent terms (the reference's tf.stack over the list)."""
    lst, lw = LISTS[case]
    B, n = 512, max(lst)
    args = default_args('NADP', PT, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=41)
    _, e = _handle(args, w, backend)
    rows_ref, _ = _check_policy_grad(e, args, w, obs, noise, lst, lw, f'list {case} full_bptt={full_bptt}',
                                     full_bptt=full_bptt)
    fwd = e.rollout_forward(e.dev(obs), lst, noise=e.dev(noise)).cpu().numpy()
    err = max(rel_l2(fwd[k], rows_ref[k]) for k in range(len(lst)))
    print(f'list {case}', 'forward-only rows, backend', e.backend, err)
    assert np.isfinite(fwd).all() and err <= TOL_STATE, err


# ------------------------------------------------------------------------------------------------
# long horizon: list steps on both sides of the tensor-core kernel's 64-bit list masks
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('full_bptt', [True, False])
def test_long_horizon_70_vs_oracle(full_bptt, backend):
    """n = 70 with list [0, 63, 64, 70]: steps 64 and 70 take the scan path of the tensor-core kernel."""
    B, n = 512, 70
    args = default_args('NADP', PT, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=51)
    _, e = _handle(args, w, backend)
    _check_policy_grad(e, args, w, obs, noise, [0, 63, 64, 70], [0.1, 0.2, 0.3, 0.4], f'n=70 full_bptt={full_bptt}',
                       full_bptt=full_bptt)
    if full_bptt:
        _check_closed_loop(e, args, w[1], obs, noise, n, 'n=70')


# ------------------------------------------------------------------------------------------------
# M = 3, ragged last tile, more tiles than SMs (tensor cores: full waves + tail wave with M > 1)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('backend', BACKENDS)
def test_m3_ragged_multi_wave_vs_oracle(backend):
    B, n, M = 6701, 3, 3
    args = default_args('NADP', PT, replay_batch_size=B, M=M)
    w, obs, noise = _inputs(args, B, n, M=M, seed=61)
    _, e = _handle(args, w, backend)
    assert (B * M) % 128 != 0 and (B * M + 127) // 128 > e.num_sms, 'the case is meant to exceed one wave of tiles'
    _check_policy_grad(e, args, w, obs, noise, [0, n], [0.4, 0.6], 'M=3 ragged multi-wave', M=M)


# ------------------------------------------------------------------------------------------------
# return statistics (mpg_returns_stats / mpg_returns_tile_mean) against numpy fp64
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('rows', [1, 37, 1000])
def test_returns_stats_vs_numpy(rows):
    from mpg_b200.engine import Engine
    n_list, M = 8, 3
    e = Engine(**vars(default_args('NADP', PT)))
    rng = np.random.default_rng(71 + rows)
    ret = (rng.standard_normal((n_list, M * rows)) - 3.0).astype(np.float32)
    mean = ret.astype(np.float64).reshape(n_list, M, rows).mean(1)
    ref = np.concatenate([mean.sum(1), (mean ** 2).sum(1)])
    stats = e.returns_stats(e.dev(ret), rows, M).cpu().numpy()
    tile_mean = e.returns_tile_mean(e.dev(ret), rows, M).cpu().numpy()
    errs = dict(sum=rel_l2(stats[:n_list], ref[:n_list]), sumsq=rel_l2(stats[n_list:], ref[n_list:]),
                tile_mean=rel_l2(tile_mean, mean))
    print('returns stats rows', rows, errs)
    assert max(errs.values()) <= TOL_STATE, errs


# ------------------------------------------------------------------------------------------------
# model adjoint (mpg_model_step_bwd) at nfd > 0: the future columns feed back into delta_y
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nfd', [0, 2, 10])
def test_model_step_bwd_vs_oracle_autograd(nfd):
    from oracle import mpg_oracle as O
    from mpg_b200.engine import Engine
    B = 256
    args = default_args('NADP', PT, num_future_data=nfd)
    e = Engine(**vars(args))
    rng = np.random.default_rng(81 + nfd)
    obs0 = synthetic.make_obs(rng, PT, B, nfd)
    state = e.model_reset(e.dev(obs0))
    act = rng.uniform(-1, 1, (B, 2)).astype(np.float32)
    eps = synthetic.make_noise(rng, 1, B)[0]
    g_obs = rng.standard_normal((B, args.obs_dim)).astype(np.float32)
    g_rew = rng.standard_normal(B).astype(np.float32)
    g_state = rng.standard_normal((B, 6)).astype(np.float32)
    gs, ga = e.model_step_bwd(state, e.dev(act), e.dev(eps), e.dev(g_obs), e.dev(g_rew), e.dev(g_state))
    m = O.PathTrackingModel(num_future_data=nfd)
    s64 = torch.tensor(state.cpu().numpy(), dtype=torch.float64, requires_grad=True)
    a64 = torch.tensor(act, dtype=torch.float64, requires_grad=True)
    m.s = s64
    o, r = m.rollout_out(a64, torch.tensor(eps, dtype=torch.float64))
    t = lambda x: torch.tensor(x, dtype=torch.float64)
    loss = (o * t(g_obs)).sum() + (r * t(g_rew)).sum() + (m.s * t(g_state)).sum()
    ref_s, ref_a = torch.autograd.grad(loss, [s64, a64])
    errs = dict(g_state_in=rel_l2(gs.cpu().numpy(), ref_s.numpy()), g_action=rel_l2(ga.cpu().numpy(), ref_a.numpy()))
    print('model_step_bwd nfd', nfd, errs)
    assert errs['g_state_in'] <= TOL_GRAD and errs['g_action'] <= TOL_GRAD, errs
