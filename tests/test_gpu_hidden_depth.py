"""1 and 3 hidden layers (value_num_hidden_layers == policy_num_hidden_layers) on the fp32 FFMA kernels at H = 64 / 128 /
256; the tensor-core backend is built for 2 hidden layers only.  The reference has golden vectors for 2 layers only, so
the truth here is the fp64 oracle run at the same depth, held to the suite's bars: states / rewards / actions 1e-5 per
step, gradients 1e-4, scalars 2e-5.  That oracle is first pinned on the CPU: its MLP against an independent
torch.nn.Sequential, its gradients against central finite differences.

The oracle (oracle/mpg_oracle.py) evaluates every MLP through its module-level mlp(), which is MLPNet.call at the
reference default of 2 hidden layers; `oracle_depth` swaps in MLPNet.call for any depth (a loop over the hidden layers,
model.py:39-43) for the duration of a comparison, so every oracle routine runs the depth under test."""
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
DEPTHS = [1, 3]
WIDTHS = [64, 128, 256]
HIDDEN_FN = {'elu': F.elu, 'relu': F.relu, 'tanh': torch.tanh}


def depth_mlp(act='elu'):
    """MLPNet.call (model.py:39-43) for weights [W1,b1,..,WL,bL,Wout,bout]: len(w) // 2 - 1 hidden layers."""
    f = HIDDEN_FN[act]

    def mlp(w, x, out_act='linear'):
        h = x
        for i in range(len(w) // 2 - 1):
            h = f(h @ w[2 * i] + w[2 * i + 1])
        y = h @ w[-2] + w[-1]
        return torch.tanh(y) if out_act == 'tanh' else y
    return mlp


@contextlib.contextmanager
def oracle_depth(act='elu'):
    from oracle import mpg_oracle as O
    saved = O.mlp
    O.mlp = depth_mlp(act)
    try:
        yield O
    finally:
        O.mlp = saved


def _args(alg, env_id, H, L, act='elu', **kw):
    return default_args(alg, env_id, value_num_hidden_units=H, policy_num_hidden_units=H, value_num_hidden_layers=L,
                        policy_num_hidden_layers=L, value_hidden_activation=act, policy_hidden_activation=act, **kw)


def _weights(seed, args, H, L, double_q):
    return synthetic.make_policy_with_qs_weights(seed, args.obs_dim, args.act_dim, H, double_q=double_q, layers=L)


def _flat(grads):
    return np.concatenate([np.asarray(g, np.float64).ravel() for g in grads])


def _unclip(g, norm, clip):
    return g * max(norm, clip) / clip


def _ffma(engine, L):
    from mpg_b200.engine import BACKEND_FFMA
    assert engine.hidden_layers == L and engine.lib.mpg_hidden_layers(engine.h) == L
    assert engine.backend == BACKEND_FFMA and not engine.tc_available()


def _learner(kind, args, weights):
    from mpg_b200.learners import MPGLearner, NADPLearner
    from mpg_b200.policy import PolicyWithQs
    learner = (NADPLearner if kind == 'nadp' else MPGLearner)(PolicyWithQs, args)
    learner.set_weights(weights)
    _ffma(learner.engine, args.policy_num_hidden_layers)
    return learner


def _policy(args, weights):
    from mpg_b200.policy import PolicyWithQs
    pol = PolicyWithQs(**vars(args))
    if weights is not None:
        pol.set_weights(weights)
    _ffma(pol.engine, args.policy_num_hidden_layers)
    return pol


# ------------------------------------------------------------------------------------------------
# CPU: the depth-general oracle, the depth checks, the weight lists
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('L', DEPTHS)
def test_depth_mlp_matches_sequential(L):
    """The loop over hidden layers equals torch.nn.Sequential(Linear, ELU, .., Linear) built from the Keras (in, out)
    arrays (Linear holds (out, in)): catches an order or transposition error in the reference MLP."""
    H, B = 32, 40
    w = synthetic.make_mlp_weights(np.random.default_rng(L), 9, H, 4, layers=L)
    assert [np.shape(a) for a in w] == [(9, H), (H,)] + [(H, H), (H,)] * (L - 1) + [(H, 4), (4,)]
    layers = []
    for i in range(L + 1):
        lin = torch.nn.Linear(*np.shape(w[2 * i]), dtype=torch.float64)
        with torch.no_grad():
            lin.weight.copy_(torch.as_tensor(w[2 * i].T, dtype=torch.float64))
            lin.bias.copy_(torch.as_tensor(w[2 * i + 1], dtype=torch.float64))
        layers += [lin, torch.nn.ELU()] if i < L else [lin]
    seq = torch.nn.Sequential(*layers)
    x = torch.as_tensor(np.random.default_rng(7).standard_normal((B, 9)))
    w64 = [torch.as_tensor(a, dtype=torch.float64) for a in w]
    with torch.no_grad():
        ref = seq(x)
        assert torch.allclose(depth_mlp()(w64, x), ref, rtol=1e-12, atol=1e-12)
        assert torch.allclose(depth_mlp()(w64, x, 'tanh'), torch.tanh(ref), rtol=1e-12, atol=1e-12)


def test_depth_mlp_is_the_oracle_at_two_layers():
    from oracle import mpg_oracle as O
    w = [torch.as_tensor(a, dtype=torch.float64) for a in synthetic.make_mlp_weights(np.random.default_rng(1), 8, 16, 2)]
    x = torch.as_tensor(np.random.default_rng(2).standard_normal((10, 8)))
    assert torch.equal(depth_mlp()(w, x), O.mlp(w, x))


@pytest.mark.parametrize('L', DEPTHS)
def test_oracle_gradients_match_finite_differences(L):
    """Policy gradient of the model rollout (NADP loss -R_n) and Q regression gradient of the depth-L oracle against
    central differences in fp64 (as test_gpu_activation.test_oracle_gradients_match_finite_differences)."""
    H, B, n, h = 32, 6, 3, 1e-6
    args = _args('NADP', PT, H, L, replay_batch_size=B)
    w = _weights(3, args, H, L, False)
    rng = np.random.default_rng(4)
    with oracle_depth() as O:
        obs = O.to_t(synthetic.make_obs(rng, PT, B), torch.float64)
        noise = O.to_t(synthetic.make_noise(rng, n, B), torch.float64)
        act_in = O.to_t(rng.uniform(-1, 1, (B, args.act_dim)), torch.float64)
        target = O.to_t(rng.standard_normal(B), torch.float64)
        sigma = O.to_t(args.obs_scale, torch.float64)
        nets = O.Nets(w, False, torch.float64)
        assert len(nets.policy) == 2 * (L + 1)

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
                vals = []
                for s in (h, -h):
                    pw = [p.detach().clone(memory_format=torch.contiguous_format) for p in params]
                    pw[i].view(-1)[j] += s
                    with torch.no_grad():
                        vals.append(float(loss_fn(pw)))
                fd = (vals[0] - vals[1]) / (2 * h)
                an = float(grads[i].reshape(-1)[j])
                assert abs(fd - an) <= 1e-6 * max(abs(an), 1e-3), (i, j, fd, an)
                checked += 1
        assert checked == 48


def test_depth_check_precedes_the_device():
    from mpg_b200 import parallel
    from mpg_b200.policy import PolicyWithQs
    for L in (0, 4):
        with pytest.raises(NotImplementedError, match='1 / 2 / 3'):
            PolicyWithQs(**vars(_args('NADP', PT, 64, L)))
    with pytest.raises(NotImplementedError, match='must be equal'):
        PolicyWithQs(**vars(default_args('NADP', PT, value_num_hidden_layers=1, policy_num_hidden_layers=3)))
    for L in DEPTHS:
        shapes = parallel.net_shapes(6, 2, 'q', 64, L)
        assert shapes == [(8, 64), (64,)] + [(64, 64), (64,)] * (L - 1) + [(64, 1), (1,)]
        nets = ['q', 'pi']
        sizes = [sum(int(np.prod(s)) for s in parallel.net_shapes(6, 2, k, 64, L)) for k in nets]
        flat = np.arange(sum(sizes), dtype=np.float32)
        out = parallel.split_flat(flat, 6, 2, nets, 64, L)
        assert [a.shape for a in out] == shapes + parallel.net_shapes(6, 2, 'pi', 64, L)
        assert np.array_equal(np.concatenate([a.ravel() for a in out]), flat)
    if torch.cuda.is_available():
        return
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        PolicyWithQs(**vars(_args('NADP', PT, 64, 3)))


def test_weight_draws_at_two_layers_are_unchanged():
    """make_mlp_weights draws in list order: at the default depth a seed gives the weights it always gave."""
    rng, ref_rng = np.random.default_rng(8), np.random.default_rng(8)
    w = synthetic.make_mlp_weights(rng, 7, 64, 3)
    g = np.sqrt(2.0)
    ref = [synthetic.orthogonal(ref_rng, 7, 64, g), (0.05 * ref_rng.standard_normal(64)).astype(np.float32),
           synthetic.orthogonal(ref_rng, 64, 64, g), (0.05 * ref_rng.standard_normal(64)).astype(np.float32),
           synthetic.orthogonal(ref_rng, 64, 3, 1.0), (0.05 * ref_rng.standard_normal(3)).astype(np.float32)]
    assert len(w) == 6 and all(np.array_equal(a, b) for a, b in zip(w, ref))
    w3 = synthetic.make_mlp_weights(np.random.default_rng(8), 7, 64, 3, layers=3)
    assert all(np.array_equal(a, b) for a, b in zip(w3[:4], ref[:4]))


# ------------------------------------------------------------------------------------------------
# compute_gradient against the oracle
# ------------------------------------------------------------------------------------------------
def _nadp_vs_oracle(env_id, B, n, H, L, act='elu', seed=0, per_row=False):
    from tests.test_gpu_parity import _row_returns_vs_oracle
    args = _args('NADP', env_id, H, L, act, replay_batch_size=B, num_rollout_list_for_policy_update=[n],
                 num_rollout_list_for_q_estimation=[n])
    w = _weights(100 + seed, args, H, L, False)
    batch = make_batch(200 + seed, env_id, B, 0)
    rng = np.random.default_rng(300 + seed)
    nq, npol = synthetic.make_noise(rng, n, B), synthetic.make_noise(rng, n, B)
    learner = _learner('nadp', args, w)
    learner.set_rollout_noise(nq, npol)
    grads = learner.compute_gradient(batch, None, None, 0)
    assert len(grads) == 4 * (L + 1) and grads[-2].shape == (H, 2 * args.act_dim)
    flat = _flat(grads)
    st = learner.get_stats()
    with oracle_depth(act) as O:
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
    print('NADP', env_id, B, n, H, L, act, errs)
    assert errs['q'] <= TOL_GRAD and errs['p'] <= TOL_GRAD and errs['clipped'] <= TOL_GRAD, errs
    return learner


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
@pytest.mark.parametrize('B', [1, 300, 2048])
def test_nadp_pathtracking_vs_oracle(B, L, H):
    _nadp_vs_oracle(PT, B, 25, H, L, per_row=(B < 16))


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_nadp_multi_wave_vs_oracle(L, H):
    """20,011 rows = 313 tiles: several tiles per CTA, so the register accumulators of every layer carry across tiles."""
    learner = _nadp_vs_oracle(PT, 20011, 3, H, L, seed=9, per_row=True)
    assert learner.engine.num_sms < 313


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_nadp_cart_pole_vs_oracle(L, H):
    _nadp_vs_oracle(IP, 200, 25, H, L)


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_nadp_double_pendulum_short_horizon_vs_oracle(L, H):
    # the falling double pendulum amplifies rounding beyond a few steps (tests/test_gpu_parity.py): n = 3
    _nadp_vs_oracle(IDP, 128, 3, H, L)


@pytest.mark.gpu
@pytest.mark.parametrize('L,H,act', [(3, 128, 'relu'), (1, 128, 'tanh')], ids=['relu-L3', 'tanh-L1'])
def test_nadp_other_activations_vs_oracle(L, H, act):
    _nadp_vs_oracle(PT, 300, 25, H, L, act)


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_mpg_v2_vs_oracle(L, H):
    """MPG-v2 with a 3-entry rollout list (first-action gradient mode): clipped double-Q targets, both Q regressions,
    the weighted policy loss and the TD errors of prioritized replay."""
    B, ite = 160, 4000
    args = _args('MPG-v2', PT, H, L, replay_batch_size=B, num_rollout_list_for_policy_update=[0, 10, 25],
                 buffer_type='priority', sample_num_in_learner=None)
    w = _weights(7, args, H, L, True)
    batch = make_batch(8, PT, B, 0)
    npol = synthetic.make_noise(np.random.default_rng(9), 25, B)
    learner = _learner('mpg', args, w)
    learner.set_rollout_noise(None, npol)
    flat = _flat(learner.compute_gradient(batch, None, None, ite))
    st = learner.get_stats()
    with oracle_depth() as O:
        ref = O.mpg_compute_gradient(args, w, batch, npol, ite, torch.float64)
    nQ = ref['q_grad1'].size
    errs = dict(clipped=rel_l2(flat, ref['compute_gradient']),
                p=rel_l2(_unclip(flat[2 * nQ:], st['policy_gradient_norm'], args.gradient_clip_norm), ref['policy_grad']),
                targets=rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), ref['batch_targets']),
                td=rel_l2(learner.get_info_for_buffer()['td_error'], ref['td_error']),
                total_loss=rel_l2(st['policy_total_loss'], ref['total_loss']),
                value_mean=rel_l2(st['value_mean'], ref['value_mean']),
                q1=rel_l2(st['q_loss1'], ref['q_loss1']), q2=rel_l2(st['q_loss2'], ref['q_loss2']))
    print('MPG-v2', H, L, errs)
    assert errs['clipped'] <= TOL_GRAD and errs['p'] <= TOL_GRAD, errs
    for k in ('targets', 'td', 'total_loss', 'value_mean', 'q1', 'q2'):
        assert errs[k] <= TOL_SCALAR, errs


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_mpg_v1_real_env_n_step_target_vs_oracle(L, H):
    """compute_n_step_target (mpg_learner.py:153-169): 25 steps of the real PathTracking environment under the policy,
    bootstrapped with Q1_target, against the oracle's n-step target."""
    B, T = 300, 25
    args = _args('MPG-v1', PT, H, L, replay_batch_size=B, sample_num_in_learner=T)
    w = _weights(5, args, H, L, False)
    batch = make_batch(6, PT, B, 0)
    learner = _learner('mpg', args, w)
    learner.get_batch_data(batch, None, None)
    with oracle_depth() as O:
        ref, _ = O.mpg_v1_n_step_target(args, w, batch, T, torch.float64)
    err = rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), ref)
    print('MPG-v1 n-step target', H, L, err)
    assert err <= TOL_SCALAR, err


# ------------------------------------------------------------------------------------------------
# closed-loop trajectories, forward entry points, Q regression
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_closed_loop_trajectories_vs_oracle(L, H):
    """Observations, rewards and actions of every step of mpg_rollout_forward <= 1e-5 norm-relative."""
    B, n = 512, 25
    args = _args('NADP', PT, H, L, replay_batch_size=B)
    w = _weights(40, args, H, L, False)
    pol = _policy(args, w)
    e = pol.engine
    rng = np.random.default_rng(60)
    obs0 = synthetic.make_obs(rng, PT, B)
    noise = synthetic.make_noise(rng, n, B)
    _, t_obs, t_rew, t_act = e.rollout_forward(e.dev(obs0), [n], noise=e.dev(noise), want_traj=True)
    with oracle_depth() as O:
        ro, rr, ra = O.closed_loop(args, w[1], obs0, noise, n, torch.float64)
    errs = dict(obs=max(rel_l2(t_obs[t].cpu().numpy(), ro[t]) for t in range(n)),
                rew=max(rel_l2(t_rew[t].cpu().numpy(), rr[t]) for t in range(n)),
                act=max(rel_l2(t_act[t].cpu().numpy(), ra[t]) for t in range(n + 1)))
    print('closed loop', H, L, errs)
    assert max(errs.values()) <= TOL_STATE, errs


@pytest.mark.gpu
@pytest.mark.parametrize('H', WIDTHS)
@pytest.mark.parametrize('L', DEPTHS)
def test_forward_entry_points_and_q_grad_vs_oracle(L, H):
    """compute_action / compute_Q1, mpg_q_target (double Q), mpg_td_error, mpg_q_bootstrap and the Q-regression
    gradient (mpg_q_grad) against the oracle's networks."""
    from mpg_b200 import _lib
    B = 1000
    args = _args('MPG-v2', PT, H, L, replay_batch_size=B)
    w = _weights(3, args, H, L, True)
    pol = _policy(args, w)
    e = pol.engine
    rng = np.random.default_rng(4)
    obs, obs1 = synthetic.make_obs(rng, PT, B), synthetic.make_obs(rng, PT, B)
    sigma = np.asarray(args.obs_scale, np.float32)
    act_in = rng.uniform(-1, 1, (B, args.act_dim)).astype(np.float32)
    rew = (-np.abs(rng.standard_normal(B))).astype(np.float32)
    target = rng.standard_normal(B).astype(np.float32)
    got_a, _ = pol.compute_action(obs * sigma)
    got_q = pol.compute_Q1(obs * sigma, act_in)
    got_tgt = e.q_target(True, e.dev(rew), e.dev(obs1))
    got_td = e.td_error(e.dev(obs), e.dev(act_in), e.dev(rew), e.dev(obs1))
    got_bs = e.q_bootstrap(e.dev(rew), 0.7, e.dev(obs))
    got_g, got_loss = e.q_grad(_lib.NET_Q1, e.dev(obs), e.dev(act_in), e.dev(target))
    assert got_g.numel() == e.param_count(_lib.NET_Q1)
    with oracle_depth() as O:
        nets = O.Nets(w, True, torch.float64)
        t64 = lambda x: O.to_t(x, torch.float64)   # noqa: E731
        p, p1 = t64(obs) * t64(sigma), t64(obs1) * t64(sigma)
        q_pred = O.q_value(nets.Q1, p, t64(act_in))
        loss = 0.5 * torch.mean((q_pred - t64(target)) ** 2)
        ref_g = np.concatenate([x.numpy().ravel() for x in torch.autograd.grad(loss, nets.Q1)])
        with torch.no_grad():
            prew = (t64(rew) + args.rew_shift) * args.rew_scale
            a1 = O.policy_action(nets.policy_t, p1, args.policy_out_activation, args.action_range)
            a0 = O.policy_action(nets.policy_t, p, args.policy_out_activation, args.action_range)
            ref = dict(
                act=O.policy_action(nets.policy, p, args.policy_out_activation, args.action_range),
                q=q_pred.detach(),
                tgt=prew + args.gamma * torch.minimum(O.q_value(nets.Q1_t, p1, a1), O.q_value(nets.Q2_t, p1, a1)),
                td=prew + args.gamma * O.q_value(nets.Q1_t, p1, a1) - q_pred.detach(),
                bs=t64(rew) + 0.7 * O.q_value(nets.Q1_t, p, a0))
    got = dict(act=got_a, q=got_q, tgt=got_tgt, td=got_td, bs=got_bs)
    errs = {k: rel_l2(got[k].cpu().numpy(), ref[k].numpy()) for k in ref}
    errs['q_grad'] = rel_l2(got_g.cpu().numpy(), ref_g)
    errs['q_loss'] = rel_l2(float(got_loss.item()) / B, float(loss.item()))
    print('forward entry points', H, L, errs)
    assert errs['act'] <= TOL_STATE and errs['q'] <= TOL_STATE, errs
    for k in ('tgt', 'td', 'bs', 'q_loss'):
        assert errs[k] <= TOL_SCALAR, errs
    assert errs['q_grad'] <= TOL_GRAD, errs


# ------------------------------------------------------------------------------------------------
# optimiser step and checkpoints
# ------------------------------------------------------------------------------------------------
def _apply_gradients_ref(O, weights, states, iteration, grads, double_q, delay_update, tau, per_net):
    """O.apply_gradients (policy.py:123-171) for nets of `per_net` arrays each."""
    w = [[np.asarray(a, np.float64) for a in net] for net in weights]
    g = [np.asarray(a, np.float64) for a in grads]
    nq = 2 if double_q else 1
    for i in range(nq):
        w[i] = states[f'Q{i + 1}'].apply(w[i], g[per_net * i: per_net * (i + 1)])
    if iteration % delay_update == 0:
        w[nq] = states['policy'].apply(w[nq], g[per_net * nq: per_net * (nq + 1)])
        nm = nq + 1
        for i in range(nm):
            w[nm + i] = [tau * s_ + (1.0 - tau) * t_ for s_, t_ in zip(w[i], w[nm + i])]
    return w


@pytest.mark.gpu
@pytest.mark.parametrize('version', ['MPG-v2', 'NADP'])
def test_apply_gradients_vs_oracle_three_layers(version):
    """Keras-Adam + delayed policy update + Polyak targets at L = 3, H = 128: every step re-packs both hidden -> hidden
    images (and their transposes) that the kernels then read."""
    from oracle import mpg_oracle as O
    H, L = 128, 3
    dq = version == 'MPG-v2'
    args = _args(version, PT, H, L, delay_update=2)
    w0 = _weights(31, args, H, L, dq)
    pol = _policy(args, w0)
    states = {'Q1': O.AdamState(args.value_lr_schedule), 'Q2': O.AdamState(args.value_lr_schedule),
              'policy': O.AdamState(args.policy_lr_schedule)}
    w = w0
    rng = np.random.default_rng(32)
    for it in range(5):
        grads = [rng.standard_normal(np.shape(a)).astype(np.float32) * 0.1 for net in w0[: (3 if dq else 2)] for a in net]
        pol.apply_gradients(it, grads if it % 2 == 0 else torch.tensor(np.concatenate([g.ravel() for g in grads]), device='cuda'))
        w = _apply_gradients_ref(O, w, states, it, grads, dq, args.delay_update, args.tau, 2 * (L + 1))
    got = pol.get_weights()
    for net_g, net_r in zip(got, w):
        assert len(net_g) == 2 * (L + 1)
        for a, b in zip(net_g, net_r):
            assert a.shape == np.shape(b)
            assert rel_l2(a, b) <= 2e-6
    # the updated weights are what the kernels now use (policy and its target: the Polyak re-pack)
    obs = synthetic.make_obs(np.random.default_rng(1), PT, 64) * np.asarray(args.obs_scale, np.float32)
    with oracle_depth() as O2, torch.no_grad():
        for slot, k in ((2, 2 if dq else 1), (5, 5 if dq else 3)):
            got_a = pol.engine.policy_forward(slot, pol._raw(obs)).cpu().numpy()
            ref = O2.policy_action([O2.to_t(x, torch.float64) for x in w[k]], O2.to_t(obs, torch.float64), 'tanh', None)
            assert rel_l2(got_a, ref.numpy()) <= TOL_STATE


@pytest.mark.gpu
def test_save_load_weights_round_trip_three_layers(tmp_path):
    from mpg_b200.policy import PolicyWithQs
    H, L = 64, 3
    args = _args('MPG-v2', PT, H, L)
    w = _weights(12, args, H, L, True)
    a = _policy(args, w)
    grads = [np.full(np.shape(x), 0.01, np.float32) for net in w[:3] for x in net]
    a.apply_gradients(0, grads)
    a.save_weights(str(tmp_path), 3)
    b = PolicyWithQs(**vars(args))
    b.load_weights(str(tmp_path), 3)
    for net_a, net_b in zip(a.get_weights(), b.get_weights()):
        assert len(net_a) == 2 * (L + 1)
        assert all(np.array_equal(x, y) for x, y in zip(net_a, net_b))
    for s in a.model_slots:
        assert all(np.array_equal(x, y) for x, y in zip(a.engine.get_adam_state(s), b.engine.get_adam_state(s)))
    assert b.opt_iterations == a.opt_iterations


# ------------------------------------------------------------------------------------------------
# bench size: B = 65,536, n = 25, L = 3, H = 256
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bench_size_properties_and_oracle_three_layers():
    """Two identical calls are bit-identical; two half batches with global scaling add up to the full batch; the bench
    path (in-kernel Philox, full BPTT) per-row returns <= 1e-5 and gradient <= 1e-4 against the fp64 oracle."""
    from mpg_b200 import _lib
    B, n, seed, H, L = 65536, 25, 7, 256, 3
    args = _args('NADP', PT, H, L, replay_batch_size=B)
    w = _weights(0, args, H, L, False)
    obs = synthetic.make_obs(np.random.default_rng(1234), PT, B)
    e = _policy(args, w).engine
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
    assert shard <= 1e-5, shard
    g, ret = e.policy_grad(x, [n], [1.0], full_bptt=True, q_net=_lib.NET_Q1, use_philox=True, noise_seed=seed)
    grad_ref, rows = None, []
    with oracle_depth() as O:
        nets = O.Nets(w, False, torch.float64)
        for lo in range(0, B, 8192):
            hi = min(B, lo + 8192)
            noise = synthetic.philox_normal(seed, hi - lo, n, global_rows=B, row_offset=lo)
            r = O.rollout(args, torch.float64, nets.policy, nets.policy, nets.Q1, O.to_t(obs[lo:hi], torch.float64),
                          O.to_t(noise, torch.float64), n)
            gc = np.concatenate([t.numpy().ravel() for t in torch.autograd.grad(-r[n].sum() / B, nets.policy)])
            grad_ref = gc if grad_ref is None else grad_ref + gc
            rows.append(r[n].detach().numpy())
    errs = dict(rows=rel_l2(ret[0].cpu().numpy(), np.concatenate(rows)), grad=rel_l2(g.cpu().numpy(), grad_ref),
                shard=shard)
    print('bench path L=3 H=256', errs)
    assert errs['rows'] <= TOL_STATE and errs['grad'] <= TOL_GRAD, errs


# ------------------------------------------------------------------------------------------------
# C ABI
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('L', DEPTHS)
def test_depth_abi(L):
    import ctypes
    from mpg_b200 import _lib
    from mpg_b200.engine import BACKEND_TC
    H = 256
    args = _args('MPG-v2', PT, H, L)
    w = _weights(2, args, H, L, True)
    e = _policy(args, w).engine
    d_o, d_a = args.obs_dim, args.act_dim
    for net, (i, o) in ((_lib.NET_Q1, (d_o + d_a, 1)), (_lib.NET_POLICY, (d_o, 2 * d_a))):
        assert e.param_count(net) == i * H + H + (L - 1) * (H * H + H) + H * o + o
    got = e.get_net_weights(_lib.NET_POLICY)
    assert len(got) == 2 * (L + 1) and all(np.array_equal(a, b) for a, b in zip(got, w[2]))
    with pytest.raises(ValueError, match=f'expected {2 * (L + 1)} weight arrays'):
        e.set_net_weights(_lib.NET_POLICY, w[2][:-1])
    with pytest.raises(ValueError, match=f'expected {2 * (L + 1)} weight arrays'):
        e.set_net_weights(_lib.NET_POLICY, synthetic.make_mlp_weights(np.random.default_rng(0), d_o, H, 2 * d_a))
    assert not e.tc_available()
    with pytest.raises(RuntimeError, match='hidden = 256') as exc:
        e.set_backend(BACKEND_TC)
    assert f'this handle has {L}' in str(exc.value)
    cfg = _lib.MpgConfig.from_buffer_copy(e.cfg)
    for bad in (0, 4):
        h = ctypes.c_void_p()
        assert e.lib.mpg_create_layers(ctypes.byref(cfg), bad, ctypes.byref(h)) == -3   # MPG_ERR_UNSUPPORTED
        assert not h.value and b'1, 2 or 3' in e.lib.mpg_last_error(None)
    h = ctypes.c_void_p()
    assert e.lib.mpg_create(ctypes.byref(cfg), ctypes.byref(h)) == 0
    try:
        assert e.lib.mpg_hidden_layers(h) == 2
        assert e.lib.mpg_param_count(h, _lib.NET_Q1) == (d_o + d_a) * H + H + H * H + H + H + 1
    finally:
        e.lib.mpg_destroy(h)


@pytest.mark.gpu
def test_capacity_growth_keeps_the_depth():
    """ensure_capacity re-creates the handle: with the same depth, weights and backend."""
    H, L, B = 64, 3, 300
    args = _args('NADP', PT, H, L, replay_batch_size=64)
    w = _weights(14, args, H, L, False)
    e = _policy(args, w).engine
    assert e.cfg.max_rows < B
    obs = e.dev(synthetic.make_obs(np.random.default_rng(15), PT, B))
    g, _ = e.policy_grad(obs, [5], [1.0], use_philox=True, noise_seed=1)
    _ffma(e, L)
    assert e.cfg.max_rows >= B and g.numel() == e.param_count(2)
    assert all(np.array_equal(a, b) for a, b in zip(e.get_net_weights(2), w[1]))


# ------------------------------------------------------------------------------------------------
# trainer smoke tests
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('L', DEPTHS)
def test_trainer_smoke(L):
    from mpg_b200.trainer import Trainer
    args = _args('MPG-v2', PT, 256, L, replay_batch_size=256, batch_size=512, num_agent=8, explore_sigma=0.1,
                 max_buffer_size=100000, replay_starts=1024, buffer_log_interval=10 ** 9, num_eval_agent=16,
                 num_eval_episode=1, fixed_steps=20, eval_interval=10 ** 9, log_interval=10 ** 9, max_iter=8, log_dir=None)
    tr = Trainer(args)
    _ffma(tr.learner.engine, L)
    tr.train(args.max_iter)
    st = tr.learner.get_stats()
    assert tr.optimizer.get_stats()['num_sampled_steps'] >= args.replay_starts
    for k in ('policy_gradient_norm', 'q_gradient_norm1', 'q_loss1', 'policy_total_loss', 'value_mean'):
        assert np.isfinite(st[k]), (k, st[k])
    assert np.isfinite(tr.evaluator.run_evaluation(args.max_iter)['episode_return'])
