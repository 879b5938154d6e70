"""Hidden widths 64 and 128 on the fp32 (FFMA) kernels.  The CUDA path is held directly to the golden vectors the
reference's own code produced at H = 64 (tests/golden/make_golden.py), to the fp64 oracle at H = 128 (there are no
goldens at that width), and to the size-independent properties at the bench size.  The tensor-core backend is built
for H = 256 only: at the other widths the handle offers the FFMA backend alone."""
import ctypes

import numpy as np
import pytest
import torch

from mpg_b200 import synthetic
from mpg_b200.config import default_args
from tests.util import load_golden, make_batch, model_case_inputs, mpg_case_inputs, nadp_case_inputs, rel_l2

TOL_STATE, TOL_GRAD, TOL_SCALAR = 1e-5, 1e-4, 2e-5
PT, IP, IDP = 'PathTracking-v0', 'InvertedPendulumConti-v0', 'InvertedDoublePendulum-v2'


def _flat(grads):
    return np.concatenate([np.asarray(g, np.float64).ravel() for g in grads])


def _unclip(g, norm, clip):
    return g * max(norm, clip) / clip


def _learner(kind, args, weights):
    from mpg_b200.engine import BACKEND_FFMA
    from mpg_b200.learners import MPGLearner, NADPLearner
    from mpg_b200.policy import PolicyWithQs
    learner = (NADPLearner if kind == 'nadp' else MPGLearner)(PolicyWithQs, args)
    learner.set_weights(weights)
    assert learner.engine.backend == BACKEND_FFMA
    return learner


def _width_args(alg, env_id, H, **kw):
    return default_args(alg, env_id, value_num_hidden_units=H, policy_num_hidden_units=H, **kw)


# ------------------------------------------------------------------------------------------------
# golden vectors from the reference's own code (H = 64)
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('name', ['nadp_pt_h64_m2_nfd2', 'nadp_ip_h64'])
def test_nadp_h64_matches_reference_golden(name):
    case, gold = load_golden(name)
    args, w, batch, nq, npol = nadp_case_inputs(case)
    learner = _learner('nadp', args, w)
    learner.set_rollout_noise(nq, npol)
    grads = learner.compute_gradient(batch, None, None, 7)
    st = learner.get_stats()
    assert len(grads) == 12 and grads[0].shape == (args.obs_dim + args.act_dim, 64)
    assert grads[6].shape == (args.obs_dim, 64) and grads[10].shape == (64, 2 * args.act_dim)
    flat = _flat(grads)
    nQ = gold['q_grad__f64'].size
    clip = args.gradient_clip_norm
    assert rel_l2(_unclip(flat[:nQ], st['q_gradient_norm'], clip), gold['q_grad__f64']) <= TOL_GRAD
    assert rel_l2(_unclip(flat[nQ:], st['policy_gradient_norm'], clip), gold['policy_grad__f64']) <= TOL_GRAD
    for k in ('q_loss', 'policy_loss', 'value_mean', 'q_gradient_norm', 'policy_gradient_norm'):
        assert rel_l2(st[k], gold[f'stat_{k}__f64']) <= TOL_SCALAR, (k, st[k], gold[f'stat_{k}__f64'])
    if 'td_error__f64' in gold:   # prioritized replay
        assert rel_l2(learner.get_info_for_buffer()['td_error'], gold['td_error__f64']) <= TOL_SCALAR
    # forward-only Q-target rollout (nadp.py:87-126)
    learner.set_rollout_noise(nq, npol)
    tgt = learner.model_rollout_for_q_estimation(learner._dev['batch_obs'], learner._dev['batch_actions'])
    assert rel_l2(tgt.cpu().numpy(), gold['q_targets__f64']) <= TOL_STATE


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['mpg2_pt_h64_list3', 'mpg2_pt_h64_deriv', 'mpg1_pt_h64', 'mpg2_ip_h64'])
def test_mpg_h64_matches_reference_golden(name):
    case, gold = load_golden(name)
    args, w, batch, npol = mpg_case_inputs(case)
    learner = _learner('mpg', args, w)
    learner.set_rollout_noise(None, npol)
    grads = learner.compute_gradient(batch, None, None, case['iteration'])
    st = learner.get_stats()
    n_q = 2 if 'q_grad2__f64' in gold else 1
    assert len(grads) == 6 * (n_q + 1) and grads[0].shape == (args.obs_dim + args.act_dim, 64)
    flat = _flat(grads)
    nQ = gold['q_grad1__f64'].size
    clip = args.gradient_clip_norm
    assert rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), gold['batch_targets__f64']) <= TOL_STATE
    assert rel_l2(_unclip(flat[:nQ], st['q_gradient_norm1'], clip), gold['q_grad1__f64']) <= TOL_GRAD
    if n_q == 2:
        assert rel_l2(_unclip(flat[nQ:2 * nQ], st['q_gradient_norm2'], clip), gold['q_grad2__f64']) <= TOL_GRAD
    pg = flat[n_q * nQ:]
    assert rel_l2(_unclip(pg, st['policy_gradient_norm'], clip), gold['policy_grad__f64']) <= TOL_GRAD
    for k in ('value_mean', 'policy_total_loss', 'policy_gradient_norm', 'q_loss1', 'q_gradient_norm1', 'q_loss2',
              'q_gradient_norm2'):
        if f'stat_{k}__f64' in gold:
            assert rel_l2(st[k], gold[f'stat_{k}__f64']) <= TOL_SCALAR, (k, st[k], gold[f'stat_{k}__f64'])
    if 'td_error__f64' in gold:   # prioritized replay
        assert rel_l2(learner.get_info_for_buffer()['td_error'], gold['td_error__f64']) <= TOL_SCALAR
    assert np.allclose(st['w_list'], gold['stat_w_list__f64'], rtol=1e-4)
    assert rel_l2(st['all_losses'], gold['stat_all_losses__f64']) <= TOL_SCALAR


@pytest.mark.gpu
def test_nadp_idp_h64_within_fp32_spread_of_reference():
    """The falling double pendulum amplifies fp32 rounding: the golden's own fp32 run is 2.6e-2 from its fp64 run on the
    policy gradient.  The FFMA path must land within K = 4 of that spread (the rule of the H = 256 oracle comparison)."""
    case, gold = load_golden('nadp_idp_h64')
    args, w, batch, nq, npol = nadp_case_inputs(case)
    learner = _learner('nadp', args, w)
    learner.set_rollout_noise(nq, npol)
    flat = _flat(learner.compute_gradient(batch, None, None, 0))
    st = learner.get_stats()
    nQ = gold['q_grad__f64'].size
    got_p = _unclip(flat[nQ:], st['policy_gradient_norm'], args.gradient_clip_norm)
    K = 4.0
    spread_p = rel_l2(gold['policy_grad__f32'], gold['policy_grad__f64'])
    spread_l = rel_l2(gold['stat_policy_loss__f32'], gold['stat_policy_loss__f64'])
    err_p = rel_l2(got_p, gold['policy_grad__f64'])
    err_l = rel_l2(st['policy_loss'], gold['stat_policy_loss__f64'])
    print(dict(err_grad=err_p, spread_grad=spread_p, err_loss=err_l, spread_loss=spread_l))
    assert err_p <= K * max(spread_p, 1e-6), (err_p, spread_p)
    assert err_l <= K * max(spread_l, 1e-7), (err_l, spread_l)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['model_pt', 'model_pt_nfd2', 'model_ip', 'model_idp'])
def test_closed_loop_h64_matches_reference_golden(name):
    """States, rewards and actions of the closed-loop rollout of an H = 64 policy, per step, against the reference's
    own trajectories; on the chaotic double pendulum the first 4 steps only."""
    from mpg_b200.policy import PolicyWithQs
    case, gold = load_golden(name)
    args, obs0, _, noise, w = model_case_inputs(case)
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(w)
    e = pol.engine
    n = case['n']
    _, t_obs, t_rew, t_act = e.rollout_forward(e.dev(obs0), [n], noise=e.dev(noise), want_traj=True)
    horizon_checked = n if args.env_id != IDP else 4
    worst = 0.0
    for t in range(horizon_checked):
        worst = max(worst, rel_l2(t_obs[t].cpu().numpy(), gold['closed_obs__f64'][t]),
                    rel_l2(t_rew[t].cpu().numpy(), gold['closed_rew__f64'][t]))
    for t in range(horizon_checked + 1):
        worst = max(worst, rel_l2(t_act[t].cpu().numpy(), gold['closed_act__f64'][t]))
    print(name, 'worst per-step rel-L2', worst)
    assert worst <= TOL_STATE, worst


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['apply_grads_v2_h64', 'apply_grads_nadp_h64'])
def test_apply_gradients_h64_matches_reference_golden(name):
    """Adam / delayed policy update / Polyak targets on the device-resident H = 64 weights against the reference's
    own run; the gradient sequence is re-derived as in test_oracle_golden.test_apply_gradients_oracle_matches_reference."""
    from mpg_b200.policy import PolicyWithQs
    case, gold = load_golden(name)
    H, dq = case['H'], case['version'] == 'MPG-v2'
    args = _width_args(case['version'], PT, H)
    w = synthetic.make_policy_with_qs_weights(case['wseed'], args.obs_dim, args.act_dim, H, double_q=dq)
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(w)
    rng = np.random.default_rng(case['gseed'])
    for it in range(case['iters']):
        grads = [rng.standard_normal(np.shape(a)).astype(np.float32) * 0.1 for net in w[: (3 if dq else 2)] for a in net]
        pol.apply_gradients(it, grads)
    got = np.concatenate([np.asarray(a, np.float64).ravel() for net in pol.get_weights() for a in net])
    assert rel_l2(got, gold['weights__f64']) <= 2e-6


@pytest.mark.gpu
def test_mpg_v1_n_step_target_h64_matches_reference_golden():
    """MPG-v1 n-step target: 25 real-env steps, nfd = 2, H = 64."""
    from mpg_b200.learners import MPGLearner
    from mpg_b200.policy import PolicyWithQs
    from tests.test_real_env import _case_inputs
    case, gold = load_golden('real_env_h64')
    _, _, args, w, batch = _case_inputs(case)
    learner = MPGLearner(PolicyWithQs, args)
    learner.set_weights(w)
    learner.get_batch_data(batch, None, None)
    assert rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), gold['batch_targets__f64']) <= 2e-5


# ------------------------------------------------------------------------------------------------
# H = 128 against the fp64 oracle
# ------------------------------------------------------------------------------------------------
def _nadp_h128_vs_oracle(B, n, seed=0, per_row=False):
    from oracle import mpg_oracle as O
    from tests.test_gpu_parity import _row_returns_vs_oracle
    H = 128
    args = _width_args('NADP', PT, H, replay_batch_size=B, num_rollout_list_for_policy_update=[n],
                       num_rollout_list_for_q_estimation=[n])
    w = synthetic.make_policy_with_qs_weights(100 + seed, args.obs_dim, args.act_dim, H, double_q=False)
    batch = make_batch(200 + seed, PT, B, 0)
    rng = np.random.default_rng(300 + seed)
    nq, npol = synthetic.make_noise(rng, n, B), synthetic.make_noise(rng, n, B)
    learner = _learner('nadp', args, w)
    learner.set_rollout_noise(nq, npol)
    grads = learner.compute_gradient(batch, None, None, 0)
    assert grads[2].shape == (H, H)
    flat = _flat(grads)
    st = learner.get_stats()
    ref = O.nadp_compute_gradient(args, w, batch, nq, npol, torch.float64)
    nQ = ref['q_grad'].size
    clip = args.gradient_clip_norm
    errs = dict(q=rel_l2(_unclip(flat[:nQ], st['q_gradient_norm'], clip), ref['q_grad']),
                p=rel_l2(_unclip(flat[nQ:], st['policy_gradient_norm'], clip), ref['policy_grad']),
                clipped=rel_l2(flat, ref['compute_gradient']))
    if per_row:
        # the means of many short-horizon returns of both signs nearly cancel: rows to 1e-5, means to the matching
        # absolute error (as test_gpu_parity._nadp_vs_oracle(per_row=True))
        row_err, scale = _row_returns_vs_oracle(learner, args, w, batch, npol, n)
        errs['rows'] = row_err
        assert row_err <= TOL_STATE, errs
        for k in ('policy_loss', 'value_mean'):
            assert abs(st[k] - ref[k]) <= TOL_SCALAR * max(scale, abs(ref[k])), (k, st[k], ref[k], scale)
        target_scale = float(np.abs(ref['q_targets']).mean())
        assert abs(st['q_loss'] - ref['q_loss']) <= 2 * TOL_SCALAR * max(target_scale ** 2, abs(ref['q_loss']))
    else:
        for k in ('q_loss', 'policy_loss', 'value_mean'):
            errs[k] = rel_l2(st[k], ref[k])
            assert errs[k] <= TOL_SCALAR, errs
    print('H=128', B, n, errs)
    assert errs['q'] <= TOL_GRAD and errs['p'] <= TOL_GRAD and errs['clipped'] <= TOL_GRAD, errs
    return learner


@pytest.mark.gpu
@pytest.mark.parametrize('B', [1, 300, 2048])
def test_nadp_h128_vs_oracle(B):
    _nadp_h128_vs_oracle(B, 25, per_row=(B < 16))


@pytest.mark.gpu
def test_nadp_h128_multi_wave_vs_oracle():
    """20,011 rows = 313 tiles: several tiles per CTA."""
    learner = _nadp_h128_vs_oracle(20011, 3, seed=9, per_row=True)
    assert learner.engine.num_sms < 313


@pytest.mark.gpu
def test_mpg_v2_h128_vs_oracle():
    from oracle import mpg_oracle as O
    H, B, ite = 128, 160, 4000
    args = _width_args('MPG-v2', PT, H, replay_batch_size=B, num_rollout_list_for_policy_update=[0, 25],
                       buffer_type='priority', sample_num_in_learner=None)
    w = synthetic.make_policy_with_qs_weights(7, args.obs_dim, args.act_dim, H, double_q=True)
    batch = make_batch(8, PT, B, 0)
    npol = synthetic.make_noise(np.random.default_rng(9), 25, B)
    learner = _learner('mpg', args, w)
    learner.set_rollout_noise(None, npol)
    flat = _flat(learner.compute_gradient(batch, None, None, ite))
    st = learner.get_stats()
    ref = O.mpg_compute_gradient(args, w, batch, npol, ite, torch.float64)
    nQ = ref['q_grad1'].size
    errs = dict(clipped=rel_l2(flat, ref['compute_gradient']),
                p=rel_l2(_unclip(flat[2 * nQ:], st['policy_gradient_norm'], args.gradient_clip_norm), ref['policy_grad']),
                targets=rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), ref['batch_targets']),
                td=rel_l2(learner.get_info_for_buffer()['td_error'], ref['td_error']),
                total_loss=rel_l2(st['policy_total_loss'], ref['total_loss']),
                value_mean=rel_l2(st['value_mean'], ref['value_mean']),
                q1=rel_l2(st['q_loss1'], ref['q_loss1']))
    print('H=128 MPG-v2', errs)
    assert errs['clipped'] <= TOL_GRAD and errs['p'] <= TOL_GRAD, errs
    for k in ('targets', 'td', 'total_loss', 'value_mean', 'q1'):
        assert errs[k] <= TOL_SCALAR, errs


@pytest.mark.gpu
def test_compute_action_and_q1_h128_vs_oracle():
    from oracle import mpg_oracle as O
    from mpg_b200.policy import PolicyWithQs
    H, B = 128, 1000
    args = _width_args('NADP', PT, H)
    w = synthetic.make_policy_with_qs_weights(3, args.obs_dim, args.act_dim, H, double_q=False)
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(w)
    rng = np.random.default_rng(4)
    p = synthetic.make_obs(rng, PT, B) * np.asarray(args.obs_scale, np.float32)   # processed observations
    act = rng.uniform(-1, 1, (B, args.act_dim)).astype(np.float32)
    got_a, _ = pol.compute_action(p)
    got_q = pol.compute_Q1(p, act)
    w64 = [[O.to_t(x, torch.float64) for x in net] for net in w]
    ref_a = O.policy_action(w64[1], O.to_t(p, torch.float64), 'tanh', None).numpy()
    ref_q = O.q_value(w64[0], O.to_t(p, torch.float64), O.to_t(act, torch.float64)).numpy()
    assert rel_l2(got_a.cpu().numpy(), ref_a) <= TOL_STATE
    assert rel_l2(got_q.cpu().numpy(), ref_q) <= TOL_STATE


# ------------------------------------------------------------------------------------------------
# properties at the bench size
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('H', [64, 128])
def test_full_size_properties_h(H):
    """B = 65,536, n = 25: two identical calls are bit-identical (the row slices of a feature are combined in a fixed
    order), and two half batches with global scaling add up to the full batch."""
    from mpg_b200.policy import PolicyWithQs
    B, n = 65536, 25
    args = _width_args('NADP', PT, H, replay_batch_size=B)
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(synthetic.make_policy_with_qs_weights(1, args.obs_dim, args.act_dim, H, double_q=False))
    e = pol.engine
    obs = e.dev(synthetic.make_obs(np.random.default_rng(2), PT, B))
    kw = dict(full_bptt=True, use_philox=True, noise_seed=11)
    g1, r1 = e.policy_grad(obs, [0, n], [0.3, 0.7], **kw)
    g2, r2 = e.policy_grad(obs, [0, n], [0.3, 0.7], **kw)
    assert g1.numel() == e.param_count(2)
    assert torch.equal(g1, g2) and torch.equal(r1, r2), 'not bit-reproducible run to run'
    assert torch.isfinite(g1).all() and torch.isfinite(r1).all()
    h = B // 2
    gl, _ = e.policy_grad(obs[:h].contiguous(), [0, n], [0.3, 0.7], global_rows=B, row_offset=0, **kw)
    gr, _ = e.policy_grad(obs[h:].contiguous(), [0, n], [0.3, 0.7], global_rows=B, row_offset=h, **kw)
    assert rel_l2((gl + gr).cpu().numpy(), g1.cpu().numpy()) <= 1e-5


# ------------------------------------------------------------------------------------------------
# errors and backend selection
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_width_errors_and_backend_selection():
    from mpg_b200 import _lib
    from mpg_b200.engine import BACKEND_FFMA, BACKEND_TC
    from mpg_b200.policy import PolicyWithQs
    with pytest.raises(NotImplementedError, match='64 / 128 / 256'):
        PolicyWithQs(**vars(_width_args('NADP', PT, 96)))
    with pytest.raises(NotImplementedError, match='must be equal'):
        PolicyWithQs(**vars(default_args('NADP', PT, policy_num_hidden_units=64, value_num_hidden_units=128)))
    for H in (64, 128):
        e = PolicyWithQs(**vars(_width_args('MPG-v2', PT, H))).engine
        assert e.cfg.hidden == H and not e.tc_available() and e.backend == BACKEND_FFMA
        with pytest.raises(RuntimeError, match='hidden = 256'):
            e.set_backend(BACKEND_TC)
    cfg = _lib.MpgConfig.from_buffer_copy(e.cfg)
    cfg.hidden = 96
    h = ctypes.c_void_p()
    assert e.lib.mpg_create(ctypes.byref(cfg), ctypes.byref(h)) == -3   # MPG_ERR_UNSUPPORTED
    assert not h.value and b'64, 128 or 256' in e.lib.mpg_last_error(None)


@pytest.mark.gpu
def test_trainer_h64_smoke():
    from mpg_b200.trainer import Trainer
    args = default_args('MPG-v2', PT, replay_batch_size=256, batch_size=512, num_agent=8, explore_sigma=0.1,
                        max_buffer_size=100000, replay_starts=1024, buffer_log_interval=10 ** 9, num_eval_agent=16,
                        num_eval_episode=1, fixed_steps=20, eval_interval=10 ** 9, log_interval=10 ** 9, max_iter=8,
                        log_dir=None, value_num_hidden_units=64, policy_num_hidden_units=64)
    tr = Trainer(args)
    assert tr.learner.engine.cfg.hidden == 64
    tr.train(args.max_iter)
    st = tr.learner.get_stats()
    assert tr.optimizer.get_stats()['num_sampled_steps'] >= args.replay_starts
    for k in ('policy_gradient_norm', 'q_gradient_norm1', 'q_loss1', 'policy_total_loss', 'value_mean'):
        assert np.isfinite(st[k]), (k, st[k])
    assert np.isfinite(tr.evaluator.run_evaluation(args.max_iter)['episode_return'])


# ------------------------------------------------------------------------------------------------
# CPU: the width check comes before the device
# ------------------------------------------------------------------------------------------------
def test_width_check_precedes_the_device():
    from mpg_b200.policy import PolicyWithQs
    with pytest.raises(NotImplementedError, match='64 / 128 / 256'):
        PolicyWithQs(**vars(_width_args('NADP', PT, 96)))
    if torch.cuda.is_available():
        return
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        PolicyWithQs(**vars(_width_args('NADP', PT, 64)))
