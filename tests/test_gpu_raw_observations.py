"""Every GPU entry point whose step 0 runs through the rollout kernels, on observations that the model's observation map
does not reproduce.  The rest of the suite draws its observations with synthetic.make_obs, for which
get_obs(reset(obs)) == obs.  Replay data is not like that:
  * PathTracking with num_future_data > 0: the real environment fills the future columns with path deltas
    y - path_y(x + k v_x 0.2); the model's get_obs writes copies of delta_y there;
  * double pendulum: the last three entries (constraint forces) are non-zero in real data; the model's get_obs zeroes them.
The reference (and the oracle, the truth here) feeds the nets sigma * obs at step 0 and starts the model from reset(obs);
later steps observe get_obs(s_t).  The input builders refuse inputs that lie on the map, and
test_inputs_are_off_the_observation_map (CPU) checks that the oracle itself tells the two routes apart on every kind of
input used here, by far more than the bars.

Bars are the suite's: per-row returns, actions and the per-step closed loop <= 1e-5 norm-relative, gradients <= 1e-4,
scalars (targets, TD errors, bootstraps, losses) <= 2e-5.  Every case prints its measured errors."""
import copy

import numpy as np
import pytest
import torch

from mpg_b200 import _lib, synthetic
from mpg_b200.config import default_args
from tests.test_gpu_config_space import (TOL_GRAD, TOL_STATE, _check_closed_loop, _check_policy_grad, _handle, _pt_args,
                                         oracle_policy_grad)
from tests.test_gpu_parity import _flat, _learner, _unclip
from tests.util import rel_l2

TOL_SCALAR = 2e-5
PT, IDP = 'PathTracking-v0', 'InvertedDoublePendulum-v2'
BACKENDS = ['ffma', 'tc']
# input kinds: nfd 7 is the widest tensor-core case, nfd 10 runs on FFMA only; nfd 3 is the sampler's and the hi-only case
KINDS = {'pt_nfd2': (PT, 2), 'pt_nfd3': (PT, 3), 'pt_nfd7': (PT, 7), 'pt_nfd10': (PT, 10), 'idp': (IDP, 0)}
CASES = ['pt_nfd2', 'pt_nfd7', 'pt_nfd10', 'idp']
MIN_OFF_MAP = 0.1


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def map_obs(env_id, nfd, obs):
    """get_obs(reset(obs)) of the model, in fp32 like the kernels, and the columns it rewrites."""
    from oracle import mpg_oracle as O
    m = O.NAME2MODELCLS[env_id](num_future_data=nfd)
    m.reset(torch.as_tensor(np.asarray(obs, np.float32)))
    cols = list(range(6, 6 + nfd)) if env_id == PT else [1, 2, 3, 4, 8, 9, 10]
    return m.get_obs(m.s).numpy().astype(np.float32), cols


def off_map(env_id, nfd, obs):
    """max |obs - get_obs(reset(obs))| over the columns the observation map rewrites."""
    mapped, cols = map_obs(env_id, nfd, obs)
    return float(np.abs(np.asarray(obs, np.float64)[:, cols] - mapped[:, cols]).max())


def _require_off_map(env_id, nfd, obs):
    d = off_map(env_id, nfd, obs)
    assert d > MIN_OFF_MAP, f'{env_id} nfd={nfd}: the inputs are {d:.3g} from the observation map, they test nothing'
    return obs


def pt_real_obs(B, nfd, seed):
    """Real-environment PathTracking observations: reset-law poses (make_obs) after 2-4 steps of the fp32 real
    environment under random actions.  Their future columns hold path deltas."""
    from oracle import mpg_oracle as O
    rng = np.random.default_rng(1000 + 16 * nfd + seed)
    env = O.PathTrackingEnvOracle(nfd, np.float32)
    env.reset(synthetic.make_obs(rng, PT, B, nfd))
    for _ in range(2 + seed % 3):
        obs, _, _ = env.step(rng.uniform(-0.3, 0.3, (B, 2)).astype(np.float32))
    return _require_off_map(PT, nfd, np.ascontiguousarray(obs, np.float32))


def idp_obs(B, seed):
    """Double-pendulum observations with non-zero constraint forces (entries 8-10) and velocities, both up to the
    reference's +-10 clip."""
    rng = np.random.default_rng(1100 + seed)
    obs = synthetic.make_obs(rng, IDP, B)
    obs[:, 5:8] = rng.uniform(-10.0, 10.0, (B, 3))
    obs[:, 8:] = rng.uniform(-10.0, 10.0, (B, 3))
    return _require_off_map(IDP, 0, obs)


def raw_obs(kind, B, seed=0):
    env_id, nfd = KINDS[kind]
    return pt_real_obs(B, nfd, seed) if env_id == PT else idp_obs(B, seed)


def case_args(kind, alg, rows, **kw):
    """Learner args of an input kind (PathTracking: random non-unit scales on the future columns) and its horizon."""
    env_id, nfd = KINDS[kind]
    if env_id == PT:
        return _pt_args(alg, nfd, replay_batch_size=rows, **kw), 25
    return default_args(alg, IDP, replay_batch_size=rows, **kw), 3   # n <= 3 on the double pendulum, as in the suite


def weights(args, seed, double_q=True):
    return synthetic.make_policy_with_qs_weights(1200 + seed, args.obs_dim, args.act_dim, 256, double_q=double_q)


# ------------------------------------------------------------------------------------------------
# CPU guard: the inputs are off the observation map, and the two step-0 routes differ far beyond the bars
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', list(KINDS))
def test_inputs_are_off_the_observation_map(kind):
    """The oracle once on the raw observations and once on get_obs(reset(obs)) (what a rollout kernel that re-derives
    its step-0 observation from the model state would see): the returns rows and the policy gradient must differ by more
    than 100 x their bars, in NADP full BPTT [n] or MPG-v2 first-action [0, n] mode."""
    env_id, nfd = KINDS[kind]
    B = 256
    args, n = case_args(kind, 'MPG-v2', B)
    obs = raw_obs(kind, B, seed=3)
    mapped, _ = map_obs(env_id, nfd, obs)
    w = weights(args, 3)
    noise = synthetic.make_noise(np.random.default_rng(5), n, B)
    diff = dict(obs=off_map(env_id, nfd, obs), rows=0.0, grad=0.0)
    for lst, lw, full in (([n], [1.0], True), ([0, n], [0.3, 0.7], False)):
        r1, g1 = oracle_policy_grad(args, w, obs, noise, lst, lw, 1, full, _lib.NET_Q1)
        r2, g2 = oracle_policy_grad(args, w, mapped, noise, lst, lw, 1, full, _lib.NET_Q1)
        diff['rows'] = max(diff['rows'], max(rel_l2(b, a) for a, b in zip(r1, r2)))
        diff['grad'] = max(diff['grad'], rel_l2(g2, g1))
    print(kind, 'raw vs mapped observations', diff)
    assert diff['obs'] > MIN_OFF_MAP, diff
    assert diff['rows'] > 100 * TOL_STATE and diff['grad'] > 100 * TOL_GRAD, diff


# ------------------------------------------------------------------------------------------------
# 1. mpg_policy_grad
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('kind', CASES)
def test_policy_grad_raw_obs_vs_oracle(kind, backend):
    """NADP full BPTT [n], MPG-v2 first-action [0, n] (Q(p_0, a_0) on the raw observation) and no bootstrap."""
    B = 512
    args, n = case_args(kind, 'MPG-v2', B)
    obs = raw_obs(kind, B)
    w = weights(args, 0)
    noise = synthetic.make_noise(np.random.default_rng(10), n, B)
    _, e = _handle(args, w, backend)
    _check_policy_grad(e, args, w, obs, noise, [n], [1.0], f'{kind} NADP full BPTT')
    _check_policy_grad(e, args, w, obs, noise, [0, n], [0.3, 0.7], f'{kind} MPG-v2 first action', full_bptt=False)
    _check_policy_grad(e, args, w, obs, noise, [0, n], [0.4, 0.6], f'{kind} no bootstrap', q_net=-1)


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_m3_ragged_raw_obs_vs_oracle(backend):
    """Each of the M tiles starts from obs[i]: 6,701 rows x 3 tiles, ragged last tile."""
    B, M = 6701, 3
    args, _ = case_args('pt_nfd7', 'MPG-v2', B, M=M)
    n = 3
    obs = raw_obs('pt_nfd7', B, seed=1)
    w = weights(args, 1)
    noise = synthetic.make_noise(np.random.default_rng(11), n, B * M)
    _, e = _handle(args, w, backend)
    assert (B * M) % 128 != 0
    _check_policy_grad(e, args, w, obs, noise, [0, n], [0.4, 0.6], 'pt_nfd7 M=3 ragged', M=M)


# ------------------------------------------------------------------------------------------------
# 2. mpg_rollout_forward: the NADP Q-estimation rollout (given start actions) and the closed loop
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('kind', CASES)
def test_rollout_forward_raw_obs_vs_oracle(kind, backend):
    from oracle import mpg_oracle as O
    B = 512
    args, n = case_args(kind, 'NADP', B)
    obs = raw_obs(kind, B, seed=2)
    w = weights(args, 2, double_q=False)
    rng = np.random.default_rng(12)
    act = rng.uniform(-1, 1, (B, args.act_dim)).astype(np.float32)
    noise = synthetic.make_noise(rng, n, B)
    _, e = _handle(args, w, backend)
    got = e.rollout_forward(e.dev(obs), [0, n], q_net=_lib.NET_Q1_TARGET, start_actions=e.dev(act),
                            noise=e.dev(noise)).cpu().numpy()
    nets = O.Nets(w, False, torch.float64)
    with torch.no_grad():
        ref = O.rollout(args, torch.float64, None, nets.policy, nets.Q1_t, O.to_t(obs, torch.float64),
                        O.to_t(noise, torch.float64), n, start_actions=O.to_t(act, torch.float64)).numpy()
    errs = dict(row0=rel_l2(got[0], ref[0]), row_n=rel_l2(got[1], ref[n]))
    print(kind, 'Q-estimation rollout, backend', e.backend, errs)
    assert max(errs.values()) <= TOL_STATE, errs
    # traj_act[0] = pi(sigma obs) on the raw observation, then every step of the closed loop
    _check_closed_loop(e, args, w[1], obs, noise, n, kind)


# ------------------------------------------------------------------------------------------------
# 3. tensor cores, hi-only dW2 records: the [p|1] record of step 0 carries the raw observation
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_tc_hi_only_records_raw_obs_vs_oracle(monkeypatch):
    monkeypatch.delenv('MPG_REC_HI_ONLY', raising=False)
    B, n = 10112, 25
    assert B * (n + 1) >= 262144, 'api.cu: rec_hi_only selects hi-only records from 262,144 (row, step) pairs'
    args, _ = case_args('pt_nfd3', 'NADP', B)
    obs = raw_obs('pt_nfd3', B, seed=4)
    w = weights(args, 4, double_q=False)
    noise = synthetic.make_noise(np.random.default_rng(14), n, B)
    _, e = _handle(args, w, 'tc')
    _check_policy_grad(e, args, w, obs, noise, [n], [1.0], 'pt_nfd3 hi-only records')


# ------------------------------------------------------------------------------------------------
# 4. mpg_q_grad: tensor-core regression mode (a horizon-0 rollout), the over-capacity FFMA fallback, FFMA
# ------------------------------------------------------------------------------------------------
ROUTES = {'tc': ('tc', None), 'tc_over_capacity': ('tc', 500), 'ffma': ('ffma', None)}


@pytest.mark.gpu
@pytest.mark.parametrize('route', list(ROUTES))
@pytest.mark.parametrize('kind', CASES)
def test_q_grad_raw_obs_vs_oracle(kind, route):
    from oracle import mpg_oracle as O
    B = 2048
    backend, cap = ROUTES[route]
    args, _ = case_args(kind, 'NADP', cap or B)
    obs = raw_obs(kind, B, seed=5)
    w = weights(args, 5, double_q=False)
    rng = np.random.default_rng(15)
    act = rng.uniform(-1, 1, (B, args.act_dim)).astype(np.float32)
    _, e = _handle(args, w, backend)
    assert (e.cfg.max_rows >= B) == (cap is None)
    nets = O.Nets(w, False, torch.float64)
    t64 = lambda x: O.to_t(x, torch.float64)   # noqa: E731
    q_pred = O.q_value(nets.Q1, t64(obs) * t64(args.obs_scale), t64(act))
    target = (0.5 * q_pred.detach().numpy() + rng.standard_normal(B)).astype(np.float32)
    loss = 0.5 * torch.mean((q_pred - t64(target)) ** 2)
    ref = np.concatenate([x.numpy().ravel() for x in torch.autograd.grad(loss, nets.Q1)])
    g, loss_sum = e.q_grad(_lib.NET_Q1, e.dev(obs), e.dev(act), e.dev(target))
    errs = dict(grad=rel_l2(g.cpu().numpy(), ref), loss=rel_l2(float(loss_sum.item()) / B, float(loss.item())))
    print(kind, 'q_grad', route, errs)
    assert errs['grad'] <= TOL_GRAD and errs['loss'] <= TOL_SCALAR, errs


# ------------------------------------------------------------------------------------------------
# 5. evaluation entry points, three routes, and the tensor-core and FFMA routes against each other
# ------------------------------------------------------------------------------------------------
def _evaluations(e, obs, act, rew, obs1, base):
    d = e.dev
    got = dict(target_double=e.q_target(True, d(rew), d(obs1)), target_single=e.q_target(False, d(rew), d(obs1)),
               td=e.td_error(d(obs), d(act), d(rew), d(obs1)), bootstrap=e.q_bootstrap(d(base), 0.7, d(obs)),
               act=e.policy_forward(_lib.NET_POLICY, d(obs)), act_target=e.policy_forward(_lib.NET_POLICY_TARGET, d(obs)),
               q=e.q_forward(_lib.NET_Q1, d(obs), d(act)))
    return {k: v.cpu().numpy() for k, v in got.items()}


def _bar(k):
    return TOL_STATE if k in ('act', 'act_target', 'q') else TOL_SCALAR


@pytest.mark.gpu
@pytest.mark.parametrize('kind', CASES)
def test_evaluations_raw_obs_vs_oracle(kind):
    from oracle import mpg_oracle as O
    B = 1000
    args, _ = case_args(kind, 'MPG-v2', B)
    obs, obs1 = raw_obs(kind, B, seed=6), raw_obs(kind, B, seed=7)
    w = weights(args, 6)
    rng = np.random.default_rng(16)
    act = rng.uniform(-1, 1, (B, args.act_dim)).astype(np.float32)
    rew = (-np.abs(rng.standard_normal(B))).astype(np.float32)
    base = rng.standard_normal(B).astype(np.float32)
    nets = O.Nets(w, True, torch.float64)
    t64 = lambda x: O.to_t(x, torch.float64)   # noqa: E731
    head = (args.policy_out_activation, args.action_range)
    with torch.no_grad():
        sigma = t64(args.obs_scale)
        p, p1 = t64(obs) * sigma, t64(obs1) * sigma
        prew = (t64(rew) + args.rew_shift) * args.rew_scale
        a1 = O.policy_action(nets.policy_t, p1, *head)
        q1t, q2t = O.q_value(nets.Q1_t, p1, a1), O.q_value(nets.Q2_t, p1, a1)
        ref = dict(target_double=prew + args.gamma * torch.minimum(q1t, q2t), target_single=prew + args.gamma * q1t,
                   td=O.td_error(args, nets, [obs, act, rew, obs1], torch.float64),
                   bootstrap=t64(base) + 0.7 * O.q_value(nets.Q1_t, p, O.policy_action(nets.policy_t, p, *head)),
                   act=O.policy_action(nets.policy, p, *head), act_target=O.policy_action(nets.policy_t, p, *head),
                   q=O.q_value(nets.Q1, p, t64(act)))
    ref = {k: v.numpy() for k, v in ref.items()}
    got = {}
    from mpg_b200.policy import PolicyWithQs
    for route, (backend, cap) in ROUTES.items():
        a = copy.copy(args)
        a.replay_batch_size = cap or B     # the handle's capacity
        pol = PolicyWithQs(**vars(a))
        pol.set_weights(w)
        e = pol.engine
        if backend == 'tc' and not e.tc_available():
            continue
        e.set_backend(1 if backend == 'tc' else 0)
        assert (e.cfg.max_rows >= B) == (cap is None)
        got[route] = _evaluations(e, obs, act, rew, obs1, base)
        errs = {k: rel_l2(got[route][k], ref[k]) for k in ref}
        print(kind, 'evaluations', route, errs)
        for k, v in errs.items():
            assert v <= _bar(k), (route, k, errs)
    if 'tc' in got:
        errs = {k: rel_l2(got['tc'][k], got['ffma'][k]) for k in ref}
        print(kind, 'evaluations, tensor cores vs FFMA', errs)
        assert max(errs.values()) <= TOL_STATE, errs


# ------------------------------------------------------------------------------------------------
# 6. learners on a batch of the project's own sampler (PathTrackingEnv + mpg_env_sample, nfd = 3, with restarts)
# ------------------------------------------------------------------------------------------------
SAMPLER_AGENTS, SAMPLER_STEPS = 128, 16


@pytest.fixture(scope='module')
def sampler_batch():
    """(obs, act, rew, obs_tp1, done) of 16 steps x 128 agents, the way worker.sample_arrays draws them.  The reference's
    judge_done flags every step (its tyre-slip bounds carry the sign of the negative cornering stiffnesses; the golden
    real_env_* vectors are all done), so every agent restarts after every step: the first step observes env.reset(), the
    later ones fresh reset draws, and obs_tp1 is one real step later."""
    from mpg_b200.envs_and_models import PathTrackingEnv
    from mpg_b200.policy import PolicyWithQs
    args, _ = case_args('pt_nfd3', 'MPG-v2', SAMPLER_AGENTS * SAMPLER_STEPS)
    pol = PolicyWithQs(**vars(args))
    pol.set_weights(weights(args, 8))
    env = PathTrackingEnv(num_future_data=3, num_agent=SAMPLER_AGENTS, seed=8)
    env.reset()
    fresh = env._draw_on_device(SAMPLER_STEPS).view(SAMPLER_STEPS, SAMPLER_AGENTS, -1)
    gen = torch.Generator(device=env.engine.device)
    gen.manual_seed(9)
    eps = torch.randn(SAMPLER_STEPS, SAMPLER_AGENTS, 2, device=env.engine.device, generator=gen)
    batch = [t.cpu().numpy() for t in pol.engine.env_sample(env.state, env.obs, fresh, eps, 0.2)]
    done = batch[4]
    print('sampler batch: restarts', int(done.sum()), 'of', done.size)
    assert done.sum() > 0, 'the batch is meant to contain restarts'
    _require_off_map(PT, 3, batch[0])
    _require_off_map(PT, 3, batch[3])
    return batch


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_nadp_learner_sampler_batch_vs_oracle(sampler_batch, backend):
    from oracle import mpg_oracle as O
    B, n = sampler_batch[0].shape[0], 25
    args, _ = case_args('pt_nfd3', 'NADP', B, buffer_type='priority')
    w = weights(args, 9, double_q=False)
    rng = np.random.default_rng(19)
    nq, npol = synthetic.make_noise(rng, n, B), synthetic.make_noise(rng, n, B)
    learner = _learner('nadp', args, w, backend)
    learner.set_rollout_noise(nq, npol)
    flat = _flat(learner.compute_gradient(sampler_batch, None, None, 0))
    st = learner.get_stats()
    ref = O.nadp_compute_gradient(args, w, sampler_batch, nq, npol, torch.float64)
    nQ, clip = ref['q_grad'].size, args.gradient_clip_norm
    errs = dict(q=rel_l2(_unclip(flat[:nQ], st['q_gradient_norm'], clip), ref['q_grad']),
                p=rel_l2(_unclip(flat[nQ:], st['policy_gradient_norm'], clip), ref['policy_grad']),
                clipped=rel_l2(flat, ref['compute_gradient']),
                q_loss=rel_l2(st['q_loss'], ref['q_loss']), policy_loss=rel_l2(st['policy_loss'], ref['policy_loss']),
                value_mean=rel_l2(st['value_mean'], ref['value_mean']),
                td=rel_l2(learner.get_info_for_buffer()['td_error'], ref['td_error']))
    print('NADP sampler batch', backend, errs)
    assert max(errs['q'], errs['p'], errs['clipped']) <= TOL_GRAD, errs
    for k in ('q_loss', 'policy_loss', 'value_mean', 'td'):
        assert errs[k] <= TOL_SCALAR, errs


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_mpg_v2_learner_sampler_batch_vs_oracle(sampler_batch, backend):
    from oracle import mpg_oracle as O
    B, lst, ite = sampler_batch[0].shape[0], [0, 10, 25], 4000
    args, _ = case_args('pt_nfd3', 'MPG-v2', B, buffer_type='priority', num_rollout_list_for_policy_update=lst,
                        sample_num_in_learner=None)
    w = weights(args, 10)
    npol = synthetic.make_noise(np.random.default_rng(20), max(lst), B)
    learner = _learner('mpg', args, w, backend)
    learner.set_rollout_noise(None, npol)
    flat = _flat(learner.compute_gradient(sampler_batch, None, None, ite))
    st = learner.get_stats()
    ref = O.mpg_compute_gradient(args, w, sampler_batch, npol, ite, torch.float64)
    nQ = ref['q_grad1'].size
    errs = dict(clipped=rel_l2(flat, ref['compute_gradient']),
                p=rel_l2(_unclip(flat[2 * nQ:], st['policy_gradient_norm'], args.gradient_clip_norm), ref['policy_grad']),
                targets=rel_l2(learner.batch_data['batch_targets'].cpu().numpy(), ref['batch_targets']),
                td=rel_l2(learner.get_info_for_buffer()['td_error'], ref['td_error']),
                total_loss=rel_l2(st['policy_total_loss'], ref['total_loss']),
                value_mean=rel_l2(st['value_mean'], ref['value_mean']),
                q1=rel_l2(st['q_loss1'], ref['q_loss1']), q2=rel_l2(st['q_loss2'], ref['q_loss2']))
    print('MPG-v2 sampler batch', backend, errs)
    assert errs['clipped'] <= TOL_GRAD and errs['p'] <= TOL_GRAD, errs
    for k in ('targets', 'td', 'total_loss', 'value_mean', 'q1', 'q2'):
        assert errs[k] <= TOL_SCALAR, errs


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_mpg_v1_real_env_target_nfd3_vs_oracle(sampler_batch, backend):
    """compute_n_step_target with 25 real-environment steps (sample_num_in_learner) at nfd = 3: the bootstrap
    evaluates Q1_target on the real environment's last observation.  25 fp32 steps of the real environment from these
    states come near the scalar bar by themselves (both backends measure 2.2e-5, an FFMA route that read obs as given
    before this check existed too): the target is held to max(2e-5, 2 x the oracle's own fp32-vs-fp64 distance)."""
    from oracle import mpg_oracle as O
    B, T = sampler_batch[0].shape[0], 25
    args, _ = case_args('pt_nfd3', 'MPG-v1', B, sample_num_in_learner=T)
    w = weights(args, 11, double_q=False)
    learner = _learner('mpg', args, w, backend)
    learner.get_batch_data(sampler_batch, None, None)
    got = learner.batch_data['batch_targets'].cpu().numpy()
    ref, _ = O.mpg_v1_n_step_target(args, w, sampler_batch, T, torch.float64)
    ref32, _ = O.mpg_v1_n_step_target(args, w, sampler_batch, T, torch.float32)
    errs = dict(err=rel_l2(got, ref), spread=rel_l2(ref32, ref))
    print('MPG-v1 real-env target nfd=3', backend, errs)
    assert errs['err'] <= max(TOL_SCALAR, 2 * errs['spread']), errs


# ------------------------------------------------------------------------------------------------
# 7. PathTrackingEnv.reset(): the first observation of an episode is the environment's own observation of its state
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('nfd', [0, 3])
def test_pt_env_reset_observes_the_drawn_state(nfd):
    from oracle import mpg_oracle as O
    from mpg_b200.envs_and_models import PathTrackingEnv
    n = 256
    env = PathTrackingEnv(num_future_data=nfd, num_agent=n, seed=12)
    obs = env.reset().cpu().numpy()
    base = synthetic.make_obs(np.random.default_rng(12), PT, n)
    ref_env = O.PathTrackingEnvOracle(nfd, np.float64)
    ref_env.reset(obs)
    ref = ref_env.get_obs()
    errs = dict(obs=rel_l2(obs, ref), future=rel_l2(obs[:, 6:], ref[:, 6:]) if nfd else 0.0)
    print('PathTrackingEnv.reset() nfd', nfd, errs)
    assert np.array_equal(obs[:, :6], base), 'the six pose columns are the seeded host draw'
    assert max(errs.values()) <= TOL_STATE, errs
