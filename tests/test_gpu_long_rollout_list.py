"""Rollout lists of up to 64 entries (mpg_set_rollout_list + n_list = MPG_LIST_FROM_HANDLE), on both kernel families,
against the fp64 oracle: dense MPG-v2 lists over the default horizon, full BPTT, 64-entry lists that are unsorted and
repeat steps, a 70-step horizon, a 260-step horizon (steps past the kernels' 256-step tables), many ragged tiles, the
forward-only kernel, the return statistics, MPGLearner and the trainer.  Lists of 8 or fewer entries take the params
struct as before; the same list through either path gives bit-identical results.

The bars are the suite's: per-row returns 1e-5, gradients 1e-4 relative L2, scalars 2e-5."""
import ctypes

import numpy as np
import pytest
import torch

from mpg_b200 import _lib, synthetic
from mpg_b200.config import default_args
from mpg_b200.learners.base import rule_based_weights
from tests.test_gpu_config_space import BACKENDS, IP, PT, _check_policy_grad, _handle, _inputs
from tests.util import make_batch, rel_l2

TOL_STATE, TOL_GRAD, TOL_SCALAR = 1e-5, 1e-4, 2e-5
N = 25


def _dense_weights(rng, n):
    """random weights over n entries, about a fifth of them zero and a fifth negative"""
    w = rng.uniform(0.05, 1.0, n)
    u = rng.uniform(size=n)
    w[u < 0.2] = 0.0
    w[(u >= 0.2) & (u < 0.4)] *= -1.0
    return [float(x) for x in w]


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def _reference_rule_based_weights(ite, total_ite, eta, lst):
    """mpg_learner.py:384-399 restated in numpy float64"""
    start, end = 1. - eta, 1. + eta
    lam = min(max(start + (end - start) / total_ite * ite, 0.), 1.5)
    if lam < 1.:
        biases = np.array([lam ** i for i in lst])
    else:
        biases = np.array([(2. - lam) ** (max(lst) - i) for i in lst])
    inv = 1. / (biases + 1e-8)
    e = np.exp(inv - inv.max())
    return e / e.sum()


@pytest.mark.parametrize('n', [26, 64])
@pytest.mark.parametrize('ite', [0, 2000, 4500, 9000, 20000])
def test_rule_based_weights_long_lists(n, ite):
    lst = list(range(n)) if n == 26 else list(range(1, 65))
    got = rule_based_weights(ite, 9000, 0.1, lst)
    ref = _reference_rule_based_weights(ite, 9000, 0.1, lst)
    assert got.shape == (n,) and got.dtype == np.float32
    assert np.abs(got - ref).max() <= 1e-6 * max(1.0, ref.max()), np.abs(got - ref).max()


def test_65_entries_raise_before_the_device():
    from mpg_b200.engine import Engine
    from mpg_b200.learners import MPGLearner
    e = object.__new__(Engine)      # no handle, no device: the check must come first
    lst = list(range(65))
    with pytest.raises(ValueError, match='64'):
        e.policy_grad(None, lst, [1.0] * 65)
    with pytest.raises(ValueError, match='64'):
        e.rollout_forward(None, lst)
    with pytest.raises(ValueError, match='64'):
        e.returns_stats(torch.zeros(65, 4), 4, 1)
    with pytest.raises(ValueError, match='64'):
        e.returns_tile_mean(torch.zeros(65, 4), 4, 1)
    # MPGLearner adds step 0 to a list without it: 64 entries without 0 are 65
    args = default_args('MPG-v2', PT, num_rollout_list_for_policy_update=list(range(1, 65)))
    with pytest.raises(ValueError, match='64'):
        MPGLearner(lambda **kw: pytest.fail('the policy was built'), args)


class _NoLib:
    def __getattr__(self, name):
        raise AssertionError(f'{name} called for a list the params struct holds')


@pytest.mark.parametrize('n', [0, 1, 8])
def test_short_lists_fill_the_struct(n):
    from mpg_b200.engine import Engine
    e = object.__new__(Engine)
    e.lib = _NoLib()
    lst, lw = list(range(3, 3 + n)), [0.5 + k for k in range(n)]
    p = e._params(4, 1, 3 + n, lst, lw, 0, _lib.NET_Q1, _lib.NET_POLICY, None, 0, 0, 0)
    assert p.n_list == n
    assert list(p.list)[:n] == lst and list(p.list_w)[:n] == lw
    assert ctypes.sizeof(p) == ctypes.sizeof(_lib.RolloutParams)


def test_long_list_selects_the_handle_list():
    from mpg_b200.engine import Engine
    calls = []

    class Lib:
        def mpg_set_rollout_list(self, h, n, lst, lw):
            calls.append((n, list(lst[:n]), list(lw[:n])))
            return 0
    e = object.__new__(Engine)
    e.lib, e.h = Lib(), None
    lst, lw = list(range(26)), [0.25] * 26
    p = e._params(4, 1, 25, lst, lw, 0, _lib.NET_Q1, _lib.NET_POLICY, None, 0, 0, 0)
    assert p.n_list == _lib.LIST_FROM_HANDLE == -1
    assert calls == [(26, lst, lw)]


# ------------------------------------------------------------------------------------------------
# GPU: path equivalence
# ------------------------------------------------------------------------------------------------
def _call_through_handle(e, obs, noise, lst, lw, full_bptt):
    """mpg_policy_grad with the list handed over by mpg_set_rollout_list, whatever its length"""
    rows, n = obs.shape[0], max(lst)
    e.ensure_capacity(rows, n)
    p = e._params(rows, 1, n, [], [], full_bptt, _lib.NET_Q1, _lib.NET_POLICY, None, 0, 0, 0)
    k = len(lst)
    e._check(e.lib.mpg_set_rollout_list(e.h, k, (ctypes.c_int32 * k)(*lst), (ctypes.c_float * k)(*lw)))
    p.n_list = _lib.LIST_FROM_HANDLE
    grad, ret = e.empty(e.param_count(_lib.NET_POLICY)), e.empty(k, rows)
    e._check(e.lib.mpg_policy_grad(e.h, ctypes.byref(p), ctypes.c_void_p(obs.data_ptr()),
                                   ctypes.c_void_p(noise.data_ptr()), ctypes.c_void_p(grad.data_ptr()),
                                   ctypes.c_void_p(ret.data_ptr()), e.stream))
    return grad, ret


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('full_bptt', [True, False])
def test_struct_and_handle_paths_are_bit_identical(full_bptt, backend):
    B = 700
    args = default_args('MPG-v2', PT, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, N, seed=101, double_q=True)
    _, e = _handle(args, w, backend)
    lst, lw = [25, 0, 7, 7, 13], [0.4, 0.1, -0.2, 0.3, 0.0]
    x, nz = e.dev(obs), e.dev(noise)
    g1, r1 = e.policy_grad(x, lst, lw, full_bptt=full_bptt, noise=nz)
    g2, r2 = _call_through_handle(e, x, nz, lst, lw, int(full_bptt))
    torch.cuda.synchronize()
    assert torch.equal(g1, g2) and torch.equal(r1, r2)
    # the handle list stays until replaced; a short list through the struct does not touch it
    g3, r3 = e.policy_grad(x, lst, lw, full_bptt=full_bptt, noise=nz)
    assert torch.equal(g1, g3) and torch.equal(r1, r3)


@pytest.mark.gpu
def test_abi_errors():
    args = default_args('MPG-v2', PT, replay_batch_size=64)
    w, obs, noise = _inputs(args, 64, N, seed=102, double_q=True)
    _, e = _handle(args, w, 'ffma')
    lst = (ctypes.c_int32 * 65)(*range(65))
    lw = (ctypes.c_float * 65)(*([1.0] * 65))
    assert e.lib.mpg_set_rollout_list(e.h, 65, lst, lw) == -1
    assert b'64' in e.lib.mpg_last_error(e.h)
    # an index beyond the call's horizon is refused at the call
    e.ensure_capacity(64, 30)
    assert e.lib.mpg_set_rollout_list(e.h, 12, lst, lw) == 0
    p = e._params(64, 1, 10, [], [], 0, _lib.NET_Q1, _lib.NET_POLICY, None, 0, 0, 0)
    p.n_list = _lib.LIST_FROM_HANDLE
    x, grad = e.dev(obs), e.empty(e.param_count(_lib.NET_POLICY))
    rc = e.lib.mpg_policy_grad(e.h, ctypes.byref(p), ctypes.c_void_p(x.data_ptr()), None,
                               ctypes.c_void_p(grad.data_ptr()), None, e.stream)
    assert rc == -1 and b'horizon' in e.lib.mpg_last_error(e.h)
    # a negative n_list other than MPG_LIST_FROM_HANDLE stays an error
    p.n_list = -2
    rc = e.lib.mpg_policy_grad(e.h, ctypes.byref(p), ctypes.c_void_p(x.data_ptr()), None,
                               ctypes.c_void_p(grad.data_ptr()), None, e.stream)
    assert rc == -1


# ------------------------------------------------------------------------------------------------
# GPU: dense lists against the oracle
# ------------------------------------------------------------------------------------------------
def _check_forward_rows(e, obs, noise, lst, rows_ref, label, M=1):
    fwd = e.rollout_forward(e.dev(obs), lst, M=M, noise=e.dev(noise)).cpu().numpy()
    err = max(rel_l2(fwd[k], rows_ref[k]) for k in range(len(lst)))
    print(label, 'forward-only rows, backend', e.backend, err)
    assert np.isfinite(fwd).all() and err <= TOL_STATE, err


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('B', [300, 2048])
@pytest.mark.parametrize('env_id', [PT, IP])
def test_dense_mpg_v2_first_action_vs_oracle(env_id, B, backend):
    n = N
    args = default_args('MPG-v2', env_id, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=110 + B, double_q=True)
    _, e = _handle(args, w, backend)
    lst = list(range(n + 1))
    lw = _dense_weights(np.random.default_rng(B), n + 1)
    rows_ref, _ = _check_policy_grad(e, args, w, obs, noise, lst, lw, f'dense {env_id} B={B}', full_bptt=False)
    _check_forward_rows(e, obs, noise, lst, rows_ref, f'dense {env_id} B={B}')


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_dense_full_bptt_vs_oracle(backend):
    B = 1000
    args = default_args('MPG-v2', PT, replay_batch_size=B, deriv_interval_policy=True)
    w, obs, noise = _inputs(args, B, N, seed=120, double_q=True)
    _, e = _handle(args, w, backend)
    lst = list(range(N + 1))
    _check_policy_grad(e, args, w, obs, noise, lst, _dense_weights(np.random.default_rng(121), N + 1),
                       'dense full BPTT', full_bptt=True)


LONG = {
    # 64 entries over steps 0..40, shuffled, every step at least once and 23 of them twice
    'unsorted_repeats_64': (40, lambda rng: list(rng.permutation(list(range(41)) + list(rng.choice(41, 23, False))))),
    # n = 70: 64 entries on both sides of step 64
    'n70_64': (70, lambda rng: list(rng.permutation([0, 63, 64, 65, 70] + list(rng.choice(np.arange(1, 70), 59))))),
}


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
@pytest.mark.parametrize('full_bptt', [True, False])
@pytest.mark.parametrize('case', list(LONG))
def test_long_lists_vs_oracle(case, full_bptt, backend):
    n, make = LONG[case]
    rng = np.random.default_rng(130 + n)
    lst = [int(k) for k in make(rng)]
    lw = _dense_weights(rng, len(lst))
    B = 512
    args = default_args('NADP', PT, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=131)
    _, e = _handle(args, w, backend)
    rows_ref, _ = _check_policy_grad(e, args, w, obs, noise, lst, lw, f'{case} full_bptt={full_bptt}',
                                     full_bptt=full_bptt)
    if full_bptt:
        _check_forward_rows(e, obs, noise, lst, rows_ref, case)


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_horizon_past_the_step_tables_vs_oracle(backend):
    """n = 260: steps 256.. read the list from the global FarStep table instead of the 256-step shared tables."""
    B, n = 256, 260
    lst, lw = [0, 100, 255, 256, 257, 259, 260, 260, 3], [0.1, 0.2, -0.1, 0.15, 0.0, 0.2, 0.1, 0.25, 0.1]
    args = default_args('NADP', PT, replay_batch_size=B)
    w, obs, noise = _inputs(args, B, n, seed=132)
    _, e = _handle(args, w, backend)
    rows_ref, _ = _check_policy_grad(e, args, w, obs, noise, lst, lw, 'n=260')
    _check_forward_rows(e, obs, noise, lst, rows_ref, 'n=260')


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_dense_m3_ragged_multi_wave_vs_oracle(backend):
    B, n, M = 6701, 6, 3
    args = default_args('MPG-v2', PT, replay_batch_size=B, M=M)
    w, obs, noise = _inputs(args, B, n, M=M, seed=140, double_q=True)
    _, e = _handle(args, w, backend)
    assert (B * M) % 128 != 0 and (B * M + 127) // 128 > e.num_sms
    lst = [6, 0, 1, 2, 2, 3, 4, 5, 6, 1, 0]
    lw = _dense_weights(np.random.default_rng(141), len(lst))
    rows_ref, _ = _check_policy_grad(e, args, w, obs, noise, lst, lw, 'dense M=3 multi-wave', M=M, full_bptt=False)
    _check_forward_rows(e, obs, noise, lst, rows_ref, 'dense M=3 multi-wave', M=M)


@pytest.mark.gpu
@pytest.mark.parametrize('rows', [1, 1000, 65536])
def test_returns_stats_64_entries_vs_numpy(rows):
    from mpg_b200.engine import Engine
    n_list, M = 64, 2
    e = Engine(**vars(default_args('NADP', PT)))
    rng = np.random.default_rng(150 + rows)
    ret = (rng.standard_normal((n_list, M * rows)) - 3.0).astype(np.float32)
    mean = ret.astype(np.float64).reshape(n_list, M, rows).mean(1)
    stats = e.returns_stats(e.dev(ret), rows, M).cpu().numpy()
    tile_mean = e.returns_tile_mean(e.dev(ret), rows, M).cpu().numpy()
    errs = dict(sum=rel_l2(stats[:n_list], mean.sum(1)), sumsq=rel_l2(stats[n_list:], (mean ** 2).sum(1)),
                tile_mean=rel_l2(tile_mean, mean))
    print('returns stats n_list=64 rows', rows, errs)
    assert max(errs.values()) <= TOL_STATE, errs


# ------------------------------------------------------------------------------------------------
# GPU: MPGLearner, bench size, trainer
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_mpg_learner_dense_list_vs_oracle(backend):
    from oracle import mpg_oracle as O
    from mpg_b200.learners import MPGLearner
    from mpg_b200.policy import PolicyWithQs
    B, ite = 300, 4000
    lst = list(range(1, N + 1))
    args = default_args('MPG-v2', PT, replay_batch_size=B, num_rollout_list_for_policy_update=lst)
    w = synthetic.make_policy_with_qs_weights(160, args.obs_dim, args.act_dim, 256, double_q=True)
    batch = make_batch(161, PT, B, 0)
    npol = synthetic.make_noise(np.random.default_rng(162), N, B)
    learner = MPGLearner(PolicyWithQs, args)
    learner.set_weights(w)
    e = learner.engine
    if backend == 'tc':
        if not e.tc_available():
            pytest.skip('tensor-core backend does not cover this configuration')
        e.set_backend(1)
    else:
        e.set_backend(0)
    learner.set_rollout_noise(None, npol)
    flat = np.concatenate([np.asarray(g, np.float64).ravel() for g in learner.compute_gradient(batch, None, None, ite)])
    st = learner.get_stats()
    ref = O.mpg_compute_gradient(args, w, batch, npol, ite, torch.float64)
    nQ = ref['q_grad1'].size
    p = flat[2 * nQ:] * max(st['policy_gradient_norm'], args.gradient_clip_norm) / args.gradient_clip_norm
    errs = dict(clipped=rel_l2(flat, ref['compute_gradient']), p=rel_l2(p, ref['policy_grad']),
                total_loss=rel_l2(st['policy_total_loss'], ref['total_loss']),
                value_mean=rel_l2(st['value_mean'], ref['value_mean']),
                all_losses=rel_l2(np.array(st['all_losses']), ref['minus_returns']),
                w_list=rel_l2(np.array(st['w_list']), ref['ws']),
                returns_var=float(np.abs(np.array(st['returns_var']) - ref['returns_var']).max()
                                  / np.abs(ref['returns_var']).max()))
    print('MPGLearner dense list, backend', e.backend, errs)
    assert len(st['all_losses']) == len(st['w_list']) == len(st['returns_var']) == len(lst)
    assert errs['clipped'] <= TOL_GRAD and errs['p'] <= TOL_GRAD, errs
    for k in ('total_loss', 'value_mean', 'all_losses', 'w_list', 'returns_var'):
        assert errs[k] <= TOL_SCALAR, errs


@pytest.mark.gpu
@pytest.mark.parametrize('backend', BACKENDS)
def test_bench_size_dense_list(backend):
    """B = 65,536 with the dense list and in-kernel Philox noise: bit-reproducible run to run, two half batches with
    global scaling add up to the full batch, returns and gradient against the fp64 oracle."""
    from oracle import mpg_oracle as O
    B, n, seed = 65536, N, 13
    args = default_args('MPG-v2', PT, replay_batch_size=B)
    w = synthetic.make_policy_with_qs_weights(170, args.obs_dim, args.act_dim, 256, double_q=True)
    obs = synthetic.make_obs(np.random.default_rng(171), PT, B)
    _, e = _handle(args, w, backend)
    lst = list(range(n + 1))
    lw = _dense_weights(np.random.default_rng(172), n + 1)
    x = e.dev(obs)
    kw = dict(full_bptt=False, use_philox=True, noise_seed=seed)
    g1, r1 = e.policy_grad(x, lst, lw, **kw)
    g2, r2 = e.policy_grad(x, lst, lw, **kw)
    assert torch.equal(g1, g2) and torch.equal(r1, r2), 'not bit-reproducible run to run'
    h = B // 2
    gl, _ = e.policy_grad(x[:h].contiguous(), lst, lw, global_rows=B, row_offset=0, **kw)
    gr, _ = e.policy_grad(x[h:].contiguous(), lst, lw, global_rows=B, row_offset=h, **kw)
    shard = rel_l2((gl + gr).cpu().numpy(), g1.cpu().numpy())
    nets = O.Nets(w, True, torch.float64)
    w_rest = [t.detach() for t in nets.policy]
    grad_ref, rows = None, []
    for lo in range(0, B, 8192):
        hi = min(B, lo + 8192)
        noise = synthetic.philox_normal(seed, hi - lo, n, global_rows=B, row_offset=lo)
        r = O.rollout(args, torch.float64, nets.policy, w_rest, nets.Q1, O.to_t(obs[lo:hi], torch.float64),
                      O.to_t(noise, torch.float64), n)
        loss = sum(wk * -r[k].sum() / B for k, wk in zip(lst, lw))
        gc = np.concatenate([t.numpy().ravel() for t in torch.autograd.grad(loss, nets.policy)])
        grad_ref = gc if grad_ref is None else grad_ref + gc
        rows.append(torch.stack([r[k] for k in lst]).detach().numpy())
    rows = np.concatenate(rows, 1)
    got = r1.cpu().numpy()
    errs = dict(rows=max(rel_l2(got[k], rows[k]) for k in range(len(lst))), grad=rel_l2(g1.cpu().numpy(), grad_ref),
                shard=shard)
    print('bench size dense list, backend', e.backend, errs)
    assert errs['shard'] <= 1e-5 and errs['rows'] <= TOL_STATE and errs['grad'] <= TOL_GRAD, errs


@pytest.mark.gpu
def test_trainer_smoke_dense_list():
    from mpg_b200.trainer import Trainer, parse_rollout_list
    lst = parse_rollout_list('1-25')
    assert lst == list(range(1, 26)) and parse_rollout_list('0,5,10-12') == [0, 5, 10, 11, 12]
    args = default_args('MPG-v2', PT, replay_batch_size=256, batch_size=512, num_agent=8, explore_sigma=0.1,
                        max_buffer_size=100000, replay_starts=1024, buffer_log_interval=10 ** 9, num_eval_agent=16,
                        num_eval_episode=1, fixed_steps=20, eval_interval=10 ** 9, log_interval=10 ** 9, max_iter=8,
                        log_dir=None, num_rollout_list_for_policy_update=lst)
    tr = Trainer(args)
    tr.train(args.max_iter)
    st = tr.learner.get_stats()
    assert len(st['all_losses']) == 25
    for k in ('policy_gradient_norm', 'q_gradient_norm1', 'q_loss1', 'policy_total_loss', 'value_mean'):
        assert np.isfinite(st[k]), (k, st[k])
