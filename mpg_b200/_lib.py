"""ctypes binding of libmpg_b200.so (include/mpg_b200.h). There is NO CPU fallback: if the
library is missing, cannot be loaded, or no CUDA device is present, every entry point raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MPG_B200_LIB', os.path.join(_HERE, 'libmpg_b200.so'))  # override: kernel-variant A/B runs
# the same library built with -DMPG_DEBUG_PROBES (GEMM self tests, cta_group::2 probe, clock64 timeline): tests / tools only
DEBUG_LIB_PATH = os.environ.get('MPG_B200_DBG_LIB', os.path.join(_HERE, 'libmpg_b200_dbg.so'))

MAX_OBS, MAX_LIST = 16, 8
MAX_LIST_LONG, LIST_FROM_HANDLE = 64, -1   # mpg_set_rollout_list: lists longer than the params struct holds
ENV_IDS = {'PathTracking-v0': 0, 'InvertedPendulumConti-v0': 1, 'InvertedDoublePendulum-v2': 2,
           'PathTracking-v0-real': 3}   # the ground-truth PathTrackingEnv (forward only)
NET_Q1, NET_Q2, NET_POLICY, NET_Q1_TARGET, NET_Q2_TARGET, NET_POLICY_TARGET = range(6)
ACTIVATIONS = {'elu': 0, 'relu': 1, 'tanh': 2}   # MPG_ACT_*: hidden activation of every net of a handle
HIDDEN_LAYERS = (1, 2, 3)   # mpg_create_layers: hidden layers of every net of a handle

# every symbol include/mpg_b200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    'mpg_create', 'mpg_destroy', 'mpg_last_error', 'mpg_workspace_bytes', 'mpg_num_sms', 'mpg_param_count',
    'mpg_set_weights', 'mpg_get_weights', 'mpg_policy_grad', 'mpg_rollout_forward', 'mpg_returns_stats',
    'mpg_returns_tile_mean', 'mpg_q_grad', 'mpg_policy_forward', 'mpg_q_forward', 'mpg_q_target', 'mpg_td_error',
    'mpg_model_reset', 'mpg_model_step', 'mpg_model_step_bwd', 'mpg_compute_rewards', 'mpg_state_dim',
    'mpg_clip_global_norm', 'mpg_philox_noise', 'mpg_launch_count', 'mpg_set_backend', 'mpg_get_backend',
    'mpg_set_timing', 'mpg_kernel_ms', 'mpg_wait_debug', 'mpg_adam_step', 'mpg_polyak_update', 'mpg_get_adam_state',
    'mpg_set_adam_state', 'mpg_env_sample',
    'mpg_replay_create', 'mpg_replay_destroy', 'mpg_replay_last_error', 'mpg_replay_size', 'mpg_replay_add',
    'mpg_replay_sample', 'mpg_replay_update_priorities', 'mpg_replay_tree_stats', 'mpg_q_bootstrap', 'mpg_env_step',
    'mpg_set_activation', 'mpg_get_activation', 'mpg_create_layers', 'mpg_hidden_layers', 'mpg_set_rollout_list',
]
# exported by libmpg_b200_dbg.so only (include/mpg_b200.h, #ifdef MPG_DEBUG_PROBES)
DEBUG_SYMBOLS = ['mpg_tc_selftest', 'mpg_set_profile_buffer']


class MpgConfig(ctypes.Structure):
    _fields_ = [('env', ctypes.c_int32), ('num_future_data', ctypes.c_int32), ('obs_dim', ctypes.c_int32),
                ('act_dim', ctypes.c_int32), ('hidden', ctypes.c_int32), ('policy_out_tanh', ctypes.c_int32),
                ('action_range', ctypes.c_float), ('obs_scale', ctypes.c_float * MAX_OBS),
                ('rew_scale', ctypes.c_float), ('rew_shift', ctypes.c_float), ('gamma', ctypes.c_float),
                ('max_rows', ctypes.c_int32), ('max_horizon', ctypes.c_int32)]


class RolloutParams(ctypes.Structure):
    _fields_ = [('rows', ctypes.c_int32), ('M', ctypes.c_int32), ('horizon', ctypes.c_int32),
                ('n_list', ctypes.c_int32), ('list', ctypes.c_int32 * MAX_LIST), ('list_w', ctypes.c_float * MAX_LIST),
                ('full_bptt', ctypes.c_int32), ('q_net', ctypes.c_int32), ('policy_net', ctypes.c_int32),
                ('global_rows', ctypes.c_int64), ('row_offset', ctypes.c_int64), ('noise_seed', ctypes.c_uint64),
                ('use_philox', ctypes.c_int32), ('real_env', ctypes.c_int32)]


_lib = None
_lib_dbg = None


def load(debug=False):
    """Load the shared library (once). Raises RuntimeError when it is absent: the product path
    must fail loudly rather than fall back to anything else.  debug=True loads libmpg_b200_dbg.so (the same code
    + the development probes) -- tests/test_gpu_tc.py and tools/ only."""
    global _lib, _lib_dbg
    if (debug and _lib_dbg is not None) or (not debug and _lib is not None):
        return _lib_dbg if debug else _lib
    path = DEBUG_LIB_PATH if debug else LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(
            f'{path} not found: build it first (python -c "import __graft_entry__ as g; g.build()" '
            f'or make -C mpg_b200/csrc all). mpg_b200 has no CPU fallback.')
    lib = ctypes.CDLL(path)
    vp, i32, i64, u64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_float
    P = ctypes.POINTER
    sig = {
        'mpg_create': (i32, [P(MpgConfig), P(vp)]),
        'mpg_create_layers': (i32, [P(MpgConfig), i32, P(vp)]),
        'mpg_hidden_layers': (i32, [vp]),
        'mpg_destroy': (None, [vp]),
        'mpg_last_error': (ctypes.c_char_p, [vp]),
        'mpg_workspace_bytes': (ctypes.c_size_t, [vp]),
        'mpg_num_sms': (i32, [vp]),
        'mpg_param_count': (i32, [vp, i32]),
        'mpg_set_weights': (i32, [vp, i32, P(vp), vp]),
        'mpg_get_weights': (i32, [vp, i32, P(vp), vp]),
        'mpg_set_rollout_list': (i32, [vp, i32, P(ctypes.c_int32), P(ctypes.c_float)]),
        'mpg_policy_grad': (i32, [vp, P(RolloutParams), vp, vp, vp, vp, vp]),
        'mpg_rollout_forward': (i32, [vp, P(RolloutParams), vp, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_returns_stats': (i32, [vp, vp, i32, i32, i32, vp, vp]),
        'mpg_returns_tile_mean': (i32, [vp, vp, i32, i32, i32, vp, vp]),
        'mpg_q_grad': (i32, [vp, i32, i32, i64, vp, vp, vp, vp, vp, vp]),
        'mpg_policy_forward': (i32, [vp, i32, i32, vp, vp, vp]),
        'mpg_q_forward': (i32, [vp, i32, i32, vp, vp, vp, vp]),
        'mpg_q_target': (i32, [vp, i32, i32, vp, vp, vp, vp]),
        'mpg_td_error': (i32, [vp, i32, vp, vp, vp, vp, vp, vp]),
        'mpg_model_reset': (i32, [vp, i32, vp, vp, vp]),
        'mpg_model_step': (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_model_step_bwd': (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_compute_rewards': (i32, [vp, i32, vp, vp, vp, vp]),
        'mpg_state_dim': (i32, [vp]),
        'mpg_clip_global_norm': (i32, [vp, vp, i32, f32, vp, vp]),
        'mpg_philox_noise': (i32, [vp, P(RolloutParams), vp, vp]),
        'mpg_launch_count': (u64, [vp]),
        'mpg_set_backend': (i32, [vp, i32]),
        'mpg_get_backend': (i32, [vp]),
        'mpg_set_activation': (i32, [vp, i32]),
        'mpg_get_activation': (i32, [vp]),
        'mpg_set_timing': (i32, [vp, i32]),
        'mpg_kernel_ms': (f32, [vp]),
        'mpg_tc_selftest': (i32, [vp, i32, vp, vp, vp, i32, vp]),
        'mpg_set_profile_buffer': (i32, [vp, vp]),
        'mpg_wait_debug': (i32, [vp]),
        'mpg_adam_step': (i32, [vp, i32, vp, f32, i64, f32, f32, f32, vp]),
        'mpg_polyak_update': (i32, [vp, i32, i32, f32, vp]),
        'mpg_get_adam_state': (i32, [vp, i32, vp, vp, vp]),
        'mpg_set_adam_state': (i32, [vp, i32, vp, vp, vp]),
        'mpg_env_sample': (i32, [vp, i32, i32, i32, f32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_q_bootstrap': (i32, [vp, i32, vp, f32, vp, vp, vp]),
        'mpg_env_step': (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_replay_create': (i32, [i32, i32, i32, ctypes.c_double, ctypes.c_double, P(vp)]),
        'mpg_replay_destroy': (None, [vp]),
        'mpg_replay_last_error': (ctypes.c_char_p, [vp]),
        'mpg_replay_size': (i32, [vp]),
        'mpg_replay_add': (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_replay_sample': (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        'mpg_replay_update_priorities': (i32, [vp, i32, vp, vp, vp]),
        'mpg_replay_tree_stats': (i32, [vp, P(ctypes.c_double), P(ctypes.c_double), P(ctypes.c_double), vp]),
    }
    for name, (res, args) in sig.items():
        if name in DEBUG_SYMBOLS and not debug:
            continue
        fn = getattr(lib, name)  # AttributeError if the header and the library ever diverge
        fn.restype, fn.argtypes = res, args
    if debug:
        _lib_dbg = lib
    else:
        _lib = lib
    return lib


def wait_debug():
    """Watchdog records of the kernels' mbarrier waits: None, or a list of dict(role, site=source line (+10000
    tc_gemm.cuh, +20000 tc_kernels.cuh), block, thread, parity), one per warpgroup that timed out before the launch trapped."""
    out = (ctypes.c_uint64 * 32)()
    load().mpg_wait_debug(out)
    if not out[0]:
        return None
    roles = ['epi0', 'epi1', 'epi2', 'epi3', 'row', 'producer', 'mma']
    return [dict(role=roles[k], site=int(out[4 + 4 * k]), block=int(out[5 + 4 * k]), thread=int(out[6 + 4 * k]),
                 parity=int(out[7 + 4 * k]) - 1) for k in range(7) if out[7 + 4 * k]]
