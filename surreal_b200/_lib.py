"""ctypes binding of libsurreal_b200.so (the C-ABI declared in include/surreal_b200.h).

The library is built in-tree by ``surreal_b200/build.py`` (nvcc, sm_100a).  There is NO fallback:
if the shared object is missing or a kernel call fails, an exception is raised.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SB200_LIB') or os.path.join(HERE, 'libsurreal_b200.so')     # SB200_LIB: a development build (tools/)
MAX_LAYERS = 4
ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2

c_f32p = C.POINTER(C.c_float)


class SB200Error(RuntimeError):
    pass


class Mlp(C.Structure):
    _fields_ = [('n_layers', C.c_int),
                ('dims', C.c_int * (MAX_LAYERS + 1)),
                ('act', C.c_int * MAX_LAYERS),
                ('W', C.c_void_p * MAX_LAYERS),
                ('b', C.c_void_p * MAX_LAYERS),
                ('ldw', C.c_int * MAX_LAYERS),
                ('aux_layer', C.c_int),
                ('aux_dim', C.c_int)]


class PPORollout(C.Structure):
    """sb200_ppo_rollout (include/surreal_b200.h)."""
    _fields_ = [('net', C.POINTER(Mlp)), ('zf_stats', C.c_void_p), ('zf_eps', C.c_float), ('log_var', C.c_void_p),
                ('log_noise', C.c_void_p), ('agent_seed', C.c_uint64), ('deterministic', C.c_int),
                ('state', C.c_void_p), ('WsT', C.c_void_p), ('WaT', C.c_void_p), ('ep_step', C.c_void_p),
                ('max_steps', C.c_int), ('env_seed', C.c_uint64), ('action', C.c_void_p), ('pd', C.c_void_p),
                ('obs_next', C.c_void_p), ('reward', C.c_void_p), ('done', C.c_void_p), ('stage_pos', C.c_void_p),
                ('stage_obs', C.c_void_p), ('stage_act', C.c_void_p), ('stage_pd', C.c_void_p),
                ('stage_rew', C.c_void_p), ('stage_done', C.c_void_p), ('o_obs', C.c_void_p), ('o_act', C.c_void_p),
                ('o_pd', C.c_void_p), ('o_rew', C.c_void_p), ('o_done', C.c_void_p), ('ev_step', C.c_void_p),
                ('ev_count', C.c_void_p), ('W', C.c_int), ('N', C.c_int), ('D', C.c_int), ('A', C.c_int),
                ('n_step', C.c_int), ('stride', C.c_int), ('T', C.c_int), ('step_counter', C.c_void_p)]


class Par(C.Structure):
    """sb200_par (include/surreal_b200.h)."""
    _fields_ = [('peers', C.c_void_p * 8), ('world', C.c_int), ('rank', C.c_int), ('max_floats', C.c_int64)]


class Epochs(C.Structure):
    """sb200_epochs (include/surreal_b200.h): argument block of the persistent learner kernel."""
    _fields_ = [('net', C.c_void_p), ('params', C.c_void_p), ('n_params', C.c_int64), ('extra_off', C.c_int),
                ('x', C.c_void_p), ('ldx', C.c_int64), ('M', C.c_int), ('zf_stats', C.c_void_p), ('zf_eps', C.c_double),
                ('x_in', C.c_void_p), ('h1', C.c_void_p), ('h2', C.c_void_p), ('out', C.c_void_p), ('d1', C.c_void_p), ('d2', C.c_void_p),
                ('dpre', C.c_void_p), ('slabs', C.c_void_p), ('splits', C.c_int), ('grad', C.c_void_p),
                ('exp_avg', C.c_void_p), ('exp_avg_sq', C.c_void_p), ('lr', C.c_void_p), ('weight_decay', C.c_double),
                ('clip_mode', C.c_int), ('clip_value', C.c_double), ('opt_workspace', C.c_void_p), ('norm_out', C.c_void_p),
                ('mode', C.c_int), ('actions', C.c_void_p), ('lda', C.c_int64), ('adv', C.c_void_p),
                ('behave_pd', C.c_void_p), ('ldb', C.c_int64), ('ref_pd', C.c_void_p), ('ldr', C.c_int64),
                ('returns', C.c_void_p), ('hyper', C.c_void_p), ('eta', C.c_double), ('kl_target', C.c_double),
                ('stop_threshold', C.c_double), ('stats', C.c_void_p), ('stop_flag', C.c_void_p), ('epochs', C.c_int),
                ('workspace', C.c_void_p), ('grid', C.c_int), ('cta_shift', C.c_int), ('par', C.c_void_p)]


class ZFilter(C.Structure):
    _fields_ = [('stats', C.c_void_p), ('eps', C.c_float)]


class Rows(C.Structure):
    _fields_ = [('x', C.c_void_p), ('x_next', C.c_void_p), ('ldx', C.c_int64), ('rows', C.c_int64),
                ('win_n', C.c_int), ('aux', C.c_void_p), ('aux_ld', C.c_int64),
                ('save_x', C.c_void_p), ('ld_save_x', C.c_int64)]


_lib = None


def _declare(lib):
    P, I, L, D, F, S = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_float, C.c_size_t
    sig = {
        'sb200_version': (I, []),
        'sb200_init': (I, []),
        'sb200_set_forward_mode': (I, [I]),
        'sb200_status_string': (C.c_char_p, [I]),
        'sb200_device_info': (I, [C.POINTER(I), C.POINTER(I), C.POINTER(I)]),
        'sb200_launch_counter': (C.c_uint64, [I]),
        'sb200_launch_counter_add': (None, [C.c_uint64]),
        'sb200_mlp_forward_f32': (I, [C.POINTER(Mlp), C.POINTER(ZFilter), C.POINTER(Rows),
                                      C.POINTER(P), C.POINTER(L), P]),
        'sb200_mlp_forward_variant_f32': (I, [C.POINTER(Mlp), C.POINTER(ZFilter), C.POINTER(Rows),
                                              C.POINTER(P), C.POINTER(L), I, P]),
        'sb200_mlp_tc5_supported': (I, [C.POINTER(Mlp), L]),
        'sb200_mlp_tc5_workspace_bytes': (S, [C.POINTER(Mlp)]),
        'sb200_mlp_forward_tc5_f32': (I, [C.POINTER(Mlp), C.POINTER(ZFilter), C.POINTER(Rows), P, L, P, P]),
        'sb200_synth_pixel_env_step_u8': (I, [P, P, I, L, I, I, P, C.c_uint64, P, P, P, P, P]),
        'sb200_synth_mixed_env_step_f32': (I, [P, P, P, P, I, I, I, I, L, I, P, C.c_uint64, P, P, P, P, P]),
        'sb200_par_buffer_bytes': (S, [L]),
        'sb200_par_alloc': (I, [L, C.POINTER(C.c_void_p), P]),
        'sb200_par_open': (I, [P, C.POINTER(C.c_void_p)]),
        'sb200_par_close': (I, [P, I]),
        'sb200_par_allreduce_f32': (I, [C.POINTER(Par), P, P, L, D, I, P, P, P]),
        'sb200_par_allreduce_f64': (I, [C.POINTER(Par), P, P, I, D, P]),
        'sb200_ppo_epochs2_supported': (I, [C.POINTER(Epochs), C.POINTER(Epochs)]),
        'sb200_ppo_epochs2_workspace_bytes': (S, [C.POINTER(Epochs), C.POINTER(Epochs)]),
        'sb200_ppo_epochs2_f32': (I, [C.POINTER(Epochs), C.POINTER(Epochs), P, P]),
        'sb200_ppo_epochs2_profile': (I, [P, C.POINTER(C.c_uint64), I, P]),
        'sb200_ppo_epochs2_cta_profile': (I, [P, C.POINTER(C.c_uint64), P]),
        'sb200_rows_zfilter_f32': (I, [P, L, L, I, I, I, P, D, P, L, P]),
        'sb200_lstm_forward_f32': (I, [P, P, P, P, P, L, I, I, I, I, P, P, P, P, P, P, P]),
        'sb200_lstm_backward_f32': (I, [P, L, P, P, P, L, P, I, I, I, P, P]),
        'sb200_conv_forward_f32': (I, [I, P, I, L, I, I, I, P, P, D, P, P]),
        'sb200_conv_backward_dw_f32': (I, [I, P, I, P, L, I, I, I, D, P, P, L, I, P]),
        'sb200_conv_backward_dx_f32': (I, [I, P, P, P, L, I, I, I, P, P]),
        'sb200_conv1_forward_u8_strided': (I, [P, L, L, I, I, I, P, P, D, P, P]),
        'sb200_conv1_backward_dw_u8_strided': (I, [P, L, P, L, I, I, I, D, P, P, L, I, P]),
        'sb200_mlp_pack_floats': (S, [C.POINTER(Mlp)]),
        'sb200_mlp_pack_tf32': (I, [C.POINTER(Mlp), P, P]),
        'sb200_mlp_forward_packed_f32': (I, [C.POINTER(Mlp), P, C.POINTER(ZFilter), C.POINTER(Rows), P, L, P]),
        'sb200_ppo_act_host_f32': (I, [C.POINTER(Mlp), C.POINTER(ZFilter), P, P, I, P, P, P, I, C.c_uint64, P, P, P, P, P, P,
                                       I, P, P, P, P, P]),
        'sb200_ppo_window_step_host_f32': (I, [P, P, P, P, P, P, P, P, I, I, I, I, I, P, P, P, P, P, P, P, P, P, P, P, P, P,
                                               P, I, P]),
        'sb200_ppo_rollout_supported': (I, [C.POINTER(Mlp), I, I]),
        'sb200_ppo_rollout_scratch_ints': (S, [I, I, I]),
        'sb200_ppo_rollout_f32': (I, [C.POINTER(PPORollout), P]),
        'sb200_ppo_rollout_commit_f32': (I, [C.POINTER(PPORollout), P, P, P, P, P, P, P, P, P]),
        'sb200_linear_bwd_dx_f32': (I, [P, L, P, I, P, L, P, L, I, I, I, P]),
        'sb200_linear_bwd_dw_f32': (I, [P, L, P, L, P, P, L, I, I, I, I, I, P]),
        'sb200_make_pd_f32': (I, [P, L, P, P, I, I, P, L, P]),
        'sb200_zfilter_update_f32': (I, [P, L, L, I, P, P]),
        'sb200_reward_filter_f32': (I, [P, L, D, D, P, P, P]),
        'sb200_gae_workspace_bytes': (S, [I, I, I]),
        'sb200_ppo_loss_workspace_bytes': (S, [I, I]),
        'sb200_ppo_policy_loss_f32': (I, [I, P, L, P, P, L, P, P, L, P, L, I, I, P, D, D, P, L, P, P, P, P, P]),
        'sb200_ppo_kl_f32': (I, [P, L, P, L, P, I, I, P, I, D, P, I, P, P]),
        'sb200_ppo_kl_apply': (I, [P, P, I, D, P, P]),
        'sb200_ppo_loss_kl_offset': (S, []),
        'sb200_moments_f32': (I, [P, L, P, P]),
        'sb200_normalize_f32': (I, [P, L, P, D, P]),
        'sb200_add_f32': (I, [P, P, L, P]),
        'sb200_value_loss_f32': (I, [P, L, P, I, P, L, P, P, P]),
        'sb200_ppo_final_stats_f32': (I, [P, L, P, P, L, P, L, P, L, I, I, P, P, P]),
        'sb200_ppo_sample_f32': (I, [P, L, P, P, P, I, I, I, C.c_uint64, P, P, P, P, P, P, I, P]),
        'sb200_ddpg_noise_f32': (I, [P, L, P, P, I, I, I, C.c_uint64, P, P, P]),
        'sb200_ddpg_target2_f32': (I, [P, P, L, P, L, P, P, L, I, I, D, P, P, P, P]),
        'sb200_ddpg_smooth_action_f32': (I, [P, L, P, I, I, D, D, C.c_uint64, P, P, L, P]),
        'sb200_ddpg_ou_noise_f32': (I, [P, L, P, P, I, I, I, C.c_uint64, P, D, D, P, P, P]),
        'sb200_synth_env_step_f32': (I, [P, P, P, P, I, I, I, I, P, C.c_uint64, P, P, P, P, P]),
        'sb200_fifo_state_bytes': (S, []),
        'sb200_ppo_window_step_f32': (I, [P, P, P, P, I, I, I, I, I, P, P, P, P, P, P, P, P, P, P, P, P, P, P, I, P]),
        'sb200_ppo_sample_assign_f32': (I, [P, L, P, P, P, I, I, I, C.c_uint64, P, P, P, P, P, P, I, P, P, P]),
        'sb200_synth_env_window_step_f32': (I, [P, P, P, P, I, I, I, I, P, C.c_uint64, P, P, P, P, I, I,
                                                P, P, P, P, P, P, P, P, P, P, P, P, P]),
        'sb200_fifo_pop': (I, [P, I, P, P, P]),
        'sb200_fifo_push': (I, [P, I, P, P]),
        'sb200_replay_gather_f32': (I, [P, L, P, P, I, P, P]),
        'sb200_replay_gather_multi_f32': (I, [P, P, P, I, P, P, I, P]),
        'sb200_uniform_state_bytes': (S, []),
        'sb200_ssar_step_f32': (I, [P, P, P, P, P, I, I, D, I, I, P, P, P, P, P, P, P, P, P, P, P, P, P, P]),
        'sb200_mt19937_state_bytes': (S, []),
        'sb200_mt19937_seed_h': (I, [P, P, I]),
        'sb200_mt19937_set_state_h': (I, [P, P, I]),
        'sb200_mt19937_get_state_h': (I, [P, P, C.POINTER(I)]),
        'sb200_mt19937_randint_fill_h': (I, [P, L, L, P]),
        'sb200_ddpg_workspace_bytes': (S, [I]),
        'sb200_ddpg_target_f32': (I, [P, P, L, P, P, L, I, I, D, P, P, P, P]),
        'sb200_ddpg_critic_loss_f32': (I, [P, L, P, I, P, L, P, P, P]),
        'sb200_ddpg_actor_seed_f32': (I, [P, L, I, P, L, P, P, P]),
        'sb200_tanh_bwd_f32': (I, [P, L, P, L, I, I, P, L, P]),
        'sb200_optim_workspace_bytes': (S, []),
        'sb200_grad_reduce_norm_f32': (I, [P, L, I, P, L, D, I, P, P, P]),
        'sb200_clip_adam_f32': (I, [P, P, P, P, L, P, D, D, D, D, I, D, P, P, P, P]),
        'sb200_soft_update_f32': (I, [P, P, L, D, P, P]),
        'sb200_ddpg_bad_action_offset': (S, []),
        'sb200_gae_window_f32': (I, [P, P, P, I, I, I, D, D, D, I, P, P, P, P]),
    }
    sig.update(_EXTRA_SIGS)
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return sig


_EXTRA_SIGS = {}


def exported_symbols():
    """Names the header declares (used by the CPU-side 'library loads and exports' test)."""
    return list(_declare(lib()).keys())


class _ProfilingProxy:
    """Wraps every C-ABI call between two CUDA events on the current stream (bench.py's live per-kernel timing;
    only meaningful for eager launches -- events cannot sit inside a captured graph)."""

    def __init__(self, real):
        self._real = real
        self.records = {}

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        if not name.endswith('_f32') and name not in ('sb200_fifo_pop', 'sb200_fifo_push', 'sb200_ppo_kl_apply',
                                                      'sb200_mlp_pack_tf32'):   # noqa: E501
            return fn
        import torch

        def wrapped(*args):
            key = name
            if name in ('sb200_mlp_forward_f32', 'sb200_mlp_forward_variant_f32'):
                key = '%s[rows=%d]' % (name, int(args[2]._obj.rows))
            elif name == 'sb200_mlp_forward_packed_f32':
                key = '%s[rows=%d]' % (name, int(args[3]._obj.rows))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*args)
            e1.record()
            self.records.setdefault(key, []).append((e0, e1))
            return rc
        return wrapped

    def report(self):
        import torch
        torch.cuda.synchronize()
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in self.records.items()}


_profiler = None


def profile_calls(enable):
    """Turn per-call CUDA-event timing on/off; returns the finished report when turning off."""
    global _profiler
    if enable:
        _profiler = _ProfilingProxy(lib())
        return None
    rep = _profiler.report() if _profiler is not None else {}
    _profiler = None
    return rep


def lib():
    global _lib
    if _profiler is not None:
        return _profiler
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SB200Error(
                'libsurreal_b200.so is not built (%s). Run `python -m surreal_b200.build` '
                '(needs nvcc); there is no CPU fallback.' % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


_device_ready = False


def ensure_device():
    """sb200_init() once per process, on first use of a compute entry."""
    global _device_ready
    if not _device_ready:
        check(lib().sb200_init(), 'sb200_init')
        _device_ready = True


def check(status, what=''):
    if status != 0:
        msg = lib().sb200_status_string(status).decode()
        raise SB200Error('%s failed: %s (status %d)' % (what or 'libsurreal_b200 call', msg, status))


def reset_call_counter():
    lib().sb200_launch_counter(1)


def call_counter_kernels():
    return int(lib().sb200_launch_counter(0))
