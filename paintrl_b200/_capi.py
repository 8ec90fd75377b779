"""ctypes binding of the C ABI declared in include/paintrl.h.

The shared library is built in-tree by `paintrl_b200.build` (nvcc, sm_100a) as
`paintrl_b200/libpaintrl_b200.so`.  There is no CPU fallback: `lib()` raises if the library is
missing, and `paintrl_create` fails if there is no CUDA device.
"""
import ctypes
import os

PAINTRL_ABI_VERSION = 2
PAINTRL_STATE_SCALARS = 12

LIB_NAME = 'libpaintrl_b200.so'
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int32_p = ctypes.POINTER(ctypes.c_int32)


class PaintrlPartPack(ctypes.Structure):
    _fields_ = [
        ('abi_version', ctypes.c_int32),
        ('width', ctypes.c_int32), ('height', ctypes.c_int32),
        ('axis0', ctypes.c_int32), ('axis1', ctypes.c_int32),
        ('n_texels', ctypes.c_int32),
        ('texel_pos', c_double_p), ('texel_ij', c_int32_p),
        ('n_planes', ctypes.c_int32),
        ('plane_n', c_double_p), ('plane_off', c_double_p),
        ('n_vertices', ctypes.c_int32),
        ('vertices', c_double_p), ('vtri_start', c_int32_p), ('vtri_idx', c_int32_p),
        ('n_tris', ctypes.c_int32),
        ('tri_a', c_double_p), ('tri_v0', c_double_p), ('tri_v1', c_double_p),
        ('tri_d00', c_double_p), ('tri_d01', c_double_p), ('tri_d11', c_double_p),
        ('tri_inv_denom', c_double_p), ('tri_n', c_double_p),
        ('range0_min', ctypes.c_double), ('range0_max', ctypes.c_double),
        ('range1_min', ctypes.c_double), ('range1_max', ctypes.c_double),
        ('length_width_ratio', ctypes.c_double),
        ('grid_granularity', ctypes.c_int32),
        ('grid_lo', c_double_p), ('grid_hi', c_double_p),
        ('n_starts', ctypes.c_int32),
        ('start_pos', c_double_p), ('start_normal', c_double_p),
        ('status_init', ctypes.c_int32),
        ('texel_nn_rep', c_int32_p),
    ]


class PaintrlConfig(ctypes.Structure):
    _fields_ = [
        ('abi_version', ctypes.c_int32),
        ('action_mode', ctypes.c_int32),
        ('action_shape', ctypes.c_int32),
        ('discrete_granularity', ctypes.c_int32),
        ('discrete_table', c_double_p),
        ('obs_mode', ctypes.c_int32),
        ('obs_grad', ctypes.c_int32),
        ('color_mode', ctypes.c_int32),
        ('termination_mode', ctypes.c_int32),
        ('switch_threshold', ctypes.c_double),
        ('expected_episode_length', ctypes.c_int32),
        ('episode_max_length', ctypes.c_int32),
        ('turning_penalty', ctypes.c_int32),
        ('overlap_penalty', ctypes.c_int32),
        ('max_possible_point', ctypes.c_double),
        ('auto_reset', ctypes.c_int32),
        ('seed', ctypes.c_uint64),
        ('paint_method', ctypes.c_int32),
        ('n_beams', ctypes.c_int32),
        ('beam_plain', c_double_p),
    ]


class PaintrlStats(ctypes.Structure):
    _fields_ = [('env_steps', ctypes.c_uint64), ('episodes_ended', ctypes.c_uint64),
                ('footprint_texels', ctypes.c_uint64), ('kernel_launches', ctypes.c_uint64),
                ('ray_full_scans', ctypes.c_uint64), ('move_bailouts', ctypes.c_uint64)]


class PaintrlParamConfig(ctypes.Structure):
    _fields_ = [('abi_version', ctypes.c_int32), ('size', ctypes.c_int32), ('max_len', ctypes.c_int32),
                ('termination_by_repeat', ctypes.c_int32), ('obs_mode', ctypes.c_int32), ('auto_reset', ctypes.c_int32)]


class PaintrlPolicyConfig(ctypes.Structure):
    _fields_ = [('abi_version', ctypes.c_int32), ('obs_dim', ctypes.c_int32), ('n_out', ctypes.c_int32), ('discrete', ctypes.c_int32),
                ('capacity', ctypes.c_int32), ('seed', ctypes.c_uint64)] + [(k, ctypes.POINTER(ctypes.c_float)) for k in ('w1', 'b1', 'w2', 'b2', 'w3', 'b3')]


class PaintrlPpoConfig(ctypes.Structure):
    _fields_ = [('abi_version', ctypes.c_int32), ('obs_dim', ctypes.c_int32), ('n_out', ctypes.c_int32), ('discrete', ctypes.c_int32),
                ('max_minibatch', ctypes.c_int32), ('clip_param', ctypes.c_float), ('vf_clip_param', ctypes.c_float),
                ('vf_loss_coeff', ctypes.c_float), ('entropy_coeff', ctypes.c_float)]


# name -> (restype, argtypes); every symbol include/paintrl.h declares
_VP = ctypes.c_void_p
_I32 = ctypes.c_int32
SIGNATURES = {
    'paintrl_create': (ctypes.c_int, [ctypes.POINTER(PaintrlPartPack), ctypes.POINTER(PaintrlConfig),
                                      _I32, _I32, ctypes.POINTER(_VP)]),
    'paintrl_destroy': (None, [_VP]),
    'paintrl_num_envs': (_I32, [_VP]),
    'paintrl_obs_dim': (_I32, [_VP]),
    'paintrl_action_dim': (_I32, [_VP]),
    'paintrl_num_texels': (_I32, [_VP]),
    'paintrl_status_bytes': (_I32, [_VP]),
    'paintrl_state_bytes_per_env': (ctypes.c_int64, [_VP]),
    'paintrl_reset': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _VP]),
    'paintrl_set_pose': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _VP, _VP]),
    'paintrl_step': (ctypes.c_int, [_VP] * 11),
    'paintrl_step_subset': (ctypes.c_int, [_VP, _VP, _I32, _I32] + [_VP] * 10),
    'paintrl_step_host': (ctypes.c_int, [_VP] * 9),
    'paintrl_step_host_submit': (ctypes.c_int, [_VP, _I32] + [_VP] * 8),
    'paintrl_step_host_submit_range': (ctypes.c_int, [_VP, _I32, _I32, _I32] + [_VP] * 8),
    'paintrl_step_host_wait': (ctypes.c_int, [_VP, _I32]),
    'paintrl_get_state': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _VP, _VP, _VP]),
    'paintrl_set_state': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _VP, _VP, _VP]),
    'paintrl_job_status': (ctypes.c_int, [_VP, _VP, _VP]),
    'paintrl_stats': (ctypes.c_int, [_VP, ctypes.POINTER(PaintrlStats)]),
    'paintrl_rasterize_texels': (ctypes.c_int, [_VP, _VP, _VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP, _VP, _VP]),
    'paintrl_silhouette_march': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP, _VP]),
    'paintrl_param_create': (ctypes.c_int, [ctypes.POINTER(PaintrlParamConfig), _I32, _I32, ctypes.POINTER(_VP)]),
    'paintrl_param_destroy': (None, [_VP]),
    'paintrl_param_obs_dim': (_I32, [_VP]),
    'paintrl_param_reset': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP]),
    'paintrl_param_step': (ctypes.c_int, [_VP] * 9),
    'paintrl_param_tables': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _VP]),
    'paintrl_param_stats': (ctypes.c_int, [_VP, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64),
                                           ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(_I32)]),
    'paintrl_policy_create': (ctypes.c_int, [ctypes.POINTER(PaintrlPolicyConfig), _I32, ctypes.POINTER(_VP)]),
    'paintrl_policy_destroy': (None, [_VP]),
    'paintrl_policy_act': (ctypes.c_int, [_VP, _VP, _I32, _VP, _VP, _VP, _VP, _I32, _VP]),
    'paintrl_policy_num_params': (_I32, [_I32, _I32]),
    'paintrl_policy_set_params': (ctypes.c_int, [_VP, _VP, _VP]),
    'paintrl_ppo_create': (ctypes.c_int, [ctypes.POINTER(PaintrlPpoConfig), _I32, ctypes.POINTER(_VP)]),
    'paintrl_ppo_destroy': (None, [_VP]),
    'paintrl_ppo_grad': (ctypes.c_int, [_VP, _VP, _VP, _I32] + [_VP] * 7 + [ctypes.c_float, _VP, _VP, _VP]),
    'paintrl_ppo_forward': (ctypes.c_int, [_VP, _VP, _VP, _I32, _VP, _VP, _VP]),
    'paintrl_adam_step': (ctypes.c_int, [_VP, _VP, _VP, _VP, _I32, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, _I32, _VP]),
    'paintrl_last_error': (ctypes.c_char_p, []),
    'paintrl_abi_version': (_I32, []),
}

_lib = None


def lib():
    """Load libpaintrl_b200.so (once).  Raises if it has not been built: no fallback."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                '%s is missing: build the CUDA library first (python -m paintrl_b200.build); '
                'paintrl_b200 has no CPU fallback' % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        if handle.paintrl_abi_version() != PAINTRL_ABI_VERSION:
            raise RuntimeError('ABI mismatch between %s and paintrl_b200._capi' % LIB_PATH)
        _lib = handle
    return _lib


class PaintrlError(RuntimeError):
    pass


def check(code):
    if code != 0:
        msg = lib().paintrl_last_error()
        raise PaintrlError('paintrl error %d: %s' % (code, msg.decode() if msg else '?'))
