"""
ctypes binding of libcopter_b200.so (include/copter_b200.h).  There is NO fallback: if the
library is missing or a launch fails, the caller gets an exception.
"""
import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
# COPTER_B200_LIB: developer knob used by tools/sweep.py to time alternative builds
LIB_PATH = os.environ.get('COPTER_B200_LIB') or os.path.join(PKG, 'libcopter_b200.so')

ABI_VERSION = 6
STATS_LEN = 16
STATS_SLOTS = 64
F_AUTO_RESET, F_KEEP_EPISODE = 1, 2
MAX_STEPS_LIMIT, MAX_STEPS_LIMIT_WIDE = 2046, 0x3FFFFFFE
MODEL_LIFT, MODEL_GYRO = 1, 2
CAUSE_LANDED, CAUSE_BONUS, CAUSE_OOB, CAUSE_ANGLE, CAUSE_CRASHED, CAUSE_TIMEOUT = 1, 2, 4, 8, 16, 32
STATUS_CRASHED, STATUS_LANDED, STATUS_LEVELING, STATUS_AIRBORNE = 0, 1, 2, 3
VARIANT_IDS = {'Lander3D': 0, 'Lander2D': 1, 'Lander1D': 2, 'Hover3D': 3, 'Hover2D': 4, 'Hover1D': 5, 'Takeoff': 6}
STAT_NAMES = ('episodes', 'return_sum', 'length_sum', 'landed', 'bonus', 'crashed', 'oob',
              'angle', 'timeout', 'env_steps')


class CopterParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        'B', 'D', 'M', 'L', 'Ix', 'Iy', 'Iz', 'Jr', 'maxrpm',
        'landing_vel_x', 'landing_vel_y', 'landing_angle', 'G',
        'fps', 'initial_random_force', 'out_of_bounds_penalty', 'max_angle_deg', 'bounds',
        'initial_altitude',
        'target_radius', 'yaw_penalty_factor', 'xyz_penalty_factor', 'dz_max', 'dz_penalty',
        'inside_radius_bonus', 'rho', 'lift_coefficient', 'takeoff_target_altitude')] + [
        ('max_steps', C.c_int32), ('dynamics_model', C.c_int32)]


class CopterBuffers(C.Structure):
    _fields_ = [('state', C.c_void_p), ('meta', C.c_void_p), ('action', C.c_void_p),
                ('obs', C.c_void_p), ('reward', C.c_void_p), ('done', C.c_void_p),
                ('init_force', C.c_void_p), ('ep_return', C.c_void_p), ('stats', C.c_void_p),
                ('final_obs', C.c_void_p), ('cause', C.c_void_p), ('state_stride', C.c_int64),
                ('meta_hi', C.c_void_p), ('state_env_stride', C.c_int64)]


class CopterActionSource(C.Structure):
    _fields_ = [('kind', C.c_int32), ('reserved', C.c_int32), ('scale', C.c_double), ('offset', C.c_double)]


class CopterPidGains(C.Structure):
    _fields_ = [(n, C.c_double) for n in ('rate_kp', 'rate_ki', 'rate_kd', 'rate_windup', 'rate_big',
                                          'pos_kp', 'pos_ki', 'pos_kd', 'pos_windup', 'pos_target',
                                          'descent_kp', 'descent_kd',
                                          'alt_kp', 'alt_ki', 'alt_kd', 'alt_windup', 'alt_target')]


class CopterMlpPolicy(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('w1', 'b1', 'w2', 'b2', 'w3', 'b3')] + [
        ('hidden', C.c_int32), ('out_scale', C.c_float), ('out_offset', C.c_float), ('action_std', C.c_void_p)]


SOURCE_KINDS = {'const': 0, 'randn': 1, 'uniform': 2, 'pid': 3, 'pid_hover': 4}


class CopterError(RuntimeError):
    pass


_ARG_ERRORS = {-1: 'COPTER_E_ARG (null or missing buffer)', -2: 'COPTER_E_VARIANT',
               -3: 'COPTER_E_ALIGN (buffer not 16-byte aligned)', -4: 'COPTER_E_RANGE'}

_lib = None


def load():
    """Loads the library once. Raises CopterError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CopterError(
            '%s is missing: build it with `python -m gym_copter_b200.build` (needs nvcc). '
            'gym_copter_b200 has no CPU or PyTorch fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    if os.environ.get('COPTER_B200_LIB'):
        # developer builds timed by tools/sweep.py may predate the newest entry points
        class _Tolerant:
            def __init__(self, real):
                self.__dict__['_real'] = real

            def __getattr__(self, name):
                try:
                    return getattr(self._real, name)
                except AttributeError:
                    return C.CFUNCTYPE(C.c_int)(lambda *a: -1)
        lib = _Tolerant(lib)
    P, B, i64, u64, vp, i32 = C.POINTER(CopterParams), C.POINTER(CopterBuffers), C.c_int64, C.c_uint64, C.c_void_p, C.c_int
    lib.copter_abi_version.restype = i32
    lib.copter_default_params.argtypes = [P]
    lib.copter_default_params.restype = None
    for f in (lib.copter_obs_size, lib.copter_action_size):
        f.argtypes, f.restype = [i32], i32
    for f in (lib.copter_reset_f32, lib.copter_reset_f64):
        f.argtypes, f.restype = [P, B, i64, i32, i32, vp], i32
    for f in (lib.copter_step_f32, lib.copter_step_f64):
        f.argtypes, f.restype = [P, B, i64, i64, u64, i32, i32, i32, vp], i32
    for f in (lib.copter_dynamics_f32, lib.copter_dynamics_f64):
        f.argtypes, f.restype = [P, vp, vp, vp, vp, vp, i64, vp], i32
    for f in (lib.copter_reset_force_f32, lib.copter_reset_force_f64):
        f.argtypes, f.restype = [P, vp, vp, i64, i64, u64, vp], i32
    for f in (lib.copter_rollout_f32, lib.copter_rollout_f64):
        f.argtypes, f.restype = [P, B, C.POINTER(CopterActionSource), i64, i64, u64, i64, i32, i32, i32, vp, vp, vp,
                                 C.POINTER(CopterPidGains), vp, vp, vp, vp], i32
    lib.copter_default_pid_gains.argtypes, lib.copter_default_pid_gains.restype = [C.POINTER(CopterPidGains)], None
    lib.copter_policy_mlp_f32.argtypes = [vp, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp, C.c_float, C.c_float, vp, vp]
    lib.copter_policy_mlp_f32.restype = i32
    lib.copter_policy_mlp_strided_f32.argtypes = [vp, i64, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp, C.c_float, C.c_float, vp, vp]
    lib.copter_policy_mlp_strided_f32.restype = i32
    lib.copter_policy_rollout_f32.argtypes = [P, B, C.POINTER(CopterMlpPolicy), i64, i64, u64, i64, i32, i32, i32, vp, vp, vp, vp,
                                              vp, vp, vp]
    lib.copter_policy_rollout_f32.restype = i32
    lib.copter_gae_f32.argtypes = [vp, vp, vp, vp, vp, i64, i32, C.c_float, C.c_float, vp, vp, vp]
    lib.copter_gae_f32.restype = i32
    lib.copter_value_mlp_f32.argtypes = [vp, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp, C.c_uint32, vp, vp]
    lib.copter_value_mlp_f32.restype = i32
    lib.copter_policy_logp_f32.argtypes = [u64, i64, i64, i64, i32, i32, vp, vp, vp]
    lib.copter_policy_logp_f32.restype = i32
    lib.copter_pipeline_create.argtypes, lib.copter_pipeline_create.restype = [i32, C.POINTER(vp)], i32
    lib.copter_pipeline_destroy.argtypes, lib.copter_pipeline_destroy.restype = [vp], i32
    for f in (lib.copter_step_host_f32, lib.copter_step_host_f64):
        f.argtypes, f.restype = [vp, P, B, vp, vp, vp, vp, vp, vp, i64, i64, u64, i32, i32, i32, i64, vp], i32
    if lib.copter_abi_version() != ABI_VERSION:
        raise CopterError('libcopter_b200.so ABI %d != binding ABI %d: rebuild'
                          % (lib.copter_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(code, what):
    if code == 0:
        return
    if code < 0:
        raise CopterError('%s: %s' % (what, _ARG_ERRORS.get(code, 'error %d' % code)))
    raise CopterError('%s: CUDA error %d' % (what, code))


def default_pid_gains(**overrides):
    g = CopterPidGains()
    load().copter_default_pid_gains(C.byref(g))
    for k, v in overrides.items():
        if not hasattr(g, k):
            raise TypeError('unknown PID gain %r' % k)
        setattr(g, k, float(v))
    return g


def default_params(**overrides):
    p = CopterParams()
    load().copter_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError('unknown copter parameter %r' % k)
        setattr(p, k, v)
    return p
