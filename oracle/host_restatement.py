"""
TEST INFRASTRUCTURE ONLY -- ctypes front end of oracle/copter_host.cpp: the KERNELS' own arithmetic
(gym_copter_b200/csrc/copter_core.h, the header the CUDA code is built from) instantiated by g++ in
fp32 and fp64 and looped over a batch one env at a time, with the reset()/step() surface of
oracle/copter_oracle.py's EnvBatch.

It is not a second restatement of the reference (copter_oracle.py, pinned to the executed reference,
is that): it is the same arithmetic as the GPU path executed by a CPU, so that
  * the arithmetic itself can be checked against the reference-pinned oracle WITHOUT a GPU, and
  * the GPU's execution of it (fast paths, warp votes, packed pairs, the compiler) can be checked
    bit for bit on the fp32 path, where comparing against an fp64 oracle can only be done to a tolerance.
Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from .copter_oracle import OracleParams, VARIANTS

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, 'libcopter_host.so')
VARIANT_ID = {'Lander3D': 0, 'Lander2D': 1, 'Lander1D': 2, 'Hover3D': 3, 'Hover2D': 4, 'Hover1D': 5, 'Takeoff': 6}
_SHAPES = dict(VARIANTS)
_SHAPES.setdefault('Takeoff', ('takeoff', tuple(range(10)), 4, (0, 1, 2, 3)))

# field order of CopterParams (include/copter_b200.h)
_FIELDS = ('B', 'D', 'M', 'L', 'Ix', 'Iy', 'Iz', 'Jr', 'maxrpm', 'landing_vel_x', 'landing_vel_y',
           'landing_angle', 'G', 'fps', 'initial_random_force', 'out_of_bounds_penalty', 'max_angle_deg',
           'bounds', 'initial_altitude', 'target_radius', 'yaw_penalty_factor', 'xyz_penalty_factor',
           'dz_max', 'dz_penalty', 'inside_radius_bonus', 'rho', 'lift_coefficient', 'takeoff_target_altitude')


class HostParams(C.Structure):
    _fields_ = [(f, C.c_double) for f in _FIELDS] + [('max_steps', C.c_int32), ('dynamics_model', C.c_int32)]


def make_params(op=None, **kw):
    op = op or OracleParams()
    d = {f: float(getattr(op, f, 5.0 if f == 'takeoff_target_altitude' else 0.0)) for f in _FIELDS}
    p = HostParams(**d, max_steps=int(op.max_steps), dynamics_model=int(op.dynamics_model))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


_libs = {}


def load(lib=None):
    """The host instantiation: the repository's own (built here on first use), or the one at path `lib`, e.g. a
    build of a modified copter_core.h."""
    path = LIB if lib is None else os.path.abspath(lib)
    if path not in _libs:
        if lib is None:
            srcs = [os.path.join(HERE, 'copter_host.cpp'),
                    os.path.join(HERE, '..', 'gym_copter_b200', 'csrc', 'copter_core.h'),
                    os.path.join(HERE, '..', 'include', 'copter_b200.h')]
            if not os.path.exists(LIB) or any(os.path.exists(s) and os.path.getmtime(LIB) < os.path.getmtime(s) for s in srcs):
                subprocess.run(['make', '-s', '-C', HERE, 'libcopter_host.so'], check=True)
        h = C.CDLL(path)
        for f in (h.copter_host_step_f32, h.copter_host_step_f64):
            f.restype = C.c_int64
        _libs[path] = h
    return _libs[path]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


# the episode statistics of include/copter_b200.h (COPTER_STAT_*), in the order of CopterVecEnv.stats()
STAT_NAMES = ('episodes', 'return_sum', 'length_sum', 'landed', 'bonus', 'crashed', 'oob', 'angle', 'timeout', 'env_steps')
CAUSE_STATS = (('landed', 1), ('bonus', 2), ('oob', 4), ('angle', 8), ('crashed', 16), ('timeout', 32))


class HostEnvBatch:
    """N envs stepped by the host instantiation of the kernels' arithmetic.  `x` [N,12], `status`,
    `steps`, `episode` are the per-env state; obs / reward / done of the last call are attributes.

    It also keeps the ledger the kernels keep with track_stats / track_returns (`stats()`, `ep_return`):
    per ended episode one count, its length final_steps - 1 and its cause bits; every executed substep
    in env_steps; with `track_returns` the running return of each env in the env dtype, added to
    return_sum and zeroed where an episode ends (with or without auto-reset) and by reset()."""

    def __init__(self, variant, n, params=None, dtype=np.float32, seed=0, env_offset=0, auto_reset=True,
                 env_ids=None, wide=False, track_returns=False, lib=None, **param_overrides):
        self.lib = load(lib)
        self.variant, self.vid, self.n = variant, VARIANT_ID[variant], int(n)
        self.obs_size, self.act_size = len(_SHAPES[variant][1]), _SHAPES[variant][2]
        self.dtype = np.dtype(dtype)
        self.f32 = self.dtype == np.float32
        self.p = params if isinstance(params, HostParams) else make_params(params, **param_overrides)
        self.seed, self.auto_reset, self.wide = int(seed), bool(auto_reset), bool(wide)
        self.env_ids = (np.arange(n, dtype=np.uint64) + np.uint64(env_offset) if env_ids is None
                        else np.ascontiguousarray(env_ids, dtype=np.uint64))
        self.x = np.zeros((n, 12), self.dtype)
        self.status, self.steps = np.zeros(n, np.int32), np.zeros(n, np.int32)
        self.episode = np.zeros(n, np.uint32)
        self.obs = np.zeros((n, self.obs_size), np.float32)
        self.final_obs = np.zeros((n, self.obs_size), np.float32)
        self.reward, self.done = np.zeros(n, self.dtype), np.zeros(n, np.uint8)
        self.cause, self.executed = np.zeros(n, np.uint8), np.zeros(n, np.int32)
        self.final_steps = np.zeros(n, np.int32)
        self._ever_reset = False
        self.ep_return = np.zeros(n, self.dtype) if track_returns else None
        self.ledger = dict.fromkeys(STAT_NAMES, 0)
        self.ledger['return_sum'] = 0.0

    def reset(self, force=None, keep_episode=None):
        """keep_episode=None mirrors the product's host shell: the first reset starts every env at
        episode 0, later ones continue each env's episode counter (COPTER_F_KEEP_EPISODE)."""
        keep = self._ever_reset if keep_episode is None else bool(keep_episode)
        fn = self.lib.copter_host_reset_f32 if self.f32 else self.lib.copter_host_reset_f64
        fn(C.byref(self.p), self.vid, int(self.wide), C.c_int64(self.n), _p(self.x), _p(self.status), _p(self.steps),
           _p(self.episode), int(keep), _p(self.obs))
        self._ever_reset = True
        if self.ep_return is not None:
            self.ep_return[:] = 0
        return self.obs

    def step(self, action, k_substeps=1, force=None):
        a = np.ascontiguousarray(action, self.dtype).reshape(self.n, self.act_size)
        f = None if force is None else np.ascontiguousarray(force, self.dtype).reshape(self.n, 3)
        fn = self.lib.copter_host_step_f32 if self.f32 else self.lib.copter_host_step_f64
        executed = fn(C.byref(self.p), self.vid, int(self.wide), C.c_int64(self.n), _p(self.x), _p(self.status), _p(self.steps),
                      _p(self.episode), _p(a), _p(self.env_ids), C.c_uint64(self.seed & 0xFFFFFFFFFFFFFFFF), _p(f),
                      int(k_substeps), int(self.auto_reset), _p(self.obs), _p(self.reward), _p(self.done), _p(self.cause),
                      _p(self.executed), _p(self.final_obs), _p(self.final_steps))
        assert executed >= 0
        self._book(self.done.view(np.bool_))
        return self.obs, self.reward, self.done.view(np.bool_), {
            'cause': self.cause, 'executed': self.executed, 'final_obs': self.final_obs, 'final_steps': self.final_steps}

    def _book(self, ended):
        led = self.ledger
        led['episodes'] += int(ended.sum())
        led['length_sum'] += int((self.final_steps[ended].astype(np.int64) - 1).sum())
        for name, bit in CAUSE_STATS:
            led[name] += int(((self.cause & bit) != 0)[ended].sum())
        led['env_steps'] += int(self.executed.astype(np.int64).sum())
        if self.ep_return is not None:
            self.ep_return += self.reward                  # one rounding in the env dtype, as the kernels' `ret += total`
            led['return_sum'] += float(self.ep_return[ended].astype(np.float64).sum())
            self.ep_return[ended] = 0

    def stats(self):
        """The ledger with the keys (and the two means) of CopterVecEnv.stats()."""
        out = {k: float(v) for k, v in self.ledger.items()}
        ep = max(out['episodes'], 1.0)
        out['mean_return'], out['mean_length'] = out['return_sum'] / ep, out['length_sum'] / ep
        return out


class HostDynamicsBatch:
    """Dynamics.setMotors driven directly (the restatement of copter_dynamics_*)."""

    def __init__(self, n, params=None, dtype=np.float64, lib=None, **param_overrides):
        self.lib = load(lib)
        self.n, self.dtype = int(n), np.dtype(dtype)
        self.p = params if isinstance(params, HostParams) else make_params(params, **param_overrides)
        self.x = np.zeros((n, 12), self.dtype)
        self.status = np.full(n, 1, np.uint8)
        self.ticks = np.zeros(n, np.int32)
        self.perturb = np.zeros((n, 6), self.dtype)

    def set_state(self, state):
        self.x[:] = np.asarray(state, self.dtype)
        self.status[:] = np.where(self.x[:, 4] < 0, 3, 1)

    def set_perturb(self, force):
        self.perturb[:] = np.asarray(force, self.dtype) / self.dtype.type(self.p.M)

    def set_motors(self, motors):
        m = np.ascontiguousarray(np.broadcast_to(np.asarray(motors, self.dtype), (self.n, 4)))
        fn = self.lib.copter_host_dynamics_f32 if self.dtype == np.float32 else self.lib.copter_host_dynamics_f64
        fn(C.byref(self.p), C.c_int64(self.n), _p(self.x), _p(self.status), _p(self.ticks), _p(self.perturb), _p(m))


def sincos_f32(a):
    a = np.ascontiguousarray(a, np.float32)
    s, c = np.empty_like(a), np.empty_like(a)
    load().copter_host_sincos_f32(_p(a), C.c_int64(a.size), _p(s), _p(c))
    return s, c
