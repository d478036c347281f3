"""
Host-side mirror of the reference's env API for the batched CUDA step.

`CopterVecEnv` keeps the reference's `reset(seed, options) -> (obs, info)` /
`step(action) -> (obs, reward, terminated, truncated, info)` surface
(/root/reference: gym_copter/envs/task.py:77-143, gym_copter/envs/lander.py:25-37) with a
leading env dimension, in the style of gymnasium.vector.VectorEnv (`num_envs`,
`single_observation_space`, `single_action_space`).  All arithmetic happens in
libcopter_b200.so; PyTorch only owns the device memory and the stream.  There is no CPU
path: constructing an env without a CUDA device or without the built library raises.

`Lander` (and `Lander2D`, `Hover3D`, ...) are the single-env facades: one env, numpy in and
out, python float reward / bool done -- the shapes the reference's callers (lander.py:29-64)
consume.
"""

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import CopterActionSource, CopterBuffers, CopterError, SOURCE_KINDS, VARIANT_IDS, STAT_NAMES

_OBS_IDX = {'Lander3D': tuple(range(10)), 'Lander2D': (2, 3, 4, 5, 6, 7), 'Lander1D': (4, 5),
            'Hover3D': tuple(range(12)), 'Hover2D': (2, 3, 4, 5, 6, 7), 'Hover1D': (4, 5),
            'Takeoff': tuple(range(10))}
_ACT_SIZE = {'Lander3D': 4, 'Lander2D': 2, 'Lander1D': 1, 'Hover3D': 4, 'Hover2D': 2, 'Hover1D': 1, 'Takeoff': 4}
# attic/gym_copter/envs/takeoff.py:45-55: starts on the ground (state zeros -> LANDED), no reset perturbation
_VARIANT_DEFAULTS = {'Takeoff': dict(initial_altitude=0.0, initial_random_force=0.0, fps=50.0)}         # :21 FRAMES_PER_SECOND = 50
_ALL_NAMES = ['X', 'dX', 'Y', 'dY', 'Z', 'dZ', 'Phi', 'dPhi', 'Theta', 'dTheta', 'Psi', 'dPsi']


class Box:
    """Duck-typed stand-in for gymnasium.spaces.Box (gymnasium is not installed in this
    image); the real class is used instead when importable."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.low = np.full(shape, low, dtype)
        self.high = np.full(shape, high, dtype)
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return np.random.uniform(lo, hi).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

    def __repr__(self):
        return 'Box(%s, %s, %s, %s)' % (self.low.min(), self.high.max(), self.shape, self.dtype)


def _make_box(low, high, shape):
    try:
        from gymnasium import spaces          # pragma: no cover (absent in this image)
        if not getattr(__import__('gymnasium'), '__shim__', False):
            return spaces.Box(low, high, shape=shape, dtype=np.float32)
    except Exception:
        pass
    return Box(low, high, shape)


class CopterVecEnv:
    """
    N independent copter envs stepped in lockstep on one GPU.

    variant      'Lander3D' (the reference's live `Lander`), 'Lander2D', 'Lander1D',
                 'Hover3D', 'Hover2D', 'Hover1D' (SURVEY.md 2.2), 'Takeoff' (the attic take-off env,
                 attic/gym_copter/envs/takeoff.py: unclipped commands, starts LANDED, reward =
                 change of -|altitude - 5|, only the step limit ends an episode)
    dtype        torch.float32 (throughput path) or torch.float64 (trajectory-exact path)
    k_substeps   reference steps fused per `step()` under one action (frame-skip)
    auto_reset   same-step auto-reset: a finished env reports done/terminal reward and is
                 replaced by a fresh reset state whose observation is returned
    env_offset   global id of env 0 of this shard (keys the per-env Philox reset stream, so
                 results do not depend on how the batch is sharded over GPUs)
    track_stats  accumulate episode statistics on the device (see `stats()`)
    track_returns  also keep a running per-env episode return (one more T[N] array read and
                 written per step) so that `stats()` reports return sums / means
    keep_final_obs  also record the terminal observation of finished envs (`info['final_obs']`)
    write_obs    False: step() returns None for the observation, and the fp64 step kernel and
                 step_host skip the [N,O] observation write.  On the fp32 path the observation is a
                 view of the state rows (`obs`), which the kernels never write twice
    report_cause  record why each env finished (`info['cause']`, COPTER_CAUSE_* bits) and report
                 the env's own step limit as `truncated` the way gymnasium's
                 TimeLimit(max_episode_steps) wrapper does for the reference (gym_copter/__init__.py:9-13)
    wide_counters  keep the step counter (30 bits) and the episode index (32 bits) in a second
                 uint32 per env instead of the packed 11 + 19 bits: any `max_steps` the reference takes
                 (task.py:35) and no repetition of an env's reset-force stream after 2^19 episodes.
                 Switched on automatically when max_steps > 2046
    kwargs       any CopterParams field, e.g. initial_altitude=5, max_steps=500 (task.py:32-38)
    """

    metadata = {'render_modes': ['human', 'rgb_array'], 'render_fps': 100}
    FRAMES_PER_SECOND = 100

    def __init__(self, variant='Lander3D', num_envs=1, dtype=torch.float32, device=None, seed=0,
                 env_offset=0, k_substeps=1, auto_reset=True, track_stats=False,
                 track_returns=False, keep_final_obs=False, write_obs=True, report_cause=False,
                 wide_counters=None, **params):
        if variant not in VARIANT_IDS:
            raise ValueError('unknown variant %r' % (variant,))
        if dtype not in (torch.float32, torch.float64):
            raise ValueError('dtype must be torch.float32 or torch.float64')
        self._lib = _lib.load()
        if not torch.cuda.is_available():
            raise CopterError('gym_copter_b200 needs a CUDA device (there is no CPU fallback)')
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != 'cuda':
            raise CopterError('device must be a CUDA device')
        self.variant, self.num_envs, self.dtype = variant, int(num_envs), dtype
        self.seed_value, self.env_offset = int(seed), int(env_offset)
        self.k_substeps, self.auto_reset = int(k_substeps), bool(auto_reset)
        self.params = _lib.default_params(**dict(_VARIANT_DEFAULTS.get(variant, {}), **params))
        self.wide = bool(self.params.max_steps > _lib.MAX_STEPS_LIMIT) if wide_counters is None else bool(wide_counters)
        self.FRAMES_PER_SECOND = self.params.fps
        self.TARGET_RADIUS = self.params.target_radius
        self.obs_size, self.action_size = len(_OBS_IDX[variant]), _ACT_SIZE[variant]
        self.STATE_NAMES = [_ALL_NAMES[j] for j in _OBS_IDX[variant]]
        self.single_observation_space = _make_box(-np.inf, np.inf, (self.obs_size,))
        self.single_action_space = _make_box(-1, 1, (self.action_size,))
        self.observation_space = _make_box(-np.inf, np.inf, (self.num_envs, self.obs_size))
        self.action_space = _make_box(-1, 1, (self.num_envs, self.action_size))
        self.viewer = None
        self.launches = 0           # kernels launched by this env (bench.py's gpu_launches)

        n, dev = self.num_envs, self.device
        V = 4 if dtype == torch.float32 else 2
        self._f32 = dtype == torch.float32
        # `state_planes` is the state seen as [12/V, N, V] vector planes; the kernels take its layout from its strides
        # (_state_layout, include/copter_b200.h "Memory layout").  fp32: one [N,12] row per env, and the observation
        # is the row slice first..first+O-1, so the step kernel writes it once, as state (125 instead of 165 B per
        # Lander3D env-step).  fp64: the observation is a cast, a buffer of its own, so rows would save nothing, and
        # the planes are kept: rows' 96-byte stride made the fp64 step 16 % slower (DESIGN.md, "State layout").
        if self._f32:
            rows = torch.zeros((n, 12), dtype=dtype, device=dev)
            self.state_planes = rows.as_strided((12 // V, n, V), (V, 12, 1))
            first = _OBS_IDX[variant][0]
            self.obs = rows[:, first:first + self.obs_size]
        else:
            self.state_planes = torch.zeros((12 // V, n, V), dtype=dtype, device=dev)
            self.obs = torch.zeros((n, self.obs_size), dtype=torch.float32, device=dev)
        self.meta = torch.zeros(n, dtype=torch.int32, device=dev)
        self.meta_hi = torch.zeros(n, dtype=torch.int32, device=dev) if self.wide else None
        # packed [N,O] rows the kernels write the observation into: fp64 `obs`; fp32 step_host's device-side
        # staging rows, made by host_buffers()
        self._obs_rows = None if self._f32 else self.obs
        self.reward = torch.zeros(n, dtype=dtype, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._truncated = torch.zeros(n, dtype=torch.bool, device=dev)
        self._truncated_host = np.zeros(n, np.bool_)
        self._action = torch.zeros((n, self.action_size), dtype=dtype, device=dev)
        track_stats = track_stats or track_returns
        self.ep_return = torch.zeros(n, dtype=dtype, device=dev) if track_returns else None
        self._stats = torch.zeros((_lib.STATS_SLOTS, _lib.STATS_LEN), dtype=torch.float64, device=dev) if track_stats else None
        self.final_obs = torch.zeros((n, self.obs_size), dtype=torch.float32, device=dev) if keep_final_obs else None
        self.write_obs = bool(write_obs)
        self.cause = torch.zeros(n, dtype=torch.uint8, device=dev) if report_cause else None
        self._force = None
        self._is_reset = False
        self._pipeline = None
        self._host = None
        self.rollout_step = 0       # global step index of the on-device action streams
        self.controller = None      # PID memories, allocated by rollout(source='pid' [N,16] | 'pid_hover' [N,24])

    # ---- plumbing -----------------------------------------------------------------------

    def _buffers(self, action=None, force=None, reward=None, done=None, device=False):
        """The launch's CopterBuffers.  device=True: a launch whose observation stays on the device, which on the
        fp32 path is the state itself, so the kernel is given no packed observation rows to write."""
        b = CopterBuffers()
        b.state, b.meta = self.state_planes.data_ptr(), self.meta.data_ptr()
        b.state_stride, b.state_env_stride = self._state_layout()
        b.action = action.data_ptr() if action is not None else None
        rows = None if device and self._f32 else self._obs_rows
        b.obs = rows.data_ptr() if rows is not None and (self.write_obs or action is None) else None
        b.cause = self.cause.data_ptr() if (self.cause is not None and action is not None) else None
        b.reward = (self.reward if reward is None else reward).data_ptr()
        b.done = (self.done if done is None else done).data_ptr()
        b.init_force = force.data_ptr() if force is not None else None
        b.ep_return = self.ep_return.data_ptr() if self.ep_return is not None else None
        b.stats = self._stats.data_ptr() if self._stats is not None else None
        b.final_obs = self.final_obs.data_ptr() if self.final_obs is not None else None
        b.meta_hi = self.meta_hi.data_ptr() if self.meta_hi is not None else None
        return b

    def _state_layout(self):
        """(state_stride, state_env_stride) of the C ABI: vectors between planes and between envs."""
        V = self.state_planes.shape[2]
        return self.state_planes.stride(0) // V, self.state_planes.stride(1) // V

    def _stream(self):
        # (the raw handle: torch.cuda.current_stream() builds a Stream object, several microseconds of a 25 us single-env step)
        raw = getattr(torch._C, '_cuda_getCurrentRawStream', None)
        if raw is not None and self.device.index is not None:
            return C.c_void_p(raw(self.device.index))
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _as_action(self, action):
        n, a = self.num_envs, self.action_size
        if isinstance(action, torch.Tensor):
            t = action
            if t.device != self.device or t.dtype != self.dtype:
                t = t.to(device=self.device, dtype=self.dtype)
        else:
            t = torch.as_tensor(np.asarray(action), dtype=self.dtype).to(self.device)
        if t.numel() != n * a:
            raise ValueError('action must have shape (%d, %d), got %s' % (n, a, tuple(t.shape)))
        t = t.reshape(n, a)
        if not t.is_contiguous() or t.data_ptr() % 16:
            self._action.copy_(t)
            t = self._action
        return t

    # ---- reference API ------------------------------------------------------------------

    def reset(self, seed=None, options=None, force=None):
        """
        Resets every env (envs/task.py:145-197).  The reset force of env i is the Philox draw for
        (seed, global env id, episode index).  The first reset() -- and any reset(seed=...), which
        re-keys the stream (the reference's seed argument is dead code, task.py:147) -- starts every
        env at episode 0, so a seeded reset is reproducible; every other reset() moves each env on to
        its NEXT episode index, so the reference's caller loop `env.reset()` once per episode
        (lander.py:29) sees a new perturbation every time, as it does with the reference's
        np.random.uniform (task.py:175-184,199-202).  `force` ([N,3], newtons) injects the reset
        perturbation instead of the Philox draw -- it is then used for every episode of the env
        until `reset()` is called without it.
        """
        keep = self._is_reset and seed is None
        if seed is not None:
            self.seed_value = int(seed)
        self._force = None
        if force is not None:
            f = torch.as_tensor(np.asarray(force) if not isinstance(force, torch.Tensor) else force)
            self._force = f.to(device=self.device, dtype=self.dtype).reshape(self.num_envs, 3).contiguous()
        with torch.cuda.device(self.device):
            fn = self._lib.copter_reset_f32 if self._f32 else self._lib.copter_reset_f64
            b = self._buffers(device=True)
            _lib.check(fn(C.byref(self.params), C.byref(b), self.num_envs, VARIANT_IDS[self.variant],
                          _lib.F_KEEP_EPISODE if keep else 0, self._stream()), 'copter_reset')
        self.launches += 1
        self._is_reset = True
        if self.controller is not None:
            self.controller.zero_()
        return self.obs, {}

    def step(self, action, reward_out=None, done_out=None, cause_out=None, final_obs_out=None):
        """
        One batched `_Task.step` (envs/task.py:77-137), k_substeps times under one action.
        Returns (obs f32 [N,O], reward [N], terminated bool [N], truncated bool [N], info).
        The returned tensors are the env's own output buffers: they are overwritten by the
        next step (clone them to keep them) -- on the fp32 path the observation is a view of the
        env state, so it is overwritten by the next step and must not be written into -- or pass `reward_out` ([N], env dtype) and
        `done_out` ([N] uint8) to have the kernel write this step's reward / done flags
        straight into a slice of a rollout buffer.  `cause_out` ([N] uint8) and `final_obs_out`
        ([N,O] f32) do the same for the ending's COPTER_CAUSE_* bits (0 where the episode goes
        on; reported as info['cause'] and `truncated` as with report_cause) and the terminal
        observation (written only where an episode ended; info['final_obs']).
        """
        if not self._is_reset:
            raise CopterError('step() called before reset()')    # gymnasium's OrderEnforcing
        t = self._as_action(action)
        n = self.num_envs
        for o, dt, numel in ((reward_out, self.dtype, n), (done_out, torch.uint8, n), (cause_out, torch.uint8, n),
                             (final_obs_out, torch.float32, n * self.obs_size)):
            if o is not None and (o.dtype != dt or o.numel() != numel or not o.is_contiguous()
                                  or o.device != self.device):
                raise ValueError('reward_out/done_out/cause_out/final_obs_out must be contiguous [N] tensors of the env dtype / '
                                 'uint8 / uint8 and an [N,O] float32 tensor on the env device')
        with torch.cuda.device(self.device):
            fn = self._lib.copter_step_f32 if self._f32 else self._lib.copter_step_f64
            b = self._buffers(t, self._force, reward_out, done_out, device=True)
            if cause_out is not None:
                b.cause = cause_out.data_ptr()
            if final_obs_out is not None:
                b.final_obs = final_obs_out.data_ptr()
            _lib.check(fn(C.byref(self.params), C.byref(b), self.num_envs, self.env_offset,
                          self.seed_value & 0xFFFFFFFFFFFFFFFF, self.k_substeps,
                          VARIANT_IDS[self.variant], _lib.F_AUTO_RESET if self.auto_reset else 0,
                          self._stream()), 'copter_step')
        self.launches += 1
        info = {}
        final_obs = self.final_obs if final_obs_out is None else final_obs_out
        if final_obs is not None:
            info['final_obs'] = final_obs
        truncated = self._truncated
        cause = self.cause if cause_out is None else cause_out
        if cause is not None:
            info['cause'] = cause
            truncated = (cause & _lib.CAUSE_TIMEOUT) != 0
        return (self.obs if self.write_obs else None, self.reward if reward_out is None else reward_out,
                (self.done if done_out is None else done_out).view(torch.bool), truncated, info)

    # ---- fused multi-step rollout with on-device action sources -----------------------

    def rollout(self, n_steps, source='const', scale=None, offset=None, record_rewards=False,
                record_dones=False, record_actions=False, pid_gains=None, record_causes=False,
                record_final_obs=False):
        """
        `n_steps` env steps in ONE kernel launch, the commands generated on the device:
          source='const'    action = offset                 (default offset 1.625e-2: the
                                                             reference heuristic, lander.py:21,42)
          source='randn'    action = offset + scale*N(0,1)  (default scale 1.625e-2, offset 0:
                                                             `lander.py --random`)
          source='uniform'  action = offset + scale*U(-1,1) (default scale 1: the action space)
          source='pid'      action = offset + scale*mixer(PID heuristic of attic/mars/lander3d.py:64-87
                            on the previous observation); `pid_gains` = dict of CopterPidGains
                            overrides; controller memories live in `self.controller` [N,16]
                            (2-D / 1-D variants: attic/heuristic/lander2d.py, lander1d.py)
          source='pid_hover' the hover demo's heuristic (attic/mars/hover3d.py:65-92: roll/pitch/yaw
                            rate PIDs, position hold, altitude hold at `alt_target` = 5 m; 2-D / 1-D:
                            attic/heuristic/hover2d.py, hover1d.py); of the four-motor variants
                            Hover3D only; `self.controller` is [N,24].  scale=0.03312 (twice the hover
                            command) holds the live vehicle at the target with the reference's gains
        Step for step identical to `n_steps` calls of step() with k_substeps=1 on the same
        commands.  Returns a dict: 'obs' (after the last step), 'reward_sum' [N], 'done_any'
        [N] bool, plus 'rewards' [T,N], 'dones' [T,N] bool, 'actions' [T,N,A] when recorded, and
        the episode endings a learner needs to bootstrap a truncation:
          'causes' [T,N] uint8      (record_causes) COPTER_CAUSE_* bits of the episode that ended on
                                    step t, 0 where it goes on; `causes & CAUSE_TIMEOUT` is the
                                    step limit (gymnasium's `truncated`), any other ending terminates
          'final_obs' [T,N,O] f32   (record_final_obs) the terminal observation where causes != 0
                                    (with auto-reset obs of step t + 1 is the next episode's first);
                                    zeros elsewhere
        """
        if not self._is_reset:
            raise CopterError('rollout() called before reset()')
        if source not in SOURCE_KINDS:
            raise ValueError('source must be one of %s' % sorted(SOURCE_KINDS))
        d_scale, d_off = {'const': (0.0, 1.625e-2), 'randn': (1.625e-2, 0.0), 'uniform': (1.0, 0.0),
                          'pid': (1.0, 0.0), 'pid_hover': (1.0, 0.0)}[source]
        gains = None
        if source in ('pid', 'pid_hover'):
            if source == 'pid_hover' and self.action_size == 4 and self.obs_size != 12:
                raise CopterError('the 3-D hover heuristic reads the yaw rate: Hover3D (12-component observation) only')
            width = 24 if source == 'pid_hover' else 16
            if self.controller is None or self.controller.shape[1] != width:
                self.controller = torch.zeros((self.num_envs, width), dtype=self.dtype, device=self.device)
            gains = _lib.default_pid_gains(**(pid_gains or {}))
        src = CopterActionSource(SOURCE_KINDS[source], 0, d_scale if scale is None else float(scale),
                                 d_off if offset is None else float(offset))
        n, T = self.num_envs, int(n_steps)
        out = {}
        rew = torch.empty((T, n), dtype=self.dtype, device=self.device) if record_rewards else None
        dn = torch.empty((T, n), dtype=torch.uint8, device=self.device) if record_dones else None
        act = torch.empty((T, n, self.action_size), dtype=self.dtype, device=self.device) if record_actions else None
        cause = torch.empty((T, n), dtype=torch.uint8, device=self.device) if record_causes else None
        fin = torch.zeros((T, n, self.obs_size), dtype=torch.float32, device=self.device) if record_final_obs else None
        with torch.cuda.device(self.device):
            fn = self._lib.copter_rollout_f32 if self._f32 else self._lib.copter_rollout_f64
            b = self._buffers(None, self._force, device=True)
            _lib.check(fn(C.byref(self.params), C.byref(b), C.byref(src), n, self.env_offset,
                          self.seed_value & 0xFFFFFFFFFFFFFFFF, self.rollout_step, T,
                          VARIANT_IDS[self.variant], _lib.F_AUTO_RESET if self.auto_reset else 0,
                          rew.data_ptr() if rew is not None else None,
                          dn.data_ptr() if dn is not None else None,
                          act.data_ptr() if act is not None else None,
                          C.byref(gains) if gains is not None else None,
                          self.controller.data_ptr() if self.controller is not None else None,
                          cause.data_ptr() if cause is not None else None,
                          fin.data_ptr() if fin is not None else None,
                          self._stream()), 'copter_rollout')
        self.launches += 1
        self.rollout_step += T
        out.update(obs=self.obs, reward_sum=self.reward, done_any=self.done.view(torch.bool))
        if rew is not None:
            out['rewards'] = rew
        if dn is not None:
            out['dones'] = dn.view(torch.bool)
        if act is not None:
            out['actions'] = act
        if cause is not None:
            out['causes'] = cause
        if fin is not None:
            out['final_obs'] = fin
        return out

    # ---- host-array API (numpy in / numpy out, as the reference's callers use it) ------

    def host_buffers(self):
        """Page-locked host arrays (numpy views) the host-array step reads and fills:
        dict(action [N,A], obs [N,O] f32, reward [N], done [N] uint8, plus cause [N] uint8 with
        report_cause and final_obs [N,O] with keep_final_obs)."""
        if self._host is None:
            n = self.num_envs
            t = {'action': torch.zeros((n, self.action_size), dtype=self.dtype).pin_memory(),
                 'obs': torch.zeros((n, self.obs_size), dtype=torch.float32).pin_memory(),
                 'reward': torch.zeros(n, dtype=self.dtype).pin_memory(),
                 'done': torch.zeros(n, dtype=torch.uint8).pin_memory()}
            if self.cause is not None:
                t['cause'] = torch.zeros(n, dtype=torch.uint8).pin_memory()
            if self.final_obs is not None:
                t['final_obs'] = torch.zeros((n, self.obs_size), dtype=torch.float32).pin_memory()
            self._host_t = t
            self._host = {k: v.numpy() for k, v in t.items()}
            if self._f32:           # the kernel writes packed rows for the device -> host copy
                self._obs_rows = torch.zeros((n, self.obs_size), dtype=torch.float32, device=self.device)
        return self._host

    def step_host(self, action=None, chunk_envs=1 << 20, n_streams=4):
        """
        `step()` for callers that live on the host: `action` is a numpy array [N,A] (or None
        when the caller has filled `host_buffers()['action']` in place, which avoids one host
        copy); returns numpy (obs, reward, terminated, truncated, info) -- views of the
        page-locked buffers, valid until the next call.  The host->device copy of the actions,
        the step kernel and the device->host copies of obs/reward/done are chunked and
        pipelined over `n_streams` CUDA streams inside copter_step_host_*.  Shards of at most 65 536 envs take a
        direct path instead: one launch whose kernel reads the commands from and writes its results to the
        page-locked host buffers themselves (the env's device-side reward / done tensors and the fp64 obs are
        then not refreshed by this call; state and counters are, and so is the fp32 obs, a view of the state).
        """
        if not self._is_reset:
            raise CopterError('step() called before reset()')
        h = self.host_buffers()
        if action is not None and action is not h['action']:
            a = np.asarray(action)
            if a.size != h['action'].size:
                raise ValueError('action must have shape %s' % (h['action'].shape,))
            np.copyto(h['action'], a.reshape(h['action'].shape), casting='same_kind')
        # (small shards -- the single-env facade -- are a latency problem: the argument block is built once per
        # injected-force tensor and the device guard is skipped when this env's device is already current)
        key = None if self._force is None else self._force.data_ptr()
        prep = getattr(self, '_host_call', None)
        if prep is None or prep[0] != key:
            t = self._host_t
            b = self._buffers(self._action, self._force)
            prep = (key, b, C.byref(b), C.byref(self.params),
                    (t['action'].data_ptr(), t['obs'].data_ptr() if self.write_obs else None, t['reward'].data_ptr(), t['done'].data_ptr(),
                     t['cause'].data_ptr() if 'cause' in t else None, t['final_obs'].data_ptr() if 'final_obs' in t else None),
                    self._lib.copter_step_host_f32 if self._f32 else self._lib.copter_step_host_f64)
            self._host_call = prep

        def call():
            if self._pipeline is None:
                out = C.c_void_p()
                _lib.check(self._lib.copter_pipeline_create(int(n_streams), C.byref(out)), 'copter_pipeline_create')
                self._pipeline = out
            _lib.check(prep[5](self._pipeline, prep[3], prep[2], *prep[4],
                               self.num_envs, self.env_offset, self.seed_value & 0xFFFFFFFFFFFFFFFF,
                               self.k_substeps, VARIANT_IDS[self.variant],
                               _lib.F_AUTO_RESET if self.auto_reset else 0, int(chunk_envs), self._stream()),
                       'copter_step_host')
        if self.device.index is not None and torch.cuda.current_device() == self.device.index:
            call()
        else:
            with torch.cuda.device(self.device):
                call()
        chunk = (int(chunk_envs) + 255) // 256 * 256
        self.launches += (self.num_envs + chunk - 1) // chunk
        info = {}
        truncated = self._truncated_host
        if 'cause' in h:                # as step(): the env's own step limit is TimeLimit's `truncated`
            info['cause'] = h['cause']
            truncated = (h['cause'] & _lib.CAUSE_TIMEOUT) != 0
        if 'final_obs' in h:
            info['final_obs'] = h['final_obs']
        return (h['obs'] if self.write_obs else None), h['reward'], h['done'].view(np.bool_), truncated, info

    def close(self):
        if self.viewer is not None:
            self.viewer.close()
            self.viewer = None
        if self._pipeline is not None:
            self._lib.copter_pipeline_destroy(self._pipeline)
            self._pipeline = None

    def __del__(self):
        try:
            if getattr(self, '_pipeline', None) is not None:
                self._lib.copter_pipeline_destroy(self._pipeline)
                self._pipeline = None
        except Exception:
            pass

    def render(self, mode='human'):
        return None if self.viewer is None else self.viewer.render(mode)    # lander.py:75-77

    def set_altitude(self, altitude):
        self.params.initial_altitude = float(altitude)                      # task.py:67-69

    def seed(self, seed=None):
        self.seed_value = 0 if seed is None else int(seed)
        return [self.seed_value]

    @property
    def unwrapped(self):
        return self

    # ---- state access -------------------------------------------------------------------

    def planar_obs(self):
        """The fp32 state seen as planes, [3, N, 4] float32 (plane p holds components 4p..4p+3 of
        dynamics/__init__.py:48-59; a view of the state rows).  For Lander3D the observation is
        components 0..9, i.e. planes 0, 1 and the first two lanes of plane 2."""
        if not self._f32:
            raise CopterError('planar_obs() needs the float32 path (observations are float32)')
        return self.state_planes

    @property
    def state(self):
        """[N,12] copy of the state in the reference's component order (dynamics:48-59)."""
        return self.state_planes.permute(1, 0, 2).clone(memory_format=torch.contiguous_format).view(self.num_envs, 12)

    def set_state(self, state, status=None, steps=None):
        """
        Overwrites the 12-component state of every env ([N,12]); status follows
        Dynamics.setState (AIRBORNE iff z < 0, dynamics:215-217) unless given.  The reward
        shaping baseline (prev_shaping) is that of the new state.
        """
        s = torch.as_tensor(np.asarray(state) if not isinstance(state, torch.Tensor) else state)
        s = s.to(device=self.device, dtype=self.dtype).reshape(self.num_envs, 12)
        V = self.state_planes.shape[2]
        self.state_planes.copy_(s.reshape(self.num_envs, 12 // V, V).permute(1, 0, 2))
        m = self._meta64()
        st = torch.where(s[:, 4] < 0, 3, 1).to(torch.int64) if status is None else \
            torch.as_tensor(status, device=self.device).to(torch.int64).expand(self.num_envs)
        stp = self.steps.to(torch.int64) if steps is None else \
            torch.as_tensor(steps, device=self.device).to(torch.int64).expand(self.num_envs)
        m = (st | (stp << 2)) if self.wide else ((m & ~0x1FFF) | st | (stp << 2))
        self.meta.copy_(torch.where(m >= 2 ** 31, m - 2 ** 32, m).to(torch.int32))
        if not self._f32:           # (fp32: obs is a view of the state just written)
            self.obs.copy_(s[:, list(_OBS_IDX[self.variant])].to(torch.float32))

    def _meta64(self):
        return self.meta.to(torch.int64) & 0xFFFFFFFF

    @property
    def status(self):
        return (self._meta64() & 3).to(torch.int32)

    @property
    def steps(self):
        m = self._meta64() >> 2
        return (m if self.wide else (m & 2047)).to(torch.int32)

    @property
    def episodes(self):
        """Episode index of every env (int64: the wide counter is a full uint32)."""
        if self.wide:
            return self.meta_hi.to(torch.int64) & 0xFFFFFFFF
        return self._meta64() >> 13

    def stats(self, reduce_group=None):
        """
        Episode statistics accumulated on the device since construction (or `clear_stats()`).
        With `reduce_group` (a torch.distributed process group, or True for the default
        group) the vector is all-reduced (SUM) over the ranks first -- the only collective
        this package ever issues.
        """
        if self._stats is None:
            raise CopterError('construct the env with track_stats=True')
        v = self._stats.sum(0)
        if reduce_group is not None:
            from .sharding import all_reduce_stats
            all_reduce_stats(v, None if reduce_group is True else reduce_group)
        v = v.cpu().numpy()
        out = {k: float(v[j]) for j, k in enumerate(STAT_NAMES)}
        ep = max(out['episodes'], 1.0)
        out['mean_return'], out['mean_length'] = out['return_sum'] / ep, out['length_sum'] / ep
        return out

    def clear_stats(self):
        if self._stats is not None:
            self._stats.zero_()

    # ---- checkpoint ---------------------------------------------------------------------

    def state_dict(self):
        """Everything a restored env needs to continue bit for bit: the SoA buffers and counters, the
        Philox keys and stream positions, the injected reset force, the PID controller memories and the
        parameter block (checked on load)."""
        d = {'variant': self.variant, 'seed': self.seed_value, 'env_offset': self.env_offset,
             'dtype': str(self.dtype), 'k_substeps': self.k_substeps, 'auto_reset': self.auto_reset,
             'rollout_step': self.rollout_step, 'params': bytes(self.params),
             'state_planes': self.state_planes.clone(), 'meta': self.meta.clone(), 'obs': self.obs.clone()}
        for k in ('meta_hi', '_stats', 'ep_return', '_force', 'controller', 'cause', 'final_obs'):
            v = getattr(self, k)
            if v is not None:
                d[k.lstrip('_')] = v.clone()
        return d

    def load_state_dict(self, d):
        if d['variant'] != self.variant or d['state_planes'].shape != self.state_planes.shape \
                or d.get('dtype', str(self.dtype)) != str(self.dtype):
            raise CopterError('checkpoint does not match this env (variant / size / dtype)')
        if 'params' in d and d['params'] != bytes(self.params):
            raise CopterError('checkpoint was taken with different CopterParams (e.g. max_steps, initial_altitude): '
                              'construct the env with the same parameters')
        if ('meta_hi' in d) != (self.meta_hi is not None):
            raise CopterError('checkpoint and env disagree on wide_counters')
        self.seed_value, self.env_offset = d['seed'], d['env_offset']
        self.rollout_step = d.get('rollout_step', 0)
        self.state_planes.copy_(d['state_planes'])
        self.meta.copy_(d['meta'])
        if not self._f32:           # (fp32: obs is a view of the state just loaded)
            self.obs.copy_(d['obs'])
        for k in ('meta_hi', '_stats', 'ep_return', 'cause', 'final_obs'):
            v = getattr(self, k)
            if v is not None and k.lstrip('_') in d:
                v.copy_(d[k.lstrip('_')])
        self._force = d['force'].to(self.device).clone() if 'force' in d else None
        self.controller = d['controller'].to(self.device).clone() if 'controller' in d else None
        self._is_reset = True


def _variant_class(name):
    def __init__(self, num_envs=1, **kw):
        CopterVecEnv.__init__(self, name, num_envs, **kw)
    return type(name + 'Vec', (CopterVecEnv,), {'__init__': __init__, '__doc__': 'CopterVecEnv(%r, ...)' % name})


Lander3DVec = _variant_class('Lander3D')
Lander2DVec = _variant_class('Lander2D')
Lander1DVec = _variant_class('Lander1D')
Hover3DVec = _variant_class('Hover3D')
Hover2DVec = _variant_class('Hover2D')
Hover1DVec = _variant_class('Hover1D')
TakeoffVec = _variant_class('Takeoff')
LanderVec = Lander3DVec


class _EnvDynamics:
    """`env.dynamics` of the single-env facade: the `Dynamics` accessors the reference's callers and
    renderer use on a live env (gym_copter/dynamics/__init__.py:199-229; the env creates a fresh
    Dynamics per reset, task.py:161), served from the env's own device buffers."""

    def __init__(self, vec):
        self._vec = vec

    def getState(self):
        s = self._vec.state_planes.reshape(12).cpu().numpy().astype(np.float64)
        return dict(zip(('x', 'dx', 'y', 'dy', 'z', 'dz', 'phi', 'dphi', 'theta', 'dtheta', 'psi', 'dpsi'), s))

    def getStatus(self):
        return int(self._vec.status[0].item())

    def getTime(self):
        # ticks * dt (dynamics:219-221): one tick per executed setMotors; the env's `steps` counter is 1
        # after reset and the priming step does not tick (task.py:93,197)
        return (int(self._vec.steps[0].item()) - 1) / float(self._vec.params.fps)

    def setState(self, state):
        self._vec.set_state(np.asarray(state, np.float64).reshape(1, 12))

    def perturb(self, force):
        """dynamics:227-229 on a freshly reset env: replaces the reset force (the first three components;
        the env path perturbs x, y, z only, task.py:179-184), exactly what the oracle harness does with the
        reference (SURVEY.md 8c)."""
        f = np.asarray(force, np.float64).reshape(-1)[:3]
        self._vec._force = torch.as_tensor(f.reshape(1, 3)).to(device=self._vec.device, dtype=self._vec.dtype).contiguous()


class SingleEnv:
    """
    The reference's single-env call shapes over a one-env batch: numpy float32 obs, python
    float reward, python bool done, `truncated` always False (envs/task.py:133-137).
    No auto-reset and float64 arithmetic by default, like the reference.  Attributes of the
    reference env its callers read are served too: `pose`, `done`, `viewer`, `steps`, `spinning`,
    `dynamics` (envs/task.py:80,87,92,102,106,130,161).
    """

    def __init__(self, variant, dtype=torch.float64, **kw):
        kw.setdefault('auto_reset', False)
        self._report_truncation = bool(kw.get('report_cause', False))
        kw['report_cause'] = True                     # one byte per step: `spinning` is derived from it
        self.vec = CopterVecEnv(variant, 1, dtype=dtype, **kw)
        for k in ('observation_space', 'action_space'):
            setattr(self, k, getattr(self.vec, 'single_' + k))
        self.STATE_NAMES, self.TARGET_RADIUS = self.vec.STATE_NAMES, self.vec.TARGET_RADIUS
        self.FRAMES_PER_SECOND, self.metadata = self.vec.FRAMES_PER_SECOND, self.vec.metadata
        self.viewer, self.done = None, False
        self.spinning = False                         # task.py:87,92: any motor commanded on the last step
        self._landed_before = False
        self.dynamics = _EnvDynamics(self.vec)
        self._host = self.vec.host_buffers()        # page-locked action / obs / reward / done of the one env

    @property
    def unwrapped(self):
        return self

    @property
    def steps(self):
        """The env's own step counter (task.py:128-130,191): 1 right after reset()."""
        return int(self.vec.steps[0].item())

    @property
    def pose(self):
        """(x, y, z, phi, theta, psi) as envs/task.py:102 sets it for the renderer thread; read from
        the device on demand (psi is not part of the Lander observation), so a plain step() loop does
        not pay for it."""
        s = self.vec.state_planes.reshape(12).cpu().numpy()         # one env: component order
        return (s[0], s[2], s[4], s[6], s[8], s[10])

    def reset(self, seed=None, options=None, force=None):
        obs, info = self.vec.reset(seed, options, None if force is None else np.asarray(force).reshape(1, 3))
        self.done, self.spinning, self._landed_before = False, False, False
        return obs[0].cpu().numpy(), info

    def step(self, action):
        # one library call per step: the command goes in and observation / reward / done / cause come back
        # through the page-locked buffers of copter_step_host_* (H2D + kernel + D2H + one stream sync)
        h = self._host
        a = np.asarray(action, dtype=h['action'].dtype).reshape(-1)
        h['action'][0, :] = a
        obs, r, term, trunc, info = self.vec.step_host(None, n_streams=1)
        self.done = bool(term[0])
        # `spinning` as the reference leaves it after the step (task.py:86-92,121-125, lander.py:64-67):
        # off when the status BEFORE the step was LANDED, or CRASHED without an out-of-bounds / over-angle
        # ending; otherwise "some motor is commanded"
        c = int(info['cause'][0])
        spin = bool(np.clip(a, 0, 1).sum() > 0)
        if (c & _lib.CAUSE_LANDED) or self._landed_before:
            spin = False
        elif (c & _lib.CAUSE_CRASHED) and not (c & (_lib.CAUSE_OOB | _lib.CAUSE_ANGLE)):
            spin = False
        self.spinning = spin
        # variants where LANDED does not end the episode (hover): remember it for the next step; the
        # device is only asked once the vehicle is at ground level (NED: z >= 0)
        zi = self.vec.STATE_NAMES.index('Z')
        self._landed_before = (self.vec.variant.startswith('Hover') and float(obs[0, zi]) >= 0.0
                               and self.dynamics.getStatus() == _lib.STATUS_LANDED)
        return obs[0].copy(), float(r[0]), self.done, bool(trunc[0]) if self._report_truncation else False, {}

    def set_altitude(self, altitude):
        self.vec.set_altitude(altitude)

    def render(self, mode='human'):
        return None if self.viewer is None else self.viewer.render(mode)

    def close(self):
        self.vec.close()


def _single_class(name):
    def __init__(self, **kw):
        SingleEnv.__init__(self, name, **kw)
    return type(name, (SingleEnv,), {'__init__': __init__})


Lander = _single_class('Lander3D')
Lander3D = Lander
Lander2D = _single_class('Lander2D')
Lander1D = _single_class('Lander1D')
Hover3D = _single_class('Hover3D')
Hover2D = _single_class('Hover2D')
Hover1D = _single_class('Hover1D')
Takeoff = _single_class('Takeoff')


def make(env_id, **kw):
    """`gym.make`-shaped constructor: 'Lander-v0' / 'gym_copter:Lander-v0' (gym_copter/__init__.py:9-13)
    and the batched ids '<Variant>Vec-v0'."""
    name = env_id.split(':')[-1]
    name = name[:-3] if name.endswith('-v0') else name
    table = {'Lander': Lander, 'Lander3D': Lander, 'Lander2D': Lander2D, 'Lander1D': Lander1D,
             'Hover3D': Hover3D, 'Hover2D': Hover2D, 'Hover1D': Hover1D, 'Takeoff': Takeoff, 'TakeoffVec': TakeoffVec,
             'LanderVec': Lander3DVec, 'Lander3DVec': Lander3DVec, 'Lander2DVec': Lander2DVec,
             'Lander1DVec': Lander1DVec, 'Hover3DVec': Hover3DVec, 'Hover2DVec': Hover2DVec,
             'Hover1DVec': Hover1DVec}
    if name not in table:
        raise ValueError('unknown env id %r' % env_id)
    return table[name](**kw)
