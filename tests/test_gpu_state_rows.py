"""The fp32 env state is one [N,12] row per env, and the fp32 observation is a view of those rows.

A float32 CopterVecEnv keeps its state as rows (CopterBuffers.state_stride 1, state_env_stride 3); `state_planes` is
the same memory seen as [3, N, 4] planes.  fp32 steps, resets and rollouts pass no observation buffer, because the
observation is the row slice first..first+O-1 of the state the kernel has just written.  fp64 keeps vector planes
and a float32 observation buffer of its own (a cast), and step_host still writes packed rows for its device-to-host
copy.  These tests check that rows and planes step alike through the kernels' one addressing formula, that the views
stay in step with the state, and that the C ABI refuses layouts whose envs overlap."""
import ctypes as C

import numpy as np
import pytest
import torch

from gym_copter_b200._lib import CopterBuffers

VARIANTS = ['Lander3D', 'Lander2D', 'Lander1D', 'Hover3D', 'Hover2D', 'Hover1D', 'Takeoff']


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


class _LaunchSpy:
    """Stands in for the env's library handle and records the CopterBuffers of every call to `names`."""

    def __init__(self, lib, names):
        self._lib, self._names, self.buffers = lib, names, []

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if name not in self._names:
            return f

        def call(*args):
            self.buffers.append((name, args[1]._obj))
            return f(*args)
        return call


def _actions(rng, n, a, t):
    act = (1.625e-2 * (1 + 0.3 * rng.standard_normal((n, a)))).astype(np.float32)
    if t % 3 == 0:
        act[::2] = rng.uniform(-1, 1, (len(act[::2]), a))           # saturating commands: frequent endings
    return torch.as_tensor(act)


def _desynchronised(pkg, variant, n, dtype, seed=11, steps=24, spy_names=()):
    """An auto-resetting env after a randn rollout and a stretch of mixed, reset-heavy steps."""
    env = pkg.CopterVecEnv(variant, n, dtype=dtype, seed=seed, auto_reset=True, max_steps=40)
    spy = _LaunchSpy(env._lib, spy_names)
    env._lib = spy
    env.reset()
    env.rollout(57, source='randn')
    rng = np.random.default_rng(seed)
    ended, obs = 0, None
    for t in range(steps):
        obs, _, term, trunc, _ = env.step(_actions(rng, n, env.action_size, t))
        ended += int((term | trunc).sum())
    assert ended > 0
    return env, spy, obs


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS)
def test_fp32_obs_is_a_view_of_the_state_rows(pkg, variant):
    from gym_copter_b200.envs import _OBS_IDX
    n = 1000 + 7
    env, spy, obs = _desynchronised(pkg, variant, n, torch.float32,
                                    spy_names=('copter_step_f32', 'copter_reset_f32', 'copter_rollout_f32'))
    assert obs is env.obs and obs.shape == (n, env.obs_size) and obs.stride() == (12, 1)
    assert obs.untyped_storage().data_ptr() == env.state_planes.untyped_storage().data_ptr()
    assert torch.equal(obs, env.state[:, list(_OBS_IDX[variant])])
    launched = {name for name, _ in spy.buffers}
    assert launched == {'copter_step_f32', 'copter_reset_f32', 'copter_rollout_f32'}
    for name, b in spy.buffers:
        assert b.obs is None, name                                   # the kernels wrote the observation as state
        assert (b.state_stride, b.state_env_stride) == (1, 3), name


@pytest.mark.gpu
@pytest.mark.parametrize('variant', ['Lander3D', 'Hover2D'])
def test_fp64_obs_is_its_own_buffer_and_the_float32_cast(pkg, variant):
    from gym_copter_b200.envs import _OBS_IDX
    n = 300
    env, spy, obs = _desynchronised(pkg, variant, n, torch.float64, spy_names=('copter_step_f64',))
    assert obs is env.obs and obs.dtype == torch.float32 and obs.is_contiguous()
    assert obs.untyped_storage().data_ptr() != env.state_planes.untyped_storage().data_ptr()
    assert torch.equal(obs, env.state[:, list(_OBS_IDX[variant])].to(torch.float32))
    assert spy.buffers and all(b.obs == obs.data_ptr() and (b.state_stride, b.state_env_stride) == (n, 1)
                               for _, b in spy.buffers)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_row_and_plane_layouts_step_alike(pkg, dtype):
    """The same launch on a copy of the state in the other layout (fp32 env: planes; fp64 env: rows), with packed
    observation rows, gives the same bits as the env's own launch."""
    n, variant = 1000 + 7, 'Lander3D'
    env, _, _ = _desynchronised(pkg, variant, n, dtype)
    V = 4 if dtype == torch.float32 else 2
    if dtype == torch.float32:
        other, layout = env.state_planes.contiguous(), (0, 0)
    else:
        other, layout = env.state.contiguous(), (1, 12 // V)
    meta = env.meta.clone()
    obs = torch.zeros((n, env.obs_size), dtype=torch.float32, device='cuda')
    reward, done = torch.zeros(n, dtype=dtype, device='cuda'), torch.zeros(n, dtype=torch.uint8, device='cuda')
    rng = np.random.default_rng(5)
    step = env._lib.copter_step_f32 if dtype == torch.float32 else env._lib.copter_step_f64
    for t in range(12):
        a = _actions(rng, n, env.action_size, t).to(device='cuda', dtype=dtype)
        b = CopterBuffers()
        b.state, b.meta, b.action, b.obs = other.data_ptr(), meta.data_ptr(), a.data_ptr(), obs.data_ptr()
        b.reward, b.done = reward.data_ptr(), done.data_ptr()
        b.state_stride, b.state_env_stride = layout
        assert step(C.byref(env.params), C.byref(b), n, 0, env.seed_value, 1, 0, 1,
                    C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        o, r, term, _, _ = env.step(a)
        assert torch.equal(o, obs) and torch.equal(r, reward) and torch.equal(term, done.view(torch.bool))
        assert torch.equal(env.state, other.reshape(-1, n, V).permute(1, 0, 2).reshape(n, 12) if dtype == torch.float32
                           else other) and torch.equal(env.meta, meta)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
@pytest.mark.parametrize('n, chunk', [(1000, 1 << 20), (70000 + 3, 1 << 14)])
def test_step_host_returns_the_device_step_observation(pkg, dtype, n, chunk):
    """step_host (the direct path for small shards, the chunked copy pipeline past 65 536 envs) still writes packed
    observation rows: they equal what step() returns on the same seeds, and the states stay equal."""
    dev_env = pkg.CopterVecEnv('Hover3D', n, dtype=dtype, seed=4, auto_reset=True, max_steps=30)
    host_env = pkg.CopterVecEnv('Hover3D', n, dtype=dtype, seed=4, auto_reset=True, max_steps=30)
    dev_env.reset(); host_env.reset()
    rng = np.random.default_rng(8)
    for t in range(35):
        a = _actions(rng, n, 4, t).numpy().astype(np.float32 if dtype == torch.float32 else np.float64)
        o_h, r_h, term_h, _, _ = host_env.step_host(a, chunk_envs=chunk)
        o_d, r_d, term_d, _, _ = dev_env.step(torch.as_tensor(a))
        assert np.array_equal(o_h, o_d.cpu().numpy()) and np.array_equal(r_h, r_d.cpu().numpy())
        assert np.array_equal(term_h, term_d.cpu().numpy())
    assert torch.equal(host_env.state, dev_env.state)
    if dtype == torch.float32:
        assert np.array_equal(o_h, host_env.obs.cpu().numpy())        # the view follows the state on this path too
    host_env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_state_writes_show_in_obs_without_a_step(pkg, dtype):
    from gym_copter_b200.envs import _OBS_IDX
    n, variant = 257, 'Lander2D'
    env = pkg.CopterVecEnv(variant, n, dtype=dtype, seed=3)
    env.reset()
    g = torch.Generator().manual_seed(2)
    s = torch.randn((n, 12), generator=g, dtype=torch.float64) * 3
    env.set_state(s)
    idx = list(_OBS_IDX[variant])
    assert torch.equal(env.obs, s[:, idx].to(dtype).to(torch.float32).cuda())
    assert torch.equal(env.state, s.to(dtype).cuda())
    if dtype == torch.float32:                     # a write through the plane view is a write of the rows
        s2 = torch.randn((n, 12), generator=g, dtype=torch.float32)
        env.state_planes.copy_(s2.reshape(n, 3, 4).permute(1, 0, 2).cuda())
        assert torch.equal(env.obs, s2[:, idx].cuda()) and torch.equal(env.state, s2.cuda())


@pytest.mark.gpu
def test_checkpoint_round_trip_keeps_the_views(pkg):
    n = 500
    env, _, _ = _desynchronised(pkg, 'Lander3D', n, torch.float32)
    d = env.state_dict()
    assert d['state_planes'].shape == (3, n, 4)
    ref = [x.clone() for x in env.step(torch.full((n, 4), 0.02))[:3]]
    other = pkg.CopterVecEnv('Lander3D', n, seed=0, max_steps=40)
    other.load_state_dict(d)
    assert torch.equal(other.obs, d['obs']) and torch.equal(other.state_planes, d['state_planes'])
    got = other.step(torch.full((n, 4), 0.02))[:3]
    assert all(torch.equal(x, y) for x, y in zip(ref, got))


@pytest.mark.gpu
@pytest.mark.parametrize('kernel', ['1', '0'])
def test_policy_on_rows_equals_policy_on_planes(pkg, kernel, monkeypatch):
    """FusedMLPPolicy reads the env's rows (copter_policy_mlp_strided_f32); copter_policy_mlp_f32 on a plane-major
    copy of the same state gives the same actions, bit for bit, with either policy kernel."""
    monkeypatch.setenv('COPTER_B200_POLICY_TC', kernel)
    n = 4099
    env, _, _ = _desynchronised(pkg, 'Lander3D', n, torch.float32)
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=5)
    rows = pkg.FusedMLPPolicy(env, pol.net, out_scale=0.5, out_offset=0.25)().clone()
    planes = env.state_planes.contiguous()
    action = torch.full((n, 4), float('nan'), device='cuda')
    p = [q.data_ptr() for m in pol.net if isinstance(m, torch.nn.Linear) for q in (m.weight, m.bias)]
    assert env._lib.copter_policy_mlp_f32(planes.data_ptr(), n, n, 0, 64, *p, C.c_float(0.5), C.c_float(0.25),
                                          action.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    assert torch.equal(rows, action)


def test_overlapping_state_layouts_are_refused():
    """The launchers check the state layout before anything else about the launch: an overlapping layout is
    COPTER_E_RANGE, and a valid one gets as far as the variant check (an unknown variant here, so nothing is
    launched and no GPU is needed)."""
    from gym_copter_b200 import _lib, default_params
    lib, p = _lib.load(), default_params()
    b = CopterBuffers()
    b.state, b.meta, b.action, b.reward, b.done = 256, 256, 256, 256, 256       # never dereferenced
    bad_variant = 99
    for stride, env_stride, ok in ((0, 0, True), (64, 1, True), (63, 1, False), (1, 3, True), (1, 2, False),
                                   (2, 3, False), (1, 4, True), (200, 3, True), (191, 3, False)):
        b.state_stride, b.state_env_stride = stride, env_stride
        want = -2 if ok else -4                                               # COPTER_E_VARIANT / COPTER_E_RANGE
        assert lib.copter_step_f32(C.byref(p), C.byref(b), 64, 0, 0, 1, bad_variant, 1, None) == want, (stride, env_stride)
        assert lib.copter_reset_f32(C.byref(p), C.byref(b), 64, bad_variant, 0, None) == want, (stride, env_stride)
    for stride, env_stride, ok in ((1, 6, True), (1, 5, False), (64, 1, True)):          # fp64: 6 vectors per env
        b.state_stride, b.state_env_stride = stride, env_stride
        assert lib.copter_step_f64(C.byref(p), C.byref(b), 64, 0, 0, 1, bad_variant, 1, None) == (-2 if ok else -4)
