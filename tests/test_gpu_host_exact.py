"""
GPU: the fp32 kernels against the fp32 CPU instantiation of the SAME arithmetic
(gym_copter_b200/csrc/copter_core.h built by g++, oracle/copter_host.cpp) -- BIT FOR BIT.

north_star asks for done / terminated flags and step counts that are bit-exact.  Against the fp64
numpy reference that can only hold away from thresholds (an fp32 rounding may flip `z > 0 && dz > 0`,
`|x| >= 10`, `|phi| >= pi/4` one step early or late; tests/test_host_restatement.py measures that rate
on the CPU).  What the GPU path itself owes is that it EXECUTES the fp32 arithmetic it is defined by
exactly: every fast path (K = 1 specialisation, straight-line substeps, calm streaks), every warp
vote, and ptxas' code generation have to reproduce the plain one-env-at-a-time loop.  Here, on every action stream, variant and K:
    state (all 12 components), observation, flight status, step counter, episode index, done flag,
    ending cause and terminal observation: identical bits / values, ZERO flips allowed;
    reward: the device takes the two square roots and the quotient of the shaping difference on the
    MUFU unit (<= 2 ulp each), the host with IEEE sqrt / division: max <= 5e-5 (a few ulps of the larger
    shaping term where the position and yaw terms cancel; north_star allows 1e-4), mean <= 1e-7.
The fp64-oracle comparisons to 1e-4 / 1e-9 stay in tests/test_gpu_parity.py.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.host_restatement import HostDynamicsBatch, HostEnvBatch       # noqa: E402
from oracle.copter_oracle import ALL_VARIANTS, OracleParams               # noqa: E402

HOVER = 0.016560178212092172


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


def mixed_streams(rng, n, t, a, takeoff=False):
    act = np.empty((t, n, a), np.float32)
    for i in range(n):
        kind = i % 4
        if kind == 0:
            act[:, i] = 1.625e-2
        elif kind == 1:
            act[:, i] = 1.625e-2 * rng.standard_normal((t, a))
        elif kind == 2:
            act[:, i] = HOVER * (1 + 0.1 * rng.uniform(-1, 1, (t, a)))
        else:
            act[:, i] = rng.uniform(-1, 1, (t, a))
    if takeoff:
        act = (np.abs(act) * np.where(np.arange(n) % 4 == 3, 0.03, 1.0)[None, :, None]).astype(np.float32)
        act[:, ::5] *= -1
    return act


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_same(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t):
    x = env.state.cpu().numpy()
    assert np.array_equal(bits(x), bits(host.x)), (t, np.argwhere(bits(x) != bits(host.x))[:5])
    assert np.array_equal(term.cpu().numpy(), h_done), t
    assert np.array_equal(env.status.cpu().numpy(), host.status), t
    assert np.array_equal(env.steps.cpu().numpy(), host.steps), t
    assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64)), t
    assert np.array_equal(bits(obs.cpu().numpy()), bits(h_obs)), t
    if 'cause' in info:
        assert np.array_equal(info['cause'].cpu().numpy(), h_info['cause']), t
    if 'final_obs' in info and h_done.any():
        assert np.array_equal(bits(info['final_obs'].cpu().numpy()[h_done]), bits(h_info['final_obs'][h_done])), t
    rr = r.cpu().numpy()
    err = np.abs(rr - h_r) / np.maximum(np.abs(h_r), 1.0)
    assert err.max() <= 5e-5 and err.mean() <= 1e-7, (t, float(err.max()), float(err.mean()))


@pytest.mark.parametrize('k', [1, 2, 3, 16])
@pytest.mark.parametrize('variant', ['Lander3D', 'Lander2D', 'Lander1D', 'Hover3D', 'Hover2D', 'Takeoff'])
def test_fp32_step_kernels_equal_the_host_instantiation(pkg, variant, k):
    N, T, seed, off = 2048 + 77, max(1000 // k, 120), 99, 123456789012
    rng = np.random.default_rng(11 + k)
    A = ALL_VARIANTS[variant][2]
    act = mixed_streams(rng, N, T, A, takeoff=variant == 'Takeoff')
    kw = dict(max_steps=150) if variant == 'Takeoff' else {}
    env = pkg.CopterVecEnv(variant, N, dtype=torch.float32, seed=seed, env_offset=off, k_substeps=k,
                           report_cause=True, keep_final_obs=True, **kw)
    hkw = dict(initial_altitude=0.0, initial_random_force=0.0, fps=50.0, max_steps=150) if variant == 'Takeoff' else {}   # the shell's Takeoff defaults
    host = HostEnvBatch(variant, N, OracleParams(**hkw), dtype=np.float32, seed=seed, env_offset=off)
    obs, _ = env.reset()
    assert np.array_equal(bits(obs.cpu().numpy()), bits(host.reset()))
    episodes = 0
    for t in range(T):
        obs, r, term, trunc, info = env.step(torch.as_tensor(act[t]))
        h_obs, h_r, h_done, h_info = host.step(act[t], k)
        assert_same(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t)
        assert np.array_equal(trunc.cpu().numpy(), (h_info['cause'] & 32) != 0)
        episodes += int(h_done.sum())
    assert episodes >= N


@pytest.mark.parametrize('k', [1, 5])
def test_fp32_bit_exact_without_auto_reset_with_statistics_and_wide_counters(pkg, k):
    """The other kernel instantiations: statistics on, no auto-reset (envs keep stepping past done like
    the reference), wide counters with a step limit past the 11-bit field, injected reset forces."""
    N, T = 1500 + 13, 700 // k
    rng = np.random.default_rng(3)
    act = mixed_streams(rng, N, T, 4)
    force = rng.uniform(-30, 30, (N, 3)).astype(np.float32)
    env = pkg.CopterVecEnv('Lander3D', N, dtype=torch.float32, seed=1, k_substeps=k, auto_reset=False,
                           track_returns=True, report_cause=True, keep_final_obs=True, max_steps=3000)
    assert env.wide
    host = HostEnvBatch('Lander3D', N, OracleParams(max_steps=3000), dtype=np.float32, seed=1, auto_reset=False, wide=True)
    env.reset(force=force); host.reset()
    for t in range(T):
        obs, r, term, trunc, info = env.step(torch.as_tensor(act[t]))
        h_obs, h_r, h_done, h_info = host.step(act[t], k, force=force)
        assert_same(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t)
    # second reset(): every env moves on to its next episode index (new Philox force), on both sides
    env.auto_reset = host.auto_reset = True
    env.reset(); host.reset()
    assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64)) and (host.episode == 1).all()
    for t in range(40):
        obs, r, term, trunc, info = env.step(torch.as_tensor(act[t]))
        h_obs, h_r, h_done, h_info = host.step(act[t], k)
        assert_same(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t)


def test_two_consecutive_resets_draw_different_forces(pkg):
    """ADVICE r1: reset() used to send every env back to episode 0, replaying the same perturbation."""
    env = pkg.CopterVecEnv('Lander3D', 256, dtype=torch.float64, seed=5, auto_reset=False)
    a = torch.full((256, 4), HOVER, dtype=torch.float64)
    env.reset(); env.step(a); s1 = env.state.clone()
    env.reset(); env.step(a); s2 = env.state.clone()
    assert (s1[:, 1] != s2[:, 1]).all() and (env.episodes == 1).all()
    env.reset(seed=5); env.step(a)                       # a seeded reset restarts the stream: reproducible
    assert torch.equal(env.state, s1) and (env.episodes == 0).all()
    single = pkg.make('gym_copter:Lander-v0')
    firsts = []
    for _ in range(3):
        single.reset()
        firsts.append(single.step(HOVER * np.ones(4))[0][1])
    assert len(set(firsts)) == 3


@pytest.mark.parametrize('source', ['uniform', 'randn', 'const'])
def test_fp32_rollout_kernel_equals_the_host_instantiation(pkg, source):
    """copter_rollout_f32 (commands drawn on the device): replay the recorded commands on the host."""
    N, T = 1000 + 9, 300
    env = pkg.CopterVecEnv('Lander3D', N, dtype=torch.float32, seed=77, env_offset=5 << 32)
    host = HostEnvBatch('Lander3D', N, dtype=np.float32, seed=77, env_offset=5 << 32)
    env.reset(); host.reset()
    for chunk in range(3):
        out = env.rollout(T // 3, source=source, record_actions=True, record_dones=True, record_rewards=True)
        acts, dones, rews = out['actions'].cpu().numpy(), out['dones'].cpu().numpy(), out['rewards'].cpu().numpy()
        for t in range(T // 3):
            h_obs, h_r, h_done, _ = host.step(acts[t], 1)
            assert np.array_equal(dones[t], h_done), (chunk, t)
            assert (np.abs(rews[t] - h_r) / np.maximum(np.abs(h_r), 1)).max() <= 5e-5
        assert np.array_equal(bits(env.state.cpu().numpy()), bits(host.x))
        assert np.array_equal(env.steps.cpu().numpy(), host.steps) and np.array_equal(env.status.cpu().numpy(), host.status)
        assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64))
        assert np.array_equal(bits(out['obs'].cpu().numpy()), bits(h_obs))


@pytest.mark.parametrize('kernel', ['1', '0'])
def test_fp32_policy_rollout_kernel_equals_the_host_instantiation(pkg, kernel, monkeypatch):
    """copter_policy_rollout_f32: the env half of the fused policy + step kernels ('1': the tcgen05 / TMEM
    kernel, '0': the warp-MMA kernel), on the recorded actions."""
    monkeypatch.setenv('COPTER_B200_POLICY_ROLLOUT_TC', kernel)
    N, T = 777, 48
    env = pkg.CopterVecEnv('Lander3D', N, dtype=torch.float32, seed=3)
    host = HostEnvBatch('Lander3D', N, dtype=np.float32, seed=3)
    env.reset(); host.reset()
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=5)
    pro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=0.5 * 0.0166, out_offset=0.0166, store_actions=True)
    for rep in range(4):
        rewards, dones, _ = pro.run()
        acts, dones = pro.actions.cpu().numpy(), dones.cpu().numpy()
        for t in range(T):
            _, _, h_done, _ = host.step(acts[t], 1)
            assert np.array_equal(dones[t], h_done), (rep, t)
        assert np.array_equal(bits(env.state.cpu().numpy()), bits(host.x))
        assert np.array_equal(env.steps.cpu().numpy(), host.steps)


def test_fp32_dynamics_facade_equals_the_host_instantiation(pkg):
    rng = np.random.default_rng(2)
    N = 1000
    s0 = (rng.normal(0, 1, (N, 12)) * np.array([3, 1, 3, 1, 2, 1, .3, .2, .3, .2, 40., .2])).astype(np.float32)   # large yaw: the fp64 reduction
    s0[: N // 4, 4] = np.abs(s0[: N // 4, 4]) * 0.01
    d = pkg.Dynamics(num=N, dtype=torch.float32)
    h = HostDynamicsBatch(N, dtype=np.float32)
    d.setState(s0); h.set_state(s0)
    for t in range(80):
        m = (HOVER * (1 + 0.5 * rng.uniform(-1, 1, (N, 4)))).astype(np.float32)
        if t % 7 == 0:
            f = rng.uniform(-5, 5, (N, 6)).astype(np.float32)
            d.perturb(f); h.set_perturb(f)
            d._perturb.copy_(torch.as_tensor(h.perturb))           # same rounding of force / M on both sides
        d.setMotors(m); h.set_motors(m)
        assert np.array_equal(d.getStatus().cpu().numpy(), h.status)
        assert np.array_equal(d._ticks.cpu().numpy(), h.ticks)
        assert np.array_equal(bits(d.state.cpu().numpy()), bits(h.x)), t
    assert len(set(h.status.tolist())) >= 3

