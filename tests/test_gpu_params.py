"""
GPU: every kernel that takes CopterParams, at the parameter sets of oracle/param_sets.py -- asymmetric inertia,
the gyroscopic and lift models, another frame rate, angle limits on both sides of the fp32 polynomial range,
non-default landing limits, penalties and reset forces.

Every other GPU comparison runs at the default DJI Phantom parameters, where Ix == Iy, Omega == 0, dt = 1/100 and
calm_angle == max_angle: a kernel that mixed up roll and pitch, dropped the gyroscopic products or tested the
calm streak against the wrong angle would compute the same bits there.  Here, at each set:
  * the step kernel in fp32, K in {1, 4, 16}: state, observation, flags, counters, causes and terminal
    observation bit for bit the fp32 host instantiation of copter_core.h, reward within 5e-5 max / 1e-7 mean
    (the device's MUFU square roots and quotient), the statistics' counts exactly the host ledger's.  At K = 16
    this runs the calm streak with calm_angle clamped to the polynomial range (asymmetric, 60 degrees) and
    equal to max_angle below it (gyro, 30 degrees);
  * the step kernel in fp64, K in {1, 16}, against the numpy oracle directly: <= 1e-9, flags exact;
  * the rollout kernel with drawn (randn, uniform) and PID-computed commands, with its ending records: fp32 bit
    for bit, fp64 <= 1e-9 against the host instantiation;
  * both fused policy rollouts (tcgen05 and warp-MMA), with and without exploration noise, bit for bit;
  * the Dynamics facade with a six-component perturbation, take-offs from the ground included: fp32 bit for
    bit, fp64 <= 1e-9 against the oracle;
  * the reset-force kernel at each set's initial_random_force, bit for bit the oracle's Philox.
tests/test_params_cpu.py pins the host instantiation itself to the oracle at the same sets.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.copter_oracle import ALL_VARIANTS, DynamicsBatch, EnvBatch, reset_force             # noqa: E402
from oracle.host_restatement import HostDynamicsBatch, HostEnvBatch                              # noqa: E402
from oracle.param_sets import CASES, SETS, hover_command, params_dict, premises                 # noqa: E402
from test_gpu_host_exact import ReturnBook, assert_counts, assert_same, bits                    # noqa: E402
from test_params_cpu import streams                                                              # noqa: E402

SEED, OFF = 17, (3 << 32) + 5


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


def case_ids(cases):
    return ['%s-%s' % c for c in cases]


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1))) if a.size else 0.0


@pytest.mark.parametrize('k', [1, 4, 16])
@pytest.mark.parametrize('name,variant', CASES, ids=case_ids(CASES))
def test_fp32_step_kernel_equals_the_host_instantiation(pkg, name, variant, k):
    """Auto-reset at K = 1 and 16, none at K = 4 (where the commands stay within 60 % of hover: without an
    ending's reset an asymmetric vehicle tumbling under saturating commands runs its rates to overflow)."""
    p = SETS[name]
    premises(name)
    auto = k != 4
    N, T = 2048 + 77, max(240 // k, 40)
    rng = np.random.default_rng(100 * k + sum(map(ord, name + variant)))
    act = streams(rng, N, T, ALL_VARIANTS[variant][2], hover_command(p), variant == 'Takeoff', auto)
    env = pkg.CopterVecEnv(variant, N, dtype=torch.float32, seed=SEED, env_offset=OFF, k_substeps=k, auto_reset=auto,
                           track_stats=True, report_cause=True, keep_final_obs=True, **params_dict(p))
    host = HostEnvBatch(variant, N, p, dtype=np.float32, seed=SEED, env_offset=OFF, auto_reset=auto)
    obs, _ = env.reset()
    assert np.array_equal(bits(obs.cpu().numpy()), bits(host.reset()))
    for t in range(T):
        obs, r, term, trunc, info = env.step(torch.as_tensor(act[t]))
        h_obs, h_r, h_done, h_info = host.step(act[t], k)
        assert_same(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t)
        assert np.array_equal(trunc.cpu().numpy(), (h_info['cause'] & 32) != 0), t
        assert_counts(env, host, t)
    s = env.stats()
    assert s['episodes'] >= N and s['timeout'] > 0 and s['env_steps'] <= N * k * T
    if variant != 'Takeoff':
        assert sum(s[c] > 0 for c in ('landed', 'oob', 'angle', 'crashed', 'timeout')) >= 2, s


@pytest.mark.parametrize('k', [1, 16])
@pytest.mark.parametrize('name,variant', CASES, ids=case_ids(CASES))
def test_fp64_step_kernel_matches_the_oracle(pkg, name, variant, k):
    """The fp64 step kernel against the numpy oracle itself (no host instantiation in between): state, reward
    and observation <= 1e-9, done flags, status, step counters, episode indices, causes exact."""
    p = SETS[name]
    auto = k == 1
    N, T = 1024 + 45, max(160 // k, 24)
    rng = np.random.default_rng(7 * k + sum(map(ord, name + variant)))
    act = streams(rng, N, T, ALL_VARIANTS[variant][2], hover_command(p), variant == 'Takeoff', auto).astype(np.float64)
    env = pkg.CopterVecEnv(variant, N, dtype=torch.float64, seed=SEED, env_offset=OFF, k_substeps=k, auto_reset=auto,
                           report_cause=True, **params_dict(p))
    orc = EnvBatch(variant, N, p, seed=SEED, env_offset=OFF, auto_reset=auto)
    env.reset(); orc.reset()
    episodes = 0
    for t in range(T):
        obs, r, term, _, info = env.step(torch.as_tensor(act[t]))
        o_obs, o_r, o_done, o_info = orc.step(act[t], k)
        assert np.array_equal(term.cpu().numpy(), o_done), t
        assert np.array_equal(env.status.cpu().numpy(), orc.dyn.status), t
        assert np.array_equal(env.steps.cpu().numpy(), orc.steps), t
        assert np.array_equal(env.episodes.cpu().numpy(), orc.episode), t
        assert np.array_equal(info['cause'].cpu().numpy(), o_info['cause']), t
        assert relerr(env.state.cpu().numpy(), orc.dyn.x) <= 1e-9, t
        assert relerr(r.cpu().numpy(), o_r) <= 1e-9, t
        assert relerr(obs.cpu().numpy(), o_obs) <= 1e-6, t          # (fp32 observations of the same states)
        episodes += int(o_done.sum())
    assert episodes >= N // 4


def _rollout_sources(name):
    """(variant, source, scale, offset, pid gains) at the set's hover command `hv`: drawn commands around hover,
    the lander PID around 0.9 hover, the hover PID as tests/test_gpu_host_exact.py runs it (3-D: twice hover and
    no offset).  Takeoff (no angle limit) keeps its commands within 20 % of hover."""
    hv = hover_command(SETS[name])
    if name == 'takeoff':
        return [('Takeoff', 'uniform', 0.15 * hv, 1.05 * hv, None), ('Takeoff', 'randn', 0.04 * hv, 1.02 * hv, None)]
    return [('Lander3D', 'randn', 0.5 * hv, hv, None), ('Lander2D', 'uniform', 0.6 * hv, hv, None),
            ('Lander3D', 'pid', 0.12 * hv, 0.9 * hv, {'descent_kd': 3.0}), ('Lander1D', 'pid', 0.06 * hv, 0.96 * hv, {'descent_kd': 3.0}),
            ('Hover3D', 'pid_hover', 2 * hv, None, None), ('Hover2D', 'pid_hover', hv, hv, None), ('Hover1D', 'pid_hover', hv, hv, None)]


ROLLOUT_CASES = [pytest.param(name, *src, dt, id='%s-%s-%s-%s' % (name, src[0], src[1], dt))
                 for name in SETS for src in _rollout_sources(name) for dt in ('f32', 'f64')]


@pytest.mark.parametrize('name,variant,source,scale,offset,gains,dt', ROLLOUT_CASES)
def test_rollout_kernel_equals_the_host_instantiation(pkg, name, variant, source, scale, offset, gains, dt):
    """copter_rollout_f32 / _f64 on commands it draws or computes itself, replayed on the host: per-step rewards,
    done flags, causes and terminal observations, then state and counters after each launch -- fp32 bit for bit,
    fp64 <= 1e-9 -- and the statistics' counts exactly."""
    p = SETS[name]
    f32 = dt == 'f32'
    dtype = np.float32 if f32 else np.float64
    N, T = 1000 + 9, 40
    env = pkg.CopterVecEnv(variant, N, dtype=torch.float32 if f32 else torch.float64, seed=SEED, env_offset=OFF,
                           track_returns=True, **params_dict(p))
    host = HostEnvBatch(variant, N, p, dtype=dtype, seed=SEED, env_offset=OFF, track_returns=True)
    env.reset(); host.reset()
    tol = 5e-5 if f32 else 1e-9
    book = ReturnBook(N, dtype, tol)
    for chunk in range(3):
        out = env.rollout(T, source=source, scale=scale, offset=offset, pid_gains=gains, record_rewards=True,
                          record_dones=True, record_actions=True, record_causes=True, record_final_obs=True)
        acts, dones, rews = out['actions'].cpu().numpy(), out['dones'].cpu().numpy(), out['rewards'].cpu().numpy()
        causes, fin = out['causes'].cpu().numpy(), out['final_obs'].cpu().numpy()
        for t in range(T):
            _, h_r, h_done, h_info = host.step(acts[t], 1)
            assert np.array_equal(dones[t], h_done), (chunk, t)
            assert np.array_equal(causes[t], h_info['cause']), (chunk, t)
            if f32:
                assert np.array_equal(bits(fin[t][h_done]), bits(h_info['final_obs'][h_done])), (chunk, t)
            else:
                assert relerr(fin[t][h_done], h_info['final_obs'][h_done]) <= 1e-6, (chunk, t)
            assert not fin[t][~h_done].any(), (chunk, t)
            assert relerr(rews[t], h_r) <= tol, (chunk, t)
            book.add(rews[t], h_r, h_done.copy())
        x = env.state.cpu().numpy()
        if f32:
            assert np.array_equal(bits(x), bits(host.x)), chunk
        else:
            assert relerr(x, host.x) <= 1e-9, chunk
        assert np.array_equal(env.steps.cpu().numpy(), host.steps) and np.array_equal(env.status.cpu().numpy(), host.status)
        assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64))
        book.check(env, host, chunk)
    s = env.stats()
    assert s['episodes'] > 0 and s['env_steps'] == 3 * T * N


POLICY_CASES = [pytest.param(name, v, kern, std, id='%s-%s-%s-%s' % (name, v, 'tc' if kern == '1' else 'mma', 'std' if std else 'nostd'))
                for name in SETS for v in (('Takeoff',) if name == 'takeoff' else ('Lander3D', 'Hover2D'))
                for kern in ('1', '0') for std in (False, True)]


@pytest.mark.parametrize('name,variant,kernel,std', POLICY_CASES)
def test_fused_policy_rollouts_equal_the_host_instantiation(pkg, name, variant, kernel, std, monkeypatch):
    """copter_policy_rollout_f32 ('1': tcgen05 / TMEM, '0': warp-MMA) on the recorded actions, N not a multiple of
    128: state, counters and flags bit for bit, ep_return bit for bit the running sum of the recorded rewards,
    the statistics' counts exactly the host ledger's."""
    monkeypatch.setenv('COPTER_B200_POLICY_ROLLOUT_TC', kernel)
    p = SETS[name]
    hv = hover_command(p)
    N, T, reps = 1500 + 13, 48, 3
    env = pkg.CopterVecEnv(variant, N, dtype=torch.float32, seed=SEED, env_offset=OFF, track_returns=True, **params_dict(p))
    host = HostEnvBatch(variant, N, p, dtype=np.float32, seed=SEED, env_offset=OFF, track_returns=True)
    env.reset(); host.reset()
    pol = pkg.mlp_policy(env.obs_size, env.action_size, dtype=torch.float32, seed=5)
    spread = 0.15 if variant == 'Takeoff' else 0.5          # (tanh head: commands within offset +- scale)
    pro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=spread * hv, out_offset=hv, store_actions=True,
                                 action_std=(0.01 if variant == 'Takeoff' else 0.25) * hv if std else None)
    book = ReturnBook(N, np.float32, 5e-5)
    for rep in range(reps):
        rewards, dones, _ = pro.run()
        acts, dones, rews = pro.actions.cpu().numpy(), dones.cpu().numpy(), rewards.cpu().numpy()
        for t in range(T):
            _, h_r, h_done, _ = host.step(acts[t], 1)
            assert np.array_equal(dones[t], h_done), (rep, t)
            book.add(rews[t], h_r, h_done.copy())
        assert np.array_equal(bits(env.state.cpu().numpy()), bits(host.x)), rep
        assert np.array_equal(env.steps.cpu().numpy(), host.steps) and np.array_equal(env.status.cpu().numpy(), host.status)
        assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64))
        book.check(env, host, rep)
    s = env.stats()
    assert s['episodes'] > 0 and s['env_steps'] == reps * T * N


@pytest.mark.parametrize('dtype', ['f32', 'f64'])
@pytest.mark.parametrize('name', list(SETS))
def test_dynamics_facade_at_the_parameter_set(pkg, name, dtype):
    """copter_dynamics_*: N vehicles driven directly, a quarter of them starting on the ground, roll and pitch past
    pi/4 and large yaw angles (the range-reduced sin / cos), a six-component perturbation every seventh call whose
    angular part acts on the set's inertia.  fp32 bit for bit the host instantiation, fp64 <= 1e-9 the oracle;
    statuses and ticks exact; vehicles take off from the ground under the set's G."""
    p = SETS[name]
    f32 = dtype == 'f32'
    hv = hover_command(p)
    rng = np.random.default_rng(sum(map(ord, name)))
    N = 1000 + 11
    s0 = rng.normal(0, 1, (N, 12)) * np.array([3, 1, 3, 1, 2, 1, .5, .2, .5, .2, 40., .2])
    s0[: N // 4, 4] = np.abs(s0[: N // 4, 4]) * 0.01                 # on the ground, level and at rest vertically: LANDED
    s0[: N // 4, 5:10] = 0
    world = {k: v for k, v in params_dict(p).items() if k != 'fps'}
    d = pkg.Dynamics(params=world, framesPerSecond=p.fps, num=N, dtype=torch.float32 if f32 else torch.float64)
    if f32:
        s0 = s0.astype(np.float32)
        ref = HostDynamicsBatch(N, p, dtype=np.float32)
    else:
        ref = DynamicsBatch(N, p, np.float64)
    d.setState(s0); ref.set_state(s0)
    took_off = np.zeros(N, bool)
    for t in range(80):
        m = (hv * (1 + 0.5 * rng.uniform(-1, 1, (N, 4)))).astype(np.float32)
        m = m if f32 else m.astype(np.float64)
        if t % 7 == 0:
            f = rng.uniform(-5, 5, (N, 6)).astype(np.float32 if f32 else np.float64)
            d.perturb(f); ref.set_perturb(f)
            if f32:
                d._perturb.copy_(torch.as_tensor(ref.perturb))       # the same rounding of force / M on both sides
        before = ref.status.copy()
        d.setMotors(m); ref.set_motors(m)
        took_off |= (before == 1) & (ref.status == 3)
        assert np.array_equal(d.getStatus().cpu().numpy(), ref.status), t
        assert np.array_equal(d._ticks.cpu().numpy(), ref.ticks), t
        x = d.state.cpu().numpy()
        if f32:
            assert np.array_equal(bits(x), bits(ref.x)), (t, np.argwhere(bits(x) != bits(ref.x))[:5])
        else:
            assert relerr(x, ref.x) <= 1e-9, t
    assert took_off[: N // 4].sum() >= N // 16 and len(set(ref.status.tolist())) >= 3
    assert (np.maximum(np.abs(ref.x[:, 6]), np.abs(ref.x[:, 8])) > np.pi / 4).any()


@pytest.mark.parametrize('name', [n for n in SETS if SETS[n].initial_random_force != 0])
def test_reset_force_kernel_at_the_parameter_set(pkg, name):
    """copter_reset_force_* at the set's initial_random_force, bit for bit the oracle's Philox draw."""
    p = SETS[name]
    lib = pkg.load_library()
    cp = pkg.default_params(**params_dict(p))
    n, seed = 5000 + 3, 0x1234ABCD5678
    ep = torch.randint(0, 2 ** 19, (n,), dtype=torch.int32, device='cuda')
    for fn, td, nd in ((lib.copter_reset_force_f64, torch.float64, np.float64),
                       (lib.copter_reset_force_f32, torch.float32, np.float32)):
        out = torch.zeros((n, 3), dtype=td, device='cuda')
        assert fn(C.byref(cp), out.data_ptr(), ep.data_ptr(), n, OFF, seed, None) == 0
        torch.cuda.synchronize()
        ref = reset_force(seed, np.arange(n, dtype=np.uint64) + np.uint64(OFF), ep.cpu().numpy(), p.initial_random_force, nd)
        got = out.cpu().numpy()
        assert np.array_equal(got, ref)
        assert np.abs(got).max() <= p.initial_random_force and np.abs(got).max() > 0.99 * p.initial_random_force
