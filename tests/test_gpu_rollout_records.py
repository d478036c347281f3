"""GPU tests of the rollouts' ending records (the COPTER_CAUSE_* bits of every step and the terminal
observations) and of the on-device GAE that consumes them: the records equal what the step kernel reports
step by step, recording changes nothing else, the step limit is reported as a truncation, and
copter_gae_f32 equals a float64 restatement of its definition."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.copter_oracle import EnvBatch, OracleParams      # noqa: E402

TIMEOUT, LANDED, OOB, ANGLE, CRASHED = 32, 1, 4, 8, 16
HOVER_CMD = 0.016560178212092172


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


@pytest.fixture
def policy_kernel_choice():
    """COPTER_B200_POLICY_TC selects the standalone policy kernel per call -- '1' tcgen05 / TMEM (its default),
    '0' warp-level mma.sync -- and COPTER_B200_POLICY_ROLLOUT_TC the fused policy + step rollout kernel (the same
    values and default).  choose(v) sets both to the same kind."""
    import os
    names = ('COPTER_B200_POLICY_TC', 'COPTER_B200_POLICY_ROLLOUT_TC')
    old = {k: os.environ.get(k) for k in names}

    def choose(v):
        for k in names:
            os.environ[k] = v
    yield choose
    for k in names:
        if old[k] is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = old[k]


def bits(x):
    return x.contiguous().view(torch.int32 if x.dtype == torch.float32 else torch.int64)


# A short step limit, a low start and tight bounds, and a reset force of up to 600 N in every direction
# (injected per env, so it pushes every episode of the env the same way): within 200 steps the envs of
# every source time out, fly out of bounds, crash or tip over, and the landing heuristics also land.
ENDING_PARAMS = dict(max_steps=60, initial_altitude=1.0, bounds=2.0)
SOURCES = [('Lander3D', 'const', None, None, None), ('Lander3D', 'randn', None, None, None),
           ('Lander3D', 'uniform', 0.01, 0.0166, None), ('Lander3D', 'pid', 2.0e-3, 0.0149, {'descent_kd': 3.0}),
           ('Lander2D', 'pid', 1e-3, 0.0159, {'descent_kd': 3.0}), ('Lander1D', 'pid', 1e-3, 0.0159, {'descent_kd': 3.0}),
           ('Hover3D', 'pid_hover', 2 * HOVER_CMD, None, None), ('Hover2D', 'pid_hover', HOVER_CMD, HOVER_CMD, None),
           ('Hover1D', 'pid_hover', HOVER_CMD, HOVER_CMD, None)]


def reset_forces(n):
    return np.random.default_rng(0).uniform(-1, 1, (n, 3)) * 600.0


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
@pytest.mark.parametrize('variant,source,scale,offset,gains', SOURCES)
def test_rollout_records_equal_the_step_loop(pkg, variant, source, scale, offset, gains, dtype):
    """copter_rollout_*: cause_tn row t holds exactly the cause bits copter_step_* (k = 1) reports for that step, and
    final_obs_tn the terminal observation it writes -- checked against a twin env replaying the recorded commands
    with step() (report_cause, keep_final_obs), bit for bit; done_tn == (cause_tn != 0); rows of steps where
    nothing ended stay zero.  For fp64 with the constant command, the causes also equal the oracle's."""
    n, T, seed = 4099, 200, 21
    kw = dict(dtype=dtype, seed=seed, **ENDING_PARAMS)
    force = reset_forces(n)
    env = pkg.CopterVecEnv(variant, n, **kw)
    env.reset(force=force)
    twin = pkg.CopterVecEnv(variant, n, report_cause=True, keep_final_obs=True, **kw)
    twin.load_state_dict(env.state_dict())
    out = env.rollout(T, source=source, scale=scale, offset=offset, pid_gains=gains, record_dones=True,
                      record_actions=True, record_causes=True, record_final_obs=True)
    causes, fin, dones, acts = out['causes'], out['final_obs'], out['dones'], out['actions']
    assert causes.shape == (T, n) and causes.dtype == torch.uint8
    assert fin.shape == (T, n, env.obs_size) and fin.dtype == torch.float32
    assert torch.equal(dones, causes != 0)
    orc, sync = None, np.ones(n, bool)
    if dtype == torch.float64 and source == 'const':
        orc = EnvBatch(variant, n, params=OracleParams(**ENDING_PARAMS), seed=seed)
        orc.reset(force=force)
    for t in range(T):
        _, _, term, trunc, info = twin.step(acts[t])
        assert torch.equal(info['cause'], causes[t]), t
        ended = causes[t] != 0
        assert torch.equal(term, ended)
        assert torch.equal(bits(info['final_obs'][ended]), bits(fin[t][ended])), t
        assert not fin[t][~ended].any()
        if orc is not None:
            _, _, _, o_info = orc.step(acts[t].cpu().numpy(), force=force)
            sync &= o_info['cause'].astype(np.uint8) == causes[t].cpu().numpy()
    assert torch.equal(env.state, twin.state) and torch.equal(env.meta, twin.meta)
    # (the fp64 path follows the oracle to ~1e-12; an ending test decided on the last bits may differ)
    assert sync.sum() >= n - n // 1000, n - sync.sum()
    seen = int(np.bitwise_or.reduce(causes.cpu().numpy().reshape(-1)))
    assert seen & TIMEOUT and seen & (OOB | ANGLE | CRASHED), seen
    if source == 'pid':
        assert seen & LANDED and seen & CRASHED and seen & OOB, seen


@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('std', [False, True])
@pytest.mark.parametrize('variant,n', [('Lander3D', 4099), ('Lander2D', 1000), ('Hover3D', 257), ('Lander1D', 31),
                                       ('Hover2D', 517), ('Hover1D', 33), ('Lander3D', 128 * 148 * 8 + 77)])
def test_fused_policy_rollout_records_equal_policy_rollout(pkg, variant, n, std, kernel, policy_kernel_choice):
    """copter_policy_rollout_f32 records (tcgen05 kernel '1', warp-MMA kernel '0') against PolicyRollout, the step
    loop under the standalone policy kernel of the same kind: causes, terminal observations, terminated and truncated
    are identical.  With exploration noise on, the reference loop replays the fused rollout's sampled commands.  The
    last size holds more tiles than the tcgen05 kernel has resident CTAs."""
    policy_kernel_choice(kernel)
    T = 150 if n < 10000 else 40
    envs = [pkg.CopterVecEnv(variant, n, seed=11, max_steps=60) for _ in range(2)]
    pol = pkg.mlp_policy(envs[0].obs_size, envs[0].action_size, dtype=torch.float32, seed=2)
    for p in pol.net.parameters():
        p.data.mul_(2.0)
    scale, offset = 0.03, 0.0166
    for e in envs:
        e.reset()
    fused = pkg.FusedPolicyRollout(envs[0], pol.net, T, out_scale=scale, out_offset=offset, store_actions=True,
                                   action_std=0.004 if std else None, store_causes=True, store_final_obs=True)
    fused.run()
    if std:
        step = [0]

        def policy(planes):
            a = fused.actions[step[0]]
            step[0] += 1
            return a
        ref = pkg.PolicyRollout(envs[1], policy, T, planar=True, use_cuda_graph=False, store_causes=True, store_final_obs=True)
    else:
        ref = pkg.PolicyRollout(envs[1], pkg.FusedMLPPolicy(envs[1], pol.net, out_scale=scale, out_offset=offset), T,
                                planar=True, store_causes=True, store_final_obs=True)
    ref.run()
    assert torch.equal(fused.causes, ref.causes)
    ended = fused.causes != 0
    assert torch.equal(bits(fused.final_obs[ended]), bits(ref.final_obs[ended]))
    assert not fused.final_obs[~ended].any()
    assert torch.equal(fused.terminated, ref.terminated) and torch.equal(fused.truncated, ref.truncated)
    assert torch.equal(fused.dones.bool(), ended) and not (fused.terminated & fused.truncated).any()
    assert torch.equal(envs[0].state, envs[1].state) and torch.equal(envs[0].meta, envs[1].meta)
    if T >= 60:
        assert fused.truncated.any()


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
@pytest.mark.parametrize('record_rewards', [False, True])
def test_rollout_records_are_a_pure_output(pkg, dtype, record_rewards):
    """env.rollout with and without the records, from one snapshot: rewards, dones, actions, the observation,
    the final state, the counters and the statistics are bit-identical (both the per-step and the telescoped
    reward path; the statistics' return sum up to the order of its atomics, see assert_same_stats)."""
    n, T = 3001, 120
    kw = dict(dtype=dtype, seed=4, track_returns=True, **ENDING_PARAMS)
    a, b = pkg.CopterVecEnv('Lander3D', n, **kw), pkg.CopterVecEnv('Lander3D', n, **kw)
    a.reset(force=reset_forces(n))
    b.load_state_dict(a.state_dict())
    common = dict(source='randn', record_rewards=record_rewards, record_dones=True, record_actions=True)
    oa = a.rollout(T, record_causes=True, record_final_obs=True, **common)
    ob = b.rollout(T, **common)
    for k in ('obs', 'reward_sum', 'done_any', 'dones', 'actions') + (('rewards',) if record_rewards else ()):
        assert torch.equal(oa[k], ob[k]), k
    assert torch.equal(bits(oa['reward_sum']), bits(ob['reward_sum']))
    assert torch.equal(a.state_planes, b.state_planes) and torch.equal(a.meta, b.meta)
    assert torch.equal(a.ep_return, b.ep_return)
    assert_same_stats(a, b)
    assert oa['causes'].any()


@pytest.mark.parametrize('kernel', ['1', '0'])
def test_fused_policy_rollout_records_are_a_pure_output(pkg, kernel, policy_kernel_choice):
    policy_kernel_choice(kernel)
    n, T = 4099, 100
    envs = [pkg.CopterVecEnv('Lander3D', n, seed=8, track_returns=True, max_steps=60) for _ in range(2)]
    for e in envs:
        e.reset()
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=3)
    kw = dict(out_scale=0.03, out_offset=0.0166, store_obs=True, store_actions=True, action_std=0.002)
    on = pkg.FusedPolicyRollout(envs[0], pol.net, T, store_causes=True, store_final_obs=True, **kw)
    off = pkg.FusedPolicyRollout(envs[1], pol.net, T, **kw)
    for _ in range(2):
        r1, d1, o1 = on.run()
        r2, d2, o2 = off.run()
        assert torch.equal(bits(r1), bits(r2)) and torch.equal(d1, d2) and torch.equal(o1, o2)
        assert torch.equal(on.actions, off.actions) and torch.equal(on.obs, off.obs)
    assert torch.equal(envs[0].state_planes, envs[1].state_planes) and torch.equal(envs[0].meta, envs[1].meta)
    assert torch.equal(envs[0].ep_return, envs[1].ep_return)
    assert_same_stats(envs[0], envs[1])
    assert on.causes.any()


def test_hover_step_limit_is_a_truncation(pkg):
    """The hover workload ends by the step limit: every recorded ending is a truncation, their count is the
    statistics' timeout count and equals n (every first episode runs to the 1000-step limit), and the terminal
    observations hold the vehicle at the 5 m set-point (NED z within 0.1 m of -5)."""
    n = 512
    env = pkg.CopterVecEnv('Hover3D', n, seed=5, track_stats=True)
    env.reset()
    causes, fin = [], []
    for chunk in range(1100 // 50):
        out = env.rollout(50, source='pid_hover', scale=2 * HOVER_CMD, record_causes=True, record_final_obs=True)
        causes.append(out['causes'].clone()); fin.append(out['final_obs'].clone())
    causes, fin = torch.cat(causes), torch.cat(fin)
    ended = causes != 0
    assert ((causes[ended] & TIMEOUT) != 0).all()
    truncated = (causes & TIMEOUT) != 0
    s = env.stats()
    assert int(truncated.sum()) == s['timeout'] == n
    assert torch.equal(truncated.sum(0), torch.ones(n, dtype=torch.int64, device='cuda'))
    z = fin[ended][:, 4]
    assert (z + 5.0).abs().max().item() < 0.1, (z.min().item(), z.max().item())


def assert_same_stats(a, b):
    """Episode statistics of two envs that ran the same episodes: the counts bit for bit; the return sum, which warps
    of different CTAs add to the same slot with fp64 atomics in whatever order they arrive, to its last bits."""
    from gym_copter_b200._lib import STAT_NAMES
    sa, sb = a._stats.sum(0), b._stats.sum(0)
    ret = STAT_NAMES.index('return_sum')
    keep = [j for j in range(sa.numel()) if j != ret]
    assert torch.equal(sa[keep], sb[keep])
    assert abs(sa[ret].item() - sb[ret].item()) <= 1e-12 * max(1.0, abs(sb[ret].item()))


# ---- GAE ---------------------------------------------------------------------------------------------------------

def gae_reference(r, v, last, c, fv, gamma, lam):
    """The definition of copter_gae_f32 in float64, with gamma and lam rounded to fp32 as the kernel receives them."""
    g, l = float(np.float32(gamma)), float(np.float32(lam))
    r, v, last = (np.asarray(x, np.float64) for x in (r, v, last))
    fv = None if fv is None else np.asarray(fv, np.float64)
    T = r.shape[0]
    adv = np.empty_like(r)
    nxt, a = last, np.zeros_like(last)
    for t in range(T - 1, -1, -1):
        run = c[t] == 0
        trunc = (c[t] & TIMEOUT) != 0
        boot = np.where(run, nxt, np.where(trunc, fv[t], 0.0) if fv is not None else 0.0)
        delta = r[t] + g * boot - v[t]
        a = delta + g * l * np.where(run, a, 0.0)
        adv[t] = a
        nxt = v[t]
    return adv, adv + v


def random_causes(rng, T, n, p_end=0.2):
    """Running (0), terminal (LANDED | BONUS, OOB, ANGLE, CRASHED) and step-limit (TIMEOUT, alone or with a
    terminal bit) endings."""
    kinds = np.array([LANDED | 2, OOB, ANGLE, CRASHED, TIMEOUT, TIMEOUT | OOB], np.uint8)
    c = kinds[rng.integers(0, len(kinds), (T, n))]
    return np.where(rng.random((T, n)) < p_end, c, 0).astype(np.uint8)


def gae_inputs(rng, T, n):
    f = lambda *s: torch.as_tensor(rng.standard_normal(s).astype(np.float32), device='cuda')    # noqa: E731
    return f(T, n), f(T, n), f(n), torch.as_tensor(random_causes(rng, T, n), device='cuda'), f(T, n)


@pytest.mark.parametrize('T', [1, 7, 8, 9, 17, 32])  # kGaeRows = 8: 8 is one block; 9 and 17 end on a one-row block
@pytest.mark.parametrize('n', [1, 31, 4099, 2 ** 20 + 3])
def test_gae_equals_float64_definition(pkg, T, n):
    """Tolerance: fp32 rounding of a T-term recursion.  Every step rounds a handful of times (gamma * boot, the two
    sums of delta, gamma * lam * A, the sum of A) on values of magnitude up to ~10 here (standard normal inputs, short
    episodes), so the error stays below T * 16 * 2^-23 relative to max(|ref|, 1)."""
    rng = np.random.default_rng(T * 1000 + n)
    r, v, last, c, fv = gae_inputs(rng, T, n)
    cn = c.cpu().numpy()
    if n >= 4099:
        assert (cn == 0).any() and ((cn & TIMEOUT) != 0).any() and ((cn != 0) & ((cn & TIMEOUT) == 0)).any()
    tol = T * 16 * 2.0 ** -23
    for gamma, lam in ((0.99, 0.95), (0.9, 0.0), (0.97, 1.0)):
        for final in (None, fv):
            adv, ret = pkg.gae(r, v, last, c, final, gamma=gamma, lam=lam)
            assert adv.shape == (T, n) and adv.dtype == torch.float32 and ret.shape == (T, n)
            ra, rr = gae_reference(r.cpu().numpy(), v.cpu().numpy(), last.cpu().numpy(), cn,
                                   None if final is None else final.cpu().numpy(), gamma, lam)
            for got, ref in ((adv, ra), (ret, rr)):
                err = np.abs(got.cpu().numpy() - ref) / np.maximum(np.abs(ref), 1.0)
                assert err.max() <= tol, (gamma, lam, final is None, err.max(), tol)


def test_gae_end_to_end_on_a_fused_rollout(pkg):
    """FusedPolicyRollout -> a torch value net on obs, final_obs and the observation after the last step -> gae,
    against the float64 definition on the same fp32 values.  The short step limit puts truncations and
    terminations in the horizon."""
    n, T = 4099, 48
    env = pkg.CopterVecEnv('Lander3D', n, seed=13, **dict(ENDING_PARAMS, max_steps=25))
    env.reset(force=reset_forces(n))
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=4)
    ro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=0.03, out_offset=0.0166, store_obs=True, action_std=0.003,
                                store_causes=True, store_final_obs=True)
    rewards, _, last_obs = ro.run()
    torch.manual_seed(0)
    critic = torch.nn.Sequential(torch.nn.Linear(10, 32), torch.nn.Tanh(), torch.nn.Linear(32, 1)).cuda()
    with torch.no_grad():
        values = critic(ro.obs).squeeze(-1).contiguous()
        final_values = critic(ro.final_obs).squeeze(-1).contiguous()
        last_values = critic(last_obs).squeeze(-1).contiguous()
    adv, ret = pkg.gae(rewards, values, last_values, ro.causes, final_values, gamma=0.99, lam=0.95)
    ra, rr = gae_reference(rewards.cpu().numpy(), values.cpu().numpy(), last_values.cpu().numpy(), ro.causes.cpu().numpy(),
                           final_values.cpu().numpy(), 0.99, 0.95)
    tol = T * 16 * 2.0 ** -23
    for got, ref in ((adv, ra), (ret, rr)):
        assert (np.abs(got.cpu().numpy() - ref) / np.maximum(np.abs(ref), 1.0)).max() <= tol
    assert ro.truncated.any() and ro.terminated.any()
    # bootstrapping the truncations moves exactly the advantages of the truncated episodes' steps
    adv0, _ = pkg.gae(rewards, values, last_values, ro.causes, None, gamma=0.99, lam=0.95)
    assert not torch.equal(adv0[ro.truncated], adv[ro.truncated])
    assert torch.equal(adv0[ro.terminated], adv[ro.terminated])


def test_gae_does_not_leak_across_episode_ends(pkg):
    """An ending at step t cuts the recursion: rewards and values after it, and the last value, do not move the
    advantages of steps <= t; a changed final value moves only the steps of the episode it bootstraps."""
    T, n, t_end, t_first = 16, 1024, 9, 3
    rng = np.random.default_rng(5)
    r, v, last, _, fv = gae_inputs(rng, T, n)
    c = np.zeros((T, n), np.uint8)
    c[t_first] = OOB                                     # every env: an earlier episode ends at t_first
    c[t_end, 0::2] = TIMEOUT                             # even envs truncated at t_end, odd ones terminated
    c[t_end, 1::2] = CRASHED
    c = torch.as_tensor(c, device='cuda')
    base, _ = pkg.gae(r, v, last, c, fv)
    r2, v2 = r.clone(), v.clone()
    r2[t_end + 1:] += 1.5
    v2[t_end + 1:] -= 0.75
    moved, _ = pkg.gae(r2, v2, last + 3.0, c, fv)
    assert torch.equal(bits(moved[:t_end + 1]), bits(base[:t_end + 1]))
    assert not torch.equal(moved[t_end + 1:], base[t_end + 1:])
    f2 = fv + 2.0
    other, _ = pkg.gae(r, v, last, c, f2)
    changed = (bits(other) != bits(base)).cpu().numpy()
    expect = np.zeros((T, n), bool)
    expect[t_first + 1:t_end + 1, 0::2] = True           # the truncated episode of the even envs
    assert np.array_equal(changed, expect)


def test_gae_argument_errors(pkg):
    T, n = 5, 64
    r, v, last, c, fv = gae_inputs(np.random.default_rng(0), T, n)
    with pytest.raises(ValueError, match='float64'):
        pkg.gae(r.double(), v, last, c)
    with pytest.raises(ValueError):
        pkg.gae(r, v.half(), last, c)
    with pytest.raises(ValueError):
        pkg.gae(r, v, last, c.to(torch.int32))
    with pytest.raises(ValueError):
        pkg.gae(r, v[:T - 1], last, c)                  # T mismatch
    with pytest.raises(ValueError):
        pkg.gae(r, v, last, c[:T - 1])
    with pytest.raises(ValueError):
        pkg.gae(r, v, last[:n - 1], c)
    with pytest.raises(ValueError):
        pkg.gae(r, v, last, c, fv[:, :n - 1])
    with pytest.raises(pkg.CopterError):
        pkg.gae(r, v.cpu(), last, c)                    # device
    with pytest.raises(pkg.CopterError):
        pkg.gae(r, v, last, c, fv.t().contiguous().t())  # same shape, not contiguous
    wide = torch.zeros((T, 2 * n), device='cuda')
    with pytest.raises(pkg.CopterError):
        pkg.gae(r, wide[:, ::2], last, c)               # strided view
    with pytest.raises(pkg.CopterError):
        pkg.PolicyRollout(pkg.CopterVecEnv('Lander3D', 8), lambda o: o[:, :4], 2).truncated
