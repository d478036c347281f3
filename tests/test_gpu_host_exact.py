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

The bookkeeping around that arithmetic is held to the host ledger (HostEnvBatch.stats()) on every kernel
that keeps it -- step, rollout and both fused policy rollouts, auto-reset on and off, compact and wide
counters: the statistics' counts (episodes, length sum, one count per ending cause, executed env-steps)
exactly, ep_return bit for bit the running sum of the device's own rewards, return_sum the fp64 sum of
the ended returns.  The counter-field edges are in tests/test_gpu_bookkeeping.py.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.host_restatement import STAT_NAMES, HostDynamicsBatch, HostEnvBatch       # noqa: E402
from oracle.copter_oracle import ALL_VARIANTS, OracleParams                            # noqa: E402

HOVER = 0.016560178212092172
# a short step limit, a low start and tight bounds: episodes end in every way within a few dozen steps
ENDINGS = dict(max_steps=60, initial_altitude=1.0, bounds=2.0)
TAKEOFF_SHELL = dict(initial_altitude=0.0, initial_random_force=0.0, fps=50.0)      # the shell's Takeoff defaults
COUNTS = tuple(k for k in STAT_NAMES if k != 'return_sum')


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


def assert_counts(env, host, t=None):
    """The device statistics' counts (summed over the slots) == the host ledger's, exactly."""
    s, h = env.stats(), host.stats()
    assert {k: s[k] for k in COUNTS} == {k: h[k] for k in COUNTS}, (t, s, h)
    return s, h


class ReturnBook:
    """What the device's ep_return and return_sum must be, from the device's own rewards: the running sum in
    the env dtype of every launch's reward since the env's last ending (the kernels' `ret += total`), and the
    fp64 sum of the returns of the ended episodes.  `bound` sums tol * max(|r_host|, 1) over the launches of the
    ended episodes: how far return_sum may be from the host ledger's."""

    def __init__(self, n, dtype, tol):
        self.ret, self.acc = np.zeros(n, dtype), np.zeros(n)
        self.ended = self.bound = 0.0
        self.tol = tol

    def add(self, r_dev, r_host, done):
        self.ret += r_dev
        self.acc += self.tol * np.maximum(np.abs(np.asarray(r_host, np.float64)), 1.0)
        self.ended += float(self.ret[done].astype(np.float64).sum())
        self.bound += float(self.acc[done].sum())
        self.ret[done] = 0
        self.acc[done] = 0.0

    def check(self, env, host, t):
        dev = env.ep_return.cpu().numpy()
        assert np.array_equal(dev.view(np.uint8), self.ret.view(np.uint8)), (t, np.argwhere(dev != self.ret)[:5])
        s, h = assert_counts(env, host, t)
        assert abs(s['return_sum'] - self.ended) <= 1e-12 * max(abs(self.ended), 1.0), (t, s['return_sum'], self.ended)
        assert abs(s['return_sum'] - h['return_sum']) <= self.bound + 1e-9, (t, s['return_sum'], h['return_sum'], self.bound)


def _step_cases():
    """The original cases (default parameters, long episodes, no statistics: the kernels' STATS=false
    instantiation) keep their ids; the bookkeeping matrix adds every variant x K in {1, 4, 16} x auto-reset on /
    off x compact / wide counters with statistics and returns, at short episodes, one wide case with a step
    limit past the compact field, and an fp64 leg."""
    old = [pytest.param(v, k, None, id='%s-%d' % (v, k)) for v in ('Lander3D', 'Lander2D', 'Lander1D', 'Hover3D', 'Hover2D', 'Takeoff')
           for k in (1, 2, 3, 16)]
    book = [pytest.param(v, k, dict(wide=w, auto=a, dtype=np.float32, max_steps=60),
                         id='%s-%d-%s-%s' % (v, k, 'wide' if w else 'compact', 'auto' if a else 'noreset'))
            for v in ALL_VARIANTS for k in (1, 4, 16) for w in (False, True) for a in (True, False)]
    book.append(pytest.param('Hover3D', 16, dict(wide=True, auto=True, dtype=np.float32, max_steps=2100), id='Hover3D-16-wide-auto-2100'))
    book += [pytest.param(v, k, dict(wide=k == 16, auto=k == 1, dtype=np.float64, max_steps=60),
                          id='%s-%d-%s-%s-f64' % (v, k, 'wide' if k == 16 else 'compact', 'auto' if k == 1 else 'noreset'))
             for v in ALL_VARIANTS for k in (1, 16)]
    return old + book


def assert_close_f64(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t):
    """fp64: flags, counters and causes equal the fp64 host instantiation; continuous values agree to 1e-9."""
    x = env.state.cpu().numpy()
    assert np.array_equal(term.cpu().numpy(), h_done), t
    assert np.array_equal(env.status.cpu().numpy(), host.status), t
    assert np.array_equal(env.steps.cpu().numpy(), host.steps), t
    assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64)), t
    assert np.array_equal(info['cause'].cpu().numpy(), h_info['cause']), t
    assert float(np.max(np.abs(x - host.x) / np.maximum(np.abs(host.x), 1))) <= 1e-9, t
    rr = r.cpu().numpy()
    assert float(np.max(np.abs(rr - h_r) / np.maximum(np.abs(h_r), 1))) <= 1e-9, t
    assert float(np.max(np.abs(obs.cpu().numpy() - h_obs) / np.maximum(np.abs(h_obs), 1))) <= 1e-6, t


@pytest.mark.parametrize('variant,k,book', _step_cases())
def test_fp32_step_kernels_equal_the_host_instantiation(pkg, variant, k, book):
    if book is not None:
        return _step_bookkeeping(pkg, variant, k, **book)
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


def _step_bookkeeping(pkg, variant, k, wide, auto, dtype, max_steps):
    """Statistics and running returns of the step kernel on every launch: ep_return bit for bit the running
    sum of the device's own rewards, the counts exactly the host ledger's, return_sum the fp64 sum of the
    ended returns and within the per-reward tolerance of the ledger; with statistics but no returns
    (K = 4), return_sum stays exactly 0."""
    f32 = dtype == np.float32
    N, T, seed, off = 1024 + 77, max(240 // k, 60), 21 + k, 7 << 33
    rng = np.random.default_rng(31 * k + len(variant))
    A = ALL_VARIANTS[variant][2]
    act = mixed_streams(rng, N, T, A, takeoff=variant == 'Takeoff')
    kw = dict(ENDINGS, max_steps=max_steps)
    if variant == 'Takeoff':
        kw = dict(TAKEOFF_SHELL, max_steps=max_steps)
    if max_steps > 2046:            # every other env hovers until its step limit, the rest tip over
        T, kw = 2240 // k, dict(max_steps=max_steps)
        act = rng.uniform(-1, 1, (T, N, A)).astype(np.float32)
        act[:, ::2] = np.float32(HOVER)
    tdt = torch.float32 if f32 else torch.float64
    common = dict(dtype=tdt, seed=seed, env_offset=off, k_substeps=k, auto_reset=auto, wide_counters=wide, **kw)
    env = pkg.CopterVecEnv(variant, N, track_returns=True, report_cause=True, keep_final_obs=True, **common)
    lean = pkg.CopterVecEnv(variant, N, track_stats=True, **common) if k == 4 else None
    host = HostEnvBatch(variant, N, OracleParams(**kw), dtype=dtype, seed=seed, env_offset=off, auto_reset=auto,
                        wide=wide, track_returns=True)
    assert env.wide == wide and env.ep_return is not None
    book = ReturnBook(N, dtype, 5e-5 if f32 else 1e-9)
    env.reset(); host.reset()
    if lean is not None:
        lean.reset()
    top = 0
    for t in range(T):
        a = torch.as_tensor(act[t]).to(tdt)
        obs, r, term, trunc, info = env.step(a)
        h_obs, h_r, h_done, h_info = host.step(act[t].astype(dtype), k)
        if f32:
            assert_same(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t)
        else:
            assert_close_f64(env, host, term, r, obs, info, h_obs, h_r, h_done, h_info, t)
        assert np.array_equal(trunc.cpu().numpy(), (h_info['cause'] & 32) != 0)
        book.add(r.cpu().numpy(), h_r, h_done.copy())
        book.check(env, host, t)
        if lean is not None:
            lean.step(a)
        top = max(top, int(host.steps.max()))
    s = env.stats()
    assert s['episodes'] >= N and s['timeout'] > 0 and s['env_steps'] <= N * k * T
    if max_steps > 2046:
        assert top > 2047
    if variant != 'Takeoff':
        assert sum(s[c] > 0 for c in ('landed', 'oob', 'angle', 'crashed', 'timeout')) >= 2
    if lean is not None:
        assert torch.equal(lean.state_planes, env.state_planes) and torch.equal(lean.meta, env.meta)
        ls = lean.stats()
        assert ls['return_sum'] == 0.0 and {c: ls[c] for c in COUNTS} == {c: s[c] for c in COUNTS}


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


# (variant, source, scale, offset, pid gains) as in tests/test_gpu_rollout_records.py: with ENDINGS and a 600 N
# injected reset force, every source's episodes time out, fly out of bounds, crash or tip over
ROLLOUT_SOURCES = [('Lander3D', 'const', None, None, None), ('Lander3D', 'randn', None, None, None),
                   ('Lander3D', 'uniform', 0.01, 0.0166, None), ('Lander3D', 'pid', 2.0e-3, 0.0149, {'descent_kd': 3.0}),
                   ('Lander2D', 'pid', 1e-3, 0.0159, {'descent_kd': 3.0}), ('Lander1D', 'pid', 1e-3, 0.0159, {'descent_kd': 3.0}),
                   ('Hover3D', 'pid_hover', 2 * HOVER, None, None), ('Hover2D', 'pid_hover', HOVER, HOVER, None),
                   ('Hover1D', 'pid_hover', HOVER, HOVER, None)]


def _rollout_cases():
    """The original cases keep their ids (Lander3D, default parameters, no statistics); the bookkeeping cases run
    every source in fp32 and fp64, and walk (per-step rewards, ending records, wide counters, auto-reset) through
    all 16 combinations, shifted between the two dtypes."""
    old = [pytest.param(None, src, None, id=src) for src in ('uniform', 'randn', 'const')]
    new = []
    for d, dtype in enumerate((np.float32, np.float64)):
        for j, (v, src, scale, offset, gains) in enumerate(ROLLOUT_SOURCES):
            c = (5 * j + 7 * d) % 16
            flags = dict(per_step=bool(c & 1), records=bool(c & 2), wide=bool(c & 4), auto=not c & 8)
            new.append(pytest.param(v, src, dict(flags, dtype=dtype, scale=scale, offset=offset, gains=gains),
                                    id='%s-%s-%s-%s-%s-%s-%s' % (v, src, 'f32' if d == 0 else 'f64', 'rewards' if flags['per_step'] else 'telescoped',
                                                                 'records' if flags['records'] else 'norecords',
                                                                 'wide' if flags['wide'] else 'compact', 'auto' if flags['auto'] else 'noreset')))
    return old + new


@pytest.mark.parametrize('variant,source,book', _rollout_cases())
def test_fp32_rollout_kernel_equals_the_host_instantiation(pkg, variant, source, book):
    """copter_rollout_f32 / _f64 (commands drawn on the device or computed by the PID heuristics): replay the
    recorded commands on the host."""
    if book is not None:
        return _rollout_bookkeeping(pkg, variant, source, **book)
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


def _rollout_bookkeeping(pkg, variant, source, dtype, scale, offset, gains, per_step, records, wide, auto):
    """Statistics and running returns of the rollout kernel: counts exactly the host ledger's after every launch,
    state and counters bit for bit (fp32) or to 1e-9 (fp64, counters exact).  ep_return: on the per-step reward
    path bit for bit the running sum of the recorded rewards; on the telescoped path (no per-step rewards) it is
    compared with a per-step twin at the tolerance of the telescoped reward sums (tests/test_gpu_rollout.py)."""
    f32 = dtype == np.float32
    tdt = torch.float32 if f32 else torch.float64
    N, T, seed, off = 1000 + 9, 40, 5, 3 << 32
    force = np.random.default_rng(0).uniform(-1, 1, (N, 3)) * 600.0
    kw = dict(dtype=tdt, seed=seed, env_offset=off, auto_reset=auto, wide_counters=wide, track_returns=True, **ENDINGS)
    env = pkg.CopterVecEnv(variant, N, **kw)
    env.reset(force=force)
    twin = None
    if not per_step:                        # the same launches with per-step rewards
        twin = pkg.CopterVecEnv(variant, N, **kw)
        twin.load_state_dict(env.state_dict())
    host = HostEnvBatch(variant, N, OracleParams(**ENDINGS), dtype=dtype, seed=seed, env_offset=off, auto_reset=auto,
                        wide=wide, track_returns=True)
    host.reset()
    h_force = force.astype(dtype)
    rec = dict(source=source, scale=scale, offset=offset, pid_gains=gains, record_actions=True, record_dones=True,
               record_causes=records, record_final_obs=records)
    book = ReturnBook(N, dtype, 5e-5 if f32 else 1e-9)
    for chunk in range(3):
        out = env.rollout(T, record_rewards=per_step, **rec)
        if twin is not None:
            t_out = twin.rollout(T, record_rewards=True, **rec)
            assert torch.equal(t_out['actions'], out['actions']) and torch.equal(t_out['dones'], out['dones'])
        rews = (out if twin is None else t_out)['rewards'].cpu().numpy()
        acts, dones = out['actions'].cpu().numpy(), out['dones'].cpu().numpy()
        for t in range(T):
            _, h_r, h_done, h_info = host.step(acts[t], 1, force=h_force)
            assert np.array_equal(dones[t], h_done), (chunk, t)
            if records:
                assert np.array_equal(out['causes'][t].cpu().numpy(), h_info['cause']), (chunk, t)
            assert float(np.max(np.abs(rews[t] - h_r) / np.maximum(np.abs(h_r), 1))) <= (5e-5 if f32 else 1e-9)
            book.add(rews[t], h_r, h_done.copy())
        x = env.state.cpu().numpy()
        if f32:
            assert np.array_equal(bits(x), bits(host.x)), chunk
        else:
            assert float(np.max(np.abs(x - host.x) / np.maximum(np.abs(host.x), 1))) <= 1e-9, chunk
        assert np.array_equal(env.steps.cpu().numpy(), host.steps) and np.array_equal(env.status.cpu().numpy(), host.status)
        assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64))
        book.check(env if twin is None else twin, host, chunk)
        s, _ = assert_counts(env, host, chunk)
        if twin is not None:                # the telescoped returns
            dev, ref = env.ep_return.cpu().numpy(), twin.ep_return.cpu().numpy()
            assert float(np.max(np.abs(dev - ref) / np.maximum(np.abs(ref), 1))) <= (1e-4 if f32 else 1e-10), chunk
            ts = twin.stats()['return_sum']
            assert abs(s['return_sum'] - ts) <= (1e-5 if f32 else 1e-10) * max(1.0, abs(ts)), chunk
    assert s['episodes'] >= N and s['env_steps'] == 3 * T * N
    assert sum(s[c] > 0 for c in ('landed', 'oob', 'angle', 'crashed', 'timeout')) >= 2


def _policy_cases():
    """The original cases ('1' the tcgen05 / TMEM kernel, '0' the warp-MMA kernel: Lander3D, compact counters,
    auto-reset) keep their ids; the bookkeeping cases run every variant x compact / wide x auto-reset on / off x
    exploration noise on / off on both kernels, and one launch with more tiles than resident CTAs."""
    cases = [pytest.param(kern, 'Lander3D', False, True, False, 777, id=kern) for kern in ('1', '0')]
    for kern in ('1', '0'):
        for v in ALL_VARIANTS:
            for wide in (False, True):
                for auto in (True, False):
                    for std in (False, True):
                        if (v, wide, auto, std) != ('Lander3D', False, True, False):
                            cases.append(pytest.param(kern, v, wide, auto, std, 777, id='%s-%s-%s-%s-%s' % (
                                kern, v, 'wide' if wide else 'compact', 'auto' if auto else 'noreset', 'std' if std else 'nostd')))
        cases.append(pytest.param(kern, 'Lander3D', True, True, True, 148 * 6 * 128 + 77, id='%s-Lander3D-wide-auto-std-manytiles' % kern))
    return cases


@pytest.mark.parametrize('kernel,variant,wide,auto,std,N', _policy_cases())
def test_fp32_policy_rollout_kernel_equals_the_host_instantiation(pkg, kernel, variant, wide, auto, std, N, monkeypatch):
    """copter_policy_rollout_f32: the env half of the fused policy + step kernels ('1': the tcgen05 / TMEM
    kernel, '0': the warp-MMA kernel), on the recorded actions: state and counters bit for bit, the statistics'
    counts exactly the host ledger's, ep_return bit for bit the running fp32 sum of the recorded rewards."""
    monkeypatch.setenv('COPTER_B200_POLICY_ROLLOUT_TC', kernel)
    T, reps, seed = (48, 4, 3) if N < 10000 else (32, 2, 3)
    kw = dict(TAKEOFF_SHELL, max_steps=60) if variant == 'Takeoff' else dict(ENDINGS)
    env = pkg.CopterVecEnv(variant, N, dtype=torch.float32, seed=seed, auto_reset=auto, wide_counters=wide, track_returns=True, **kw)
    host = HostEnvBatch(variant, N, OracleParams(**kw), dtype=np.float32, seed=seed, auto_reset=auto, wide=wide, track_returns=True)
    env.reset(); host.reset()
    O, A = env.obs_size, env.action_size
    pol = pkg.mlp_policy(O, A, dtype=torch.float32, seed=5)
    pro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=0.5 * 0.0166, out_offset=0.0166, store_actions=True,
                                 action_std=0.004 if std else None)
    book = ReturnBook(N, np.float32, 5e-5)
    for rep in range(reps):
        rewards, dones, _ = pro.run()
        acts, dones, rews = pro.actions.cpu().numpy(), dones.cpu().numpy(), rewards.cpu().numpy()
        for t in range(T):
            _, h_r, h_done, _ = host.step(acts[t], 1)
            assert np.array_equal(dones[t], h_done), (rep, t)
            book.add(rews[t], h_r, h_done.copy())
        assert np.array_equal(bits(env.state.cpu().numpy()), bits(host.x))
        assert np.array_equal(env.steps.cpu().numpy(), host.steps) and np.array_equal(env.status.cpu().numpy(), host.status)
        assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64))
        book.check(env, host, rep)
    s = env.stats()
    assert s['episodes'] > 0 and s['env_steps'] == reps * T * N


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

