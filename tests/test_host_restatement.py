"""CPU checks of the KERNEL arithmetic itself: gym_copter_b200/csrc/copter_core.h -- the header the
CUDA kernels are built from -- instantiated on the host (oracle/copter_host.cpp) and compared with the
oracle that is pinned to the executed reference.

  * fp64 instantiation vs the numpy oracle: state / reward <= 1e-9 (measured ~2e-13), done flags, flight
    status, step counters and episode indices exact -- every variant, K in {1, 3}.
  * fp32 instantiation vs the fp64 C oracle: state / obs / reward <= 1e-4 over 1000 steps (north_star),
    and the rate at which an fp32 rounding flips a threshold comparison (z > 0 && dz > 0, |x| >= 10,
    |phi| >= pi/4, |dz| > 10 ...) one step early / late is MEASURED per action stream, printed, recorded in
    profiles/r2_fp32_flip_rates.json (by tools/flip_rates.py, same code) and bounded here at the measured
    rate plus margin.  The GPU then has to reproduce this instantiation bit for bit
    (tests/test_gpu_host_exact.py), so these rates are the fp32 path's, not one compiler's.
"""
import numpy as np
import pytest

from oracle.copter_oracle import ALL_VARIANTS, DynamicsBatch, EnvBatch, OracleParams, reset_force
from oracle.c_oracle import CEnvBatch
from oracle.host_restatement import CAUSE_STATS, STAT_NAMES, HostDynamicsBatch, HostEnvBatch, sincos_f32, load, make_params

HOVER = 0.016560178212092172


def stream(kind, rng, n, t, a):
    if kind == 'const':
        return np.full((t, n, a), 1.625e-2, np.float32)
    if kind == 'randn':
        return (1.625e-2 * rng.standard_normal((t, n, a))).astype(np.float32)
    if kind == 'hover':
        return (HOVER * (1 + 0.1 * rng.uniform(-1, 1, (t, n, a)))).astype(np.float32)
    return rng.uniform(-1, 1, (t, n, a)).astype(np.float32)


def mixed_streams(rng, n, t, a):
    act = np.empty((t, n, a), np.float32)
    for i, kind in enumerate(('const', 'randn', 'hover', 'unif')):
        act[:, i::4] = stream(kind, rng, len(range(i, n, 4)), t, a)
    return act


@pytest.mark.parametrize('k', [1, 3])
@pytest.mark.parametrize('variant', list(ALL_VARIANTS))
def test_fp64_instantiation_matches_the_reference_pinned_oracle(variant, k):
    N, T = 256, 360
    rng = np.random.default_rng(sum(map(ord, variant)) + k)
    A = ALL_VARIANTS[variant][2]
    act = mixed_streams(rng, N, T, A).astype(np.float64)
    kw = dict(initial_altitude=0.0, initial_random_force=0.0, max_steps=150) if variant == 'Takeoff' else {}
    if variant == 'Takeoff':
        act = np.abs(act) + rng.uniform(0, 0.01, act.shape)          # commands that do take off
        act[:, ::5] *= -1                                           # unclipped: the sign must not matter
    h = HostEnvBatch(variant, N, OracleParams(**kw), dtype=np.float64, seed=7, env_offset=1 << 33)
    o = EnvBatch(variant, N, OracleParams(**kw), seed=7, env_offset=1 << 33)
    assert np.array_equal(h.reset(), o.reset())
    worst = worst_r = 0.0
    episodes = 0
    for t in range(T):
        ob, r, d, info = h.step(act[t], k)
        o_ob, o_r, o_d, o_info = o.step(act[t], k)
        assert np.array_equal(d, o_d), (t, np.nonzero(d != o_d))
        assert np.array_equal(h.status, o.dyn.status) and np.array_equal(h.steps, o.steps)
        assert np.array_equal(h.episode, o.episode) and np.array_equal(info['cause'], o_info['cause'])
        assert np.array_equal(info['executed'], o_info['steps_taken'])
        assert np.array_equal(info['final_steps'][o_d], o_info['final_steps'][o_d])
        worst = max(worst, float(np.max(np.abs(h.x - o.dyn.x) / np.maximum(np.abs(o.dyn.x), 1))))
        worst_r = max(worst_r, float(np.max(np.abs(r - o_r) / np.maximum(np.abs(o_r), 1))))
        assert np.array_equal(ob, h.x[:, list(ALL_VARIANTS[variant][1])].astype(np.float32))
        episodes += int(o_d.sum())
    assert worst <= 1e-9 and worst_r <= 1e-9, (worst, worst_r)
    assert episodes >= 40
    if variant == 'Takeoff':
        assert (h.x[:, 4] < -0.5).any() and (h.status == 3).any()       # vehicles did leave the ground


@pytest.mark.parametrize('auto_reset', [True, False], ids=['auto', 'noreset'])
@pytest.mark.parametrize('k', [1, 3, 16])
@pytest.mark.parametrize('variant', list(ALL_VARIANTS))
def test_host_ledger_counts_equal_the_oracle(variant, k, auto_reset):
    """HostEnvBatch.stats() -- the statistics the kernels keep -- against the same counts derived from the
    numpy oracle's endings (steps_taken, final_steps, cause) on the same commands: exact.  A short step limit,
    a low start and tight bounds end episodes of every kind; the runs stay below 2047 steps, where the oracle's
    unsaturated counter and the counter field agree."""
    N, T = 64, 384 // k
    rng = np.random.default_rng(5 * k + sum(map(ord, variant)))
    A = ALL_VARIANTS[variant][2]
    act = mixed_streams(rng, N, T, A).astype(np.float64)
    kw = dict(max_steps=60, initial_altitude=1.0, bounds=2.0)
    if variant == 'Takeoff':
        kw.update(initial_altitude=0.0, initial_random_force=0.0)
        act = np.abs(act) + rng.uniform(0, 0.01, act.shape)
    h = HostEnvBatch(variant, N, OracleParams(**kw), dtype=np.float64, seed=9, auto_reset=auto_reset, track_returns=True)
    o = EnvBatch(variant, N, OracleParams(**kw), seed=9, auto_reset=auto_reset)
    h.reset(); o.reset()
    want = dict.fromkeys(('episodes', 'length_sum', 'env_steps') + tuple(c for c, _ in CAUSE_STATS), 0)
    o_ret, o_return_sum = np.zeros(N), 0.0
    for t in range(T):
        _, r, d, _ = h.step(act[t], k)
        _, o_r, o_d, o_info = o.step(act[t], k)
        assert np.array_equal(d, o_d), t
        want['episodes'] += int(o_d.sum())
        want['length_sum'] += int((o_info['final_steps'][o_d] - 1).sum())
        want['env_steps'] += int(o_info['steps_taken'].sum())
        for name, bit in CAUSE_STATS:
            want[name] += int(((o_info['cause'][o_d] & bit) != 0).sum())
        o_ret += o_r
        o_return_sum += float(o_ret[o_d].sum())
        o_ret[o_d] = 0.0
    assert int(o.steps.max()) < 2047
    s = h.stats()
    assert {k_: s[k_] for k_ in want} == {k_: float(v) for k_, v in want.items()}, (s, want)
    assert set(s) == set(STAT_NAMES) | {'mean_return', 'mean_length'}
    assert s['episodes'] >= N and s['timeout'] > 0
    assert variant == 'Takeoff' or sum(s[c] > 0 for c, _ in CAUSE_STATS) >= (2 if variant.endswith('1D') else 3), s
    # the returns: the K-fused host telescopes what the oracle sums step by step
    assert abs(s['return_sum'] - o_return_sum) <= 1e-9 * max(abs(o_return_sum), 1.0) * T, (s['return_sum'], o_return_sum)
    assert np.allclose(h.ep_return, o_ret, rtol=1e-9, atol=1e-9)
    # reset() zeroes the running returns, not the ledger
    h.reset()
    assert not h.ep_return.any() and h.stats() == s


def fp32_flip_study(variant, kind, k, n, t, seed=3):
    """fp32 host instantiation vs the fp64 C oracle on one action stream: returns a dict with the
    number of oracle episodes, the number of envs whose discrete outputs diverged (and left the
    comparison), and the worst errors over the envs still in step."""
    rng = np.random.default_rng(seed)
    A = ALL_VARIANTS[variant][2]
    act = stream(kind, rng, n, t // k, A)
    h = HostEnvBatch(variant, n, dtype=np.float32, seed=11)
    o = CEnvBatch(variant, n, seed=11)
    h.reset(); o.reset()
    sync = np.ones(n, bool)
    out = dict(variant=variant, stream=kind, k=k, envs=n, steps=t, episodes=0, flips=0, state=0.0, state_by_norm=0.0, reward=0.0)
    for i in range(t // k):
        ob, r, d, info = h.step(act[i], k)
        o_ob, o_r, o_d, o_info = o.step(act[i].astype(np.float64), k)
        # a K-fused reward is the sum of K step rewards, each held to |err| <= tol * max(|r_step|, 1)
        r_err = np.abs(r - o_r) / np.maximum(np.abs(o_r), k)
        bad = (d != o_d) | (h.status != o.status) | (h.steps != o.steps) | (h.episode.astype(np.int64) != o.episode)
        # two more signatures of a flipped threshold: inside a K-fused launch both sides can end one substep
        # apart (both done, different step counters at the end), and |dz| > dz_max (lander.py:55) moves the
        # 100-point shaping penalty to the neighbouring step.  The env leaves the comparison as a flip.
        bad |= (o_d & d & (info['final_steps'] != o_info['final_steps'])) | (np.abs(r - o_r) > 10.0)
        bad &= sync
        out['flips'] += int(bad.sum())
        sync &= ~bad
        out['episodes'] += int((o_d & sync).sum())
        if sync.any():
            e = np.abs(h.x - o.x)
            out['state'] = max(out['state'], float((e / np.maximum(np.abs(o.x), 1))[sync].max()))
            out['state_by_norm'] = max(out['state_by_norm'], float((e / np.maximum(np.abs(o.x).max(1, keepdims=True), 1))[sync].max()))
            out['reward'] = max(out['reward'], float(r_err[sync].max()))
    out['flips_per_episode'] = out['flips'] / max(out['episodes'], 1)
    return out


# measured (tools/flip_rates.py, 16384 envs x 1000 steps, profiles/r2_fp32_flip_rates.json): const 2.1e-3,
# randn 1.1e-4, hover 0, unif 3e-6 flips per episode.  The constant-thrust stream is the worst case by
# construction: every episode ends by crossing z = 0 at dz = 2.7 m/s, and z is then known to 5e-5.
FLIP_BOUND = {'const': 6e-3, 'randn': 1e-3, 'hover': 1e-3, 'unif': 1e-4}


@pytest.mark.parametrize('k', [1, 4])
@pytest.mark.parametrize('kind', ['const', 'randn', 'hover', 'unif'])
def test_fp32_instantiation_within_tolerance_and_flip_rate(kind, k):
    s = fp32_flip_study('Lander3D', kind, k, 2048, 1000)
    print('fp32 vs fp64 oracle:', s)
    assert s['episodes'] >= 2000
    # saturating commands (U(-1,1): 60x hover thrust) are judged against the size of the state vector
    assert (s['state_by_norm'] if kind == 'unif' else s['state']) <= 1e-4, s
    assert s['state'] <= 1e-3 and s['reward'] <= 1e-4, s
    assert s['flips'] <= max(2, FLIP_BOUND[kind] * s['episodes']), s


def test_fp32_sincos_reduction_accuracy():
    """The shared fp32 sin / cos: polynomials on [-pi/4, pi/4], fp64 Cody-Waite reduction beyond."""
    rng = np.random.default_rng(0)
    a = np.concatenate([rng.uniform(-np.pi / 4, np.pi / 4, 20000), rng.uniform(-200, 200, 20000),
                        rng.uniform(-1e5, 1e5, 20000), [0.0, np.pi / 4, -np.pi / 4, 0.78539816, 0.7853982, 1e6, -3e7]]).astype(np.float32)
    s, c = sincos_f32(a)
    rs, rc = np.sin(a.astype(np.float64)), np.cos(a.astype(np.float64))
    assert np.max(np.abs(s - rs)) <= 1.5e-7 and np.max(np.abs(c - rc)) <= 1.5e-7
    bad = np.array([np.inf, -np.inf, np.nan], np.float32)
    s, c = sincos_f32(bad)
    assert np.isnan(s).all() and np.isnan(c).all()


@pytest.mark.parametrize('dtype,tol', [(np.float64, 1e-11), (np.float32, 2e-5)])
def test_dynamics_facade_instantiation_vs_oracle(dtype, tol):
    rng = np.random.default_rng(2)
    N = 600
    s0 = rng.normal(0, 1, (N, 12)) * np.array([3, 1, 3, 1, 2, 1, .3, .2, .3, .2, .5, .2])
    s0[: N // 4, 4] = np.abs(s0[: N // 4, 4]) * 0.01
    h, o = HostDynamicsBatch(N, dtype=dtype), DynamicsBatch(N)
    h.set_state(s0); o.set_state(s0.astype(dtype).astype(np.float64))
    for t in range(60):
        m = (HOVER * (1 + 0.5 * rng.uniform(-1, 1, (N, 4)))).astype(np.float32).astype(np.float64)
        if t % 7 == 0:
            f = rng.uniform(-5, 5, (N, 6)).astype(np.float32).astype(np.float64)
            h.set_perturb(f); o.set_perturb(f)
        h.set_motors(m); o.set_motors(m)
        if dtype == np.float64:
            assert np.array_equal(h.status, o.status) and np.array_equal(h.ticks, o.ticks)
    same = h.status == o.status
    assert same.mean() > 0.99
    assert float(np.max((np.abs(h.x - o.x) / np.maximum(np.abs(o.x), 1))[same])) <= tol


def test_wide_counters_and_reset_episode_semantics():
    """max_steps beyond the 11-bit field with wide counters (the reference takes any max_steps,
    envs/task.py:35), and reset(): first call -> episode 0, later calls -> next episode (new force)."""
    N = 64
    kw = dict(max_steps=5000, initial_random_force=1e-3)         # (almost) unperturbed hover: nothing else ends the episode
    h = HostEnvBatch('Hover3D', N, OracleParams(**kw), dtype=np.float64, seed=5, wide=True)
    o = EnvBatch('Hover3D', N, OracleParams(**kw), seed=5)
    o.ep_mask = 0xFFFFFFFF
    h.reset(); o.reset()
    rng = np.random.default_rng(1)
    a = np.full((N, 4), HOVER)
    top = 0
    for t in range(5100):
        ob, r, d, _ = h.step(a)
        o_ob, o_r, o_d, _ = o.step(a)
        assert np.array_equal(d, o_d) and np.array_equal(h.steps, o.steps)
        top = max(top, int(h.steps.max()))
    assert top == 5000 and (h.episode == 1).all()        # counted past 2047, timed out at max_steps, reset
    assert float(np.max(np.abs(h.x - o.dyn.x))) <= 1e-9
    # reset() again: every env moves to its next episode, and the reset force follows the episode index
    e0 = h.episode.copy()
    h.reset(); o.reset()
    assert np.array_equal(h.episode, e0 + 1) and np.array_equal(h.episode, o.episode)
    h.step(a); o.step(a)
    assert float(np.max(np.abs(h.x - o.dyn.x))) <= 1e-12
    f = reset_force(5, h.env_ids, h.episode, 30.0)          # (default parameters: +-30 N)
    out = np.zeros((N, 3), np.float32)
    import ctypes as C
    load().copter_host_reset_force_f32(C.byref(make_params()), C.c_int64(N), h.env_ids.ctypes.data_as(C.c_void_p),
                                       h.episode.ctypes.data_as(C.c_void_p), C.c_uint64(5), out.ctypes.data_as(C.c_void_p))
    assert np.array_equal(out, f.astype(np.float32))
    # compact counters refuse what they cannot count
    with pytest.raises(AssertionError):
        HostEnvBatch('Hover3D', 4, OracleParams(max_steps=5000), dtype=np.float64).step(np.zeros((4, 4)))
