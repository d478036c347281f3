"""GPU tests of the rows next to the step (SURVEY.md 8f): fused multi-step rollouts with
on-device action sources, policy-in-the-loop rollouts under a CUDA graph, the host-array
pipeline, and the lander.py-compatible CSV export."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import noise_oracle                                           # noqa: E402
from oracle.copter_oracle import EnvBatch, VARIANTS, source_actions      # noqa: E402


def merr(a, ref):
    a, ref = np.asarray(a, np.float64), np.asarray(ref, np.float64)
    return float(np.max(np.abs(a - ref) / np.maximum(np.abs(ref), 1.0)))


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


@pytest.mark.parametrize('dtype,nd', [(torch.float64, np.float64), (torch.float32, np.float32)])
@pytest.mark.parametrize('source', ['const', 'randn', 'uniform'])
def test_action_sources_match_their_definition(pkg, source, dtype, nd):
    n, T, off, seed = 3001, 5, 10 ** 11, 0xFEEDFACE1234
    env = pkg.CopterVecEnv('Lander3D', n, dtype=dtype, seed=seed, env_offset=off)
    env.reset()
    env.rollout_step = 2 ** 33 + 5          # exercises the high word of the step counter
    out = env.rollout(T, source=source, record_actions=True)
    acts = out['actions'].cpu().numpy()
    ids = np.arange(n, dtype=np.uint64) + np.uint64(off)
    for t in range(T):
        kw = dict(const=(0.0, 1.625e-2), randn=(1.625e-2, 0.0), uniform=(1.0, 0.0))[source]
        ref = source_actions(seed, ids, 2 ** 33 + 5 + t, source, kw[0], kw[1], 4, nd)
        if source == 'randn':
            assert np.max(np.abs(acts[t] - ref)) <= (1e-13 if nd == np.float64 else 2e-7)
        else:
            assert np.array_equal(acts[t], ref)
    if source == 'randn':
        z = acts / 1.625e-2
        assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02
        assert abs(np.corrcoef(z.reshape(-1, 4).T)[0, 1]) < 0.02


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('variant,source', [('Lander3D', 'randn'), ('Lander3D', 'uniform'), ('Lander2D', 'randn'),
                                            ('Hover3D', 'const'), ('Lander1D', 'uniform')])
def test_rollout_equals_single_steps_and_oracle(pkg, variant, source, dtype):
    """One fused launch of T steps == T launches of step() on the recorded commands (same
    device arithmetic; the compiler may contract FMAs differently in the two kernels, so
    floats are compared at a few ulp, flags and counters bit for bit), and == the oracle
    within the path's tolerance."""
    n, T, seed = 1500, 120, 77
    fused = pkg.CopterVecEnv(variant, n, dtype=dtype, seed=seed, track_returns=True)
    lean = pkg.CopterVecEnv(variant, n, dtype=dtype, seed=seed, track_returns=True)     # no per-step rewards: telescoped sums
    single = pkg.CopterVecEnv(variant, n, dtype=dtype, seed=seed, track_returns=True)
    orc = EnvBatch(variant, n, seed=seed)
    fused.reset(); lean.reset(); single.reset(); orc.reset()
    out = fused.rollout(T, source=source, record_rewards=True, record_dones=True, record_actions=True)
    out_lean = lean.rollout(T, source=source, record_dones=True)
    acts = out['actions']
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    ulps = 1e-12 if dtype == torch.float64 else 1e-5
    sync = np.ones(n, bool)
    rsum = torch.zeros(n, dtype=dtype, device='cuda')
    dany = torch.zeros(n, dtype=torch.bool, device='cuda')
    for t in range(T):
        obs, r, term, _, _ = single.step(acts[t])
        assert torch.equal(term, out['dones'][t])
        assert merr(out['rewards'][t].cpu().numpy(), r.cpu().numpy()) <= ulps
        rsum += r
        dany |= term
        o_obs, o_r, o_done, _ = orc.step(acts[t].cpu().numpy().astype(np.float64))
        d = term.cpu().numpy()
        sync &= (d == o_done) & (single.status.cpu().numpy() == orc.dyn.status)
        assert merr(r.cpu().numpy()[sync], o_r[sync]) <= tol
    assert torch.equal(fused.meta, single.meta) and torch.equal(out['done_any'], dany)
    assert merr(fused.state.cpu().numpy(), single.state.cpu().numpy()) <= ulps
    assert merr(out['obs'].cpu().numpy(), single.obs.cpu().numpy()) <= max(ulps, 1.2e-7)
    assert merr(out['reward_sum'].cpu().numpy(), rsum.cpu().numpy()) <= 10 * ulps
    # the telescoped path: same states and flags, reward sums equal up to summation order
    assert torch.equal(out_lean['dones'], out['dones']) and torch.equal(lean.meta, fused.meta)
    assert merr(lean.state.cpu().numpy(), fused.state.cpu().numpy()) <= ulps
    assert merr(out_lean['reward_sum'].cpu().numpy(), rsum.cpu().numpy()) <= (1e-10 if dtype == torch.float64 else 1e-4)
    ls = lean.stats()
    fs, ss = fused.stats(), single.stats()
    assert ls['episodes'] == ss['episodes'] and ls['length_sum'] == ss['length_sum']
    assert abs(ls['return_sum'] - ss['return_sum']) <= 1e-5 * max(1.0, abs(ss['return_sum']))
    for k in ('episodes', 'length_sum', 'landed', 'bonus', 'crashed', 'oob', 'angle', 'timeout', 'env_steps'):
        assert fs[k] == ss[k], k
    assert abs(fs['return_sum'] - ss['return_sum']) <= 1e-6 * max(1.0, abs(ss['return_sum']))
    assert fs['env_steps'] == n * T
    assert sync.sum() >= (n if dtype == torch.float64 else 0.99 * n)
    if source != 'uniform' or dtype == torch.float64:
        assert merr(fused.state.cpu().numpy()[sync], orc.dyn.x[sync]) <= tol


def test_rollout_is_independent_of_launch_partition(pkg):
    n, seed = 777, 3
    a = pkg.CopterVecEnv('Lander3D', n, seed=seed)
    b = pkg.CopterVecEnv('Lander3D', n, seed=seed)
    a.reset(); b.reset()
    a.rollout(60, source='randn')
    for chunk in (1, 7, 20, 32):
        b.rollout(chunk, source='randn')
    assert torch.equal(a.state, b.state) and torch.equal(a.meta, b.meta) and a.rollout_step == b.rollout_step == 60


def test_policy_rollout_graph_equals_eager(pkg):
    n, T = 4096, 6
    envs = [pkg.CopterVecEnv('Lander3D', n, seed=5) for _ in range(2)]
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=1)
    scaled = lambda obs: 0.0166 * (1 + 0.2 * pol(obs))         # noqa: E731  (keeps the copters flying)
    for e in envs:
        e.reset()
    graph = pkg.PolicyRollout(envs[0], scaled, T, store_obs=True, use_cuda_graph=True)
    eager = pkg.PolicyRollout(envs[1], scaled, T, store_obs=True, use_cuda_graph=False)
    for it in range(3):
        r1, d1, o1 = graph.run()
        r2, d2, o2 = eager.run()
        assert torch.equal(r1, r2) and torch.equal(d1, d2) and torch.equal(o1, o2)
        assert torch.equal(graph.obs, eager.obs)
    assert torch.equal(envs[0].state, envs[1].state)
    assert r1.shape == (T, n) and d1.dtype == torch.bool


def test_step_host_matches_device_step(pkg):
    n = 70000            # above the direct path's limit: the chunked copy pipeline
    rng = np.random.default_rng(0)
    e1 = pkg.CopterVecEnv('Lander3D', n, seed=4, track_stats=True)
    e2 = pkg.CopterVecEnv('Lander3D', n, seed=4, track_stats=True)
    e1.reset(); e2.reset()
    for t in range(12):
        a = (1.625e-2 * rng.standard_normal((n, 4))).astype(np.float32)
        if t % 2:
            a[::3] = rng.uniform(-1, 1, (len(a[::3]), 4)).astype(np.float32)
        obs, r, term, trunc, _ = e1.step_host(a, chunk_envs=8192, n_streams=3)
        o2, r2, t2, _, _ = e2.step(torch.as_tensor(a))
        assert isinstance(obs, np.ndarray) and obs.dtype == np.float32 and term.dtype == np.bool_
        assert np.array_equal(obs, o2.cpu().numpy()) and np.array_equal(r, r2.cpu().numpy())
        assert np.array_equal(term, t2.cpu().numpy()) and not trunc.any()
    assert torch.equal(e1.state, e2.state) and e1.stats() == e2.stats()
    e1.close()


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
@pytest.mark.parametrize('n', [1, 37, 256, 5000])
def test_step_host_direct_path_matches_device_step(pkg, n, dtype):
    """Shards of at most 65 536 envs with page-locked host arrays: the step kernel reads the commands from and writes
    observation / reward / done / cause / terminal observation to the HOST arrays themselves (one launch, one
    synchronisation: the single-env facade's path).  Same numbers as the device-tensor step, K = 1 and K = 3."""
    rng = np.random.default_rng(n)
    for k in (1, 3):
        kw = dict(seed=6, dtype=dtype, k_substeps=k, report_cause=True, keep_final_obs=True, max_steps=40)
        e1, e2 = pkg.CopterVecEnv('Lander3D', n, **kw), pkg.CopterVecEnv('Lander3D', n, **kw)
        e1.reset(); e2.reset()
        npdt = np.float32 if dtype == torch.float32 else np.float64
        ended = 0
        for t in range(60):
            a = (1.625e-2 * (1 + 0.5 * rng.standard_normal((n, 4)))).astype(npdt)
            if t % 5 == 4:
                a[::2] = rng.uniform(-1, 1, (len(a[::2]), 4)).astype(npdt)
            obs, r, term, trunc, info = e1.step_host(a)
            o2, r2, t2, tr2, i2 = e2.step(torch.as_tensor(a))
            assert np.array_equal(obs, o2.cpu().numpy()) and np.array_equal(r, r2.cpu().numpy())
            assert np.array_equal(term | trunc, (t2 | tr2).cpu().numpy()) and np.array_equal(trunc, tr2.cpu().numpy())
            assert np.array_equal(info['cause'], i2['cause'].cpu().numpy())
            done = term | trunc
            assert np.array_equal(info['final_obs'][done], i2['final_obs'].cpu().numpy()[done])
            ended += int(done.sum())
        assert ended > 0 and torch.equal(e1.state, e2.state) and torch.equal(e1.steps, e2.steps)
        e1.close()


def test_step_host_with_pageable_arrays_takes_the_copy_pipeline(pkg):
    """A caller of the C ABI whose host arrays are NOT page-locked (plain numpy): the direct path must not be taken
    (the kernel cannot address pageable memory) -- the call falls back to the copy pipeline and gives the same numbers."""
    import ctypes as C
    from gym_copter_b200 import _lib
    n = 64
    e1, e2 = pkg.CopterVecEnv('Lander3D', n, seed=9), pkg.CopterVecEnv('Lander3D', n, seed=9)
    e1.reset(); e2.reset()
    e1.host_buffers()                                   # creates the pipeline-side state lazily, as step_host would
    pipe = C.c_void_p()
    _lib.check(e1._lib.copter_pipeline_create(2, C.byref(pipe)), 'copter_pipeline_create')
    rng = np.random.default_rng(3)
    obs, rew, done = np.zeros((n, 10), np.float32), np.zeros(n, np.float32), np.zeros(n, np.uint8)     # pageable
    for t in range(20):
        a = (1.625e-2 * (1 + 0.3 * rng.standard_normal((n, 4)))).astype(np.float32)
        b = e1._buffers(e1._action, e1._force)
        rc = e1._lib.copter_step_host_f32(pipe, C.byref(e1.params), C.byref(b), a.ctypes.data, obs.ctypes.data, rew.ctypes.data,
                                          done.ctypes.data, None, None, n, 0, e1.seed_value, 1, 0, _lib.F_AUTO_RESET, 1 << 20,
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, rc
        o2, r2, t2, _, _ = e2.step(torch.as_tensor(a))
        assert np.array_equal(obs, o2.cpu().numpy()) and np.array_equal(rew, r2.cpu().numpy()) and np.array_equal(done.astype(bool), t2.cpu().numpy())
    assert torch.equal(e1.state, e2.state)
    e1._lib.copter_pipeline_destroy(pipe)


def test_csv_export_matches_lander_py_format(pkg, tmp_path):
    env = pkg.make('gym_copter:Lander-v0')
    obs, _ = env.reset(force=[1.0, 2.0, 3.0])
    path = os.path.join(tmp_path, 'traj.csv')
    with pkg.CsvTrajectoryWriter(path, env) as w:
        for k in range(5):
            a = 1.625e-2 * np.ones(4)
            obs, r, done, _, _ = env.step(a)
            w.write(a, obs)
    lines = open(path).read().strip().split('\n')
    # lander.py:33-38 header, :48-54 rows
    assert lines[0] == 't,m1,m2,m3,m4,X,dX,Y,dY,Z,dZ,Phi,dPhi,Theta,dTheta'
    assert len(lines) == 6 and all(len(l.split(',')) == 15 for l in lines[1:])
    first = lines[1].split(',')
    assert first[0] == '0.000000' and first[1] == '0.016250' and lines[2].split(',')[0] == '0.010000'
    assert abs(float(first[9]) - (-10.0)) < 1e-6


def test_cause_and_timelimit_truncation(pkg):
    """`truncated` mirrors gymnasium's TimeLimit(max_episode_steps): set exactly on the step on
    which the env's own step limit fires (SURVEY.md 3.4: both fire on the same user step)."""
    from gym_copter_b200._lib import CAUSE_TIMEOUT, CAUSE_OOB, CAUSE_ANGLE, CAUSE_CRASHED
    n = 600
    env = pkg.CopterVecEnv('Hover3D', n, dtype=torch.float64, seed=1, report_cause=True, max_steps=40)
    orc = EnvBatch('Hover3D', n, seed=1, params=__import__('oracle.copter_oracle', fromlist=['OracleParams']).OracleParams(max_steps=40))
    env.reset(); orc.reset()
    rng = np.random.default_rng(0)
    seen = 0
    for t in range(100):
        a = 0.01656 * (1 + 0.02 * rng.uniform(-1, 1, (n, 4)))           # calm half: runs into the step limit
        a[1::2, 1:3] *= 4.0                                              # other half: rolls over (task.py:116)
        a = a.astype(np.float32)
        obs, r, term, trunc, info = env.step(a)
        o_obs, o_r, o_done, o_info = orc.step(a.astype(np.float64))
        assert np.array_equal(info['cause'].cpu().numpy(), o_info['cause'].astype(np.uint8))
        assert np.array_equal(trunc.cpu().numpy(), (o_info['cause'] & CAUSE_TIMEOUT) != 0)
        assert not (trunc & ~term).any()
        seen |= int(np.bitwise_or.reduce(o_info['cause']))
    assert seen & CAUSE_TIMEOUT and seen & (CAUSE_OOB | CAUSE_ANGLE | CAUSE_CRASHED)


def test_zero_copy_observation_mode(pkg):
    """write_obs=False changes nothing but the skipped observation write; a policy whose first
    layer reads the state planes in place computes the same actions as one reading obs."""
    n = 5000
    a_env = pkg.CopterVecEnv('Lander3D', n, seed=9)
    b_env = pkg.CopterVecEnv('Lander3D', n, seed=9, write_obs=False)
    a_env.reset(); b_env.reset()
    lin = torch.nn.Linear(10, 64).cuda()
    planar = pkg.PlanarLinear(lin, 10)
    g = torch.Generator(device='cuda').manual_seed(0)
    for t in range(25):
        act = 1.625e-2 * torch.randn((n, 4), device='cuda', generator=g)
        obs, r1, d1, _, _ = a_env.step(act)
        none, r2, d2, _, _ = b_env.step(act)
        assert none is None and torch.equal(r1, r2) and torch.equal(d1, d2)
        assert torch.equal(a_env.state, b_env.state)
        with torch.no_grad():
            y1, y2 = lin(obs), planar(b_env.planar_obs())
        assert torch.allclose(y1, y2, rtol=1e-5, atol=1e-5)
    ro = pkg.PolicyRollout(b_env, lambda planes: 0.0166 * (1 + 0.1 * torch.tanh(planar(planes)[:, :4])), 4, planar=True)
    r, d, _ = ro.run()
    assert r.shape == (4, n)


@pytest.mark.parametrize('dtype,tol', [(torch.float64, 1e-7), (torch.float32, 1e-4)])
def test_pid_heuristic_rollout_vs_oracle(pkg, dtype, tol):
    """Closed loop on the device (PID heuristic + env, one launch per chunk) against the closed
    loop of the two oracles (PID restatement pinned to the reference's controller classes +
    env restatement), with gains scaled to the live vehicle so that the copters really land.
    The controller reads the float32 observation, as the reference's caller does, so the loop
    contains a quantiser: a last-bit difference of the fp64 state can flip a float32 rounding
    and move the command by 6e-8 relative -- hence 1e-7, not 1e-9, for the fp64 closed loop."""
    from oracle.pid_oracle import LanderHeuristicBatch
    n, T, seed = 1024, 1000, 12
    # the reference's gains drive its attic vehicle model; for the live vehicle (hover command
    # 0.01656) the mixer output is scaled into motor units and the descent loop damped harder
    scale, offset, kd = 2.0e-3, 0.0149, 3.0
    env = pkg.CopterVecEnv('Lander3D', n, dtype=dtype, seed=seed, track_stats=True)
    orc = EnvBatch('Lander3D', n, seed=seed)
    pid = LanderHeuristicBatch(n, scale=scale, offset=offset, descent_kd=kd)
    obs = env.reset()[0].cpu().numpy()
    o_obs = orc.reset()
    sync = np.ones(n, bool)
    worst_a = worst_s = 0.0
    for chunk in range(T // 50):
        out = env.rollout(50, source='pid', scale=scale, offset=offset, pid_gains={'descent_kd': kd},
                          record_actions=True, record_dones=True)
        acts, dones = out['actions'].cpu().numpy(), out['dones'].cpu().numpy()
        for t in range(50):
            a = pid.act(o_obs)
            worst_a = max(worst_a, float((np.abs(acts[t] - a) / np.maximum(np.abs(a), 1e-2))[sync].max()))
            o_obs, o_r, o_done, _ = orc.step(a)
            sync &= dones[t] == o_done
        sync &= env.status.cpu().numpy() == orc.dyn.status
        worst_s = max(worst_s, merr(env.state.cpu().numpy()[sync], orc.dyn.x[sync]))
    assert sync.sum() >= (n if dtype == torch.float64 else 0.97 * n), sync.sum()
    assert worst_s <= tol and worst_a <= (1e-5 if dtype == torch.float64 else 2e-3), (worst_s, worst_a)
    s = env.stats()
    assert s['bonus'] > 0.9 * s['episodes'] > 0            # a landing workload: soft touch-downs inside the target


@pytest.mark.parametrize('dtype,tol', [(torch.float64, 5e-6), (torch.float32, 1e-4)])
def test_pid_hover_heuristic_rollout_vs_oracle(pkg, dtype, tol):
    """The hover demo's heuristic (attic/mars/hover3d.py:65-92: altitude hold + position hold +
    roll/pitch/yaw rate loops) closed around Hover3D on the device, against the closed loop of the
    two oracles.  The reference's own gains, with the mixer output scaled by twice the hover
    command so that t = 1/2 hovers the live vehicle: every copter climbs from the reset altitude to
    the 5 m set-point, holds it, and the episode ends by the 1000-step limit.
    Tolerance of the fp64 loop: the controllers read the float32 observation, and this loop
    regulates z to the set-point THROUGH that quantiser (ulp32(5 m) = 4.8e-7): a last-bit
    difference of the fp64 state that flips one float32 rounding moves the closed-loop state by
    about one such ulp (measured 8e-7 over 1200 steps), so the bound is a few float32 ulps of the
    regulated altitude instead of the open-loop 1e-9.  Commands agree to 1e-5 relative throughout."""
    from oracle.pid_oracle import HoverHeuristicBatch
    n, T, seed = 512, 1200, 5
    scale = 2 * 0.016560178212092172
    env = pkg.CopterVecEnv('Hover3D', n, dtype=dtype, seed=seed, track_stats=True)
    orc = EnvBatch('Hover3D', n, seed=seed)
    pid = HoverHeuristicBatch(n, scale=scale)
    env.reset()
    o_obs = orc.reset()
    sync = np.ones(n, bool)
    worst_a = worst_s = 0.0
    for chunk in range(T // 50):
        out = env.rollout(50, source='pid_hover', scale=scale, record_actions=True, record_dones=True)
        acts, dones = out['actions'].cpu().numpy(), out['dones'].cpu().numpy()
        for t in range(50):
            a = pid.act(o_obs)
            worst_a = max(worst_a, float((np.abs(acts[t] - a) / np.maximum(np.abs(a), 1e-2))[sync].max()))
            o_obs, o_r, o_done, _ = orc.step(a)
            sync &= dones[t] == o_done
        sync &= env.status.cpu().numpy() == orc.dyn.status
        worst_s = max(worst_s, merr(env.state.cpu().numpy()[sync], orc.dyn.x[sync]))
        if chunk == 15:              # step 800 of the first episode: holding the set-point
            z = env.state.cpu().numpy()[:, 4]
            assert np.abs(z + 5.0).max() < 0.1, (z.min(), z.max())
    assert env.controller.shape == (n, 24)
    assert sync.sum() >= (n if dtype == torch.float64 else 0.97 * n), sync.sum()
    assert worst_s <= tol and worst_a <= (1e-5 if dtype == torch.float64 else 2e-3), (worst_s, worst_a)
    s = env.stats()
    assert s['episodes'] == n and s['timeout'] == n          # every first episode ran to the step limit
    with pytest.raises(pkg.CopterError):
        pkg.CopterVecEnv('Lander3D', 8).rollout(1, source='pid_hover')      # no yaw rate in that observation


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('variant,source,scale,offset,gains', [
    ('Lander2D', 'pid', 1e-3, 0.0159, {'descent_kd': 3.0}), ('Lander1D', 'pid', 1e-3, 0.0159, {'descent_kd': 3.0}),
    ('Hover2D', 'pid_hover', 0.016560178212092172, 0.016560178212092172, {}),
    ('Hover1D', 'pid_hover', 0.016560178212092172, 0.016560178212092172, {})])
def test_planar_heuristics_rollout_vs_oracle(pkg, variant, source, scale, offset, gains, dtype):
    """The 2-D / 1-D heuristic demos (attic/heuristic/lander2d.py, lander1d.py, hover2d.py,
    hover1d.py) as on-device action sources, closed around their envs, against the two oracles.
    Offsets / scales map the demand onto the live vehicle's hover command (no (t+1)/2 in these
    demos); the landers touch down softly, the hovers run to the step limit.
    Tolerances as in the 3-D closed-loop tests (float32 observation quantiser in the loop)."""
    from oracle.pid_oracle import PlanarHeuristicBatch
    n, T, seed = 512, 1100, 9
    kind, dims = ('lander' if source == 'pid' else 'hover'), int(variant[-2])
    env = pkg.CopterVecEnv(variant, n, dtype=dtype, seed=seed, track_stats=True)
    orc = EnvBatch(variant, n, seed=seed)
    pid = PlanarHeuristicBatch(n, kind, dims, scale=scale, offset=offset, **gains)
    env.reset()
    o_obs = orc.reset()
    sync = np.ones(n, bool)
    worst_a = worst_s = 0.0
    for chunk in range(T // 50):
        out = env.rollout(50, source=source, scale=scale, offset=offset, pid_gains=gains, record_actions=True, record_dones=True)
        acts, dones = out['actions'].cpu().numpy(), out['dones'].cpu().numpy()
        for t in range(50):
            a = pid.act(o_obs)
            worst_a = max(worst_a, float((np.abs(acts[t] - a) / np.maximum(np.abs(a), 1e-2))[sync].max()))
            o_obs, o_r, o_done, _ = orc.step(a)
            sync &= dones[t] == o_done
        sync &= env.status.cpu().numpy() == orc.dyn.status
        worst_s = max(worst_s, merr(env.state.cpu().numpy()[sync], orc.dyn.x[sync]))
    assert sync.sum() >= (n if dtype == torch.float64 else 0.97 * n), sync.sum()
    assert worst_s <= (5e-6 if dtype == torch.float64 else 1e-4) and worst_a <= (1e-5 if dtype == torch.float64 else 2e-3), (worst_s, worst_a)
    s = env.stats()
    assert s['episodes'] >= n
    if kind == 'lander':          # soft touch-downs; the axes these demos do not control drift, so only some are on target
        assert s['landed'] > 0.9 * s['episodes'] and 0 < s['bonus'] < s['episodes']
    else:
        assert s['timeout'] == s['episodes']


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


@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('variant', ['Lander3D', 'Lander2D', 'Hover3D', 'Lander1D', 'Takeoff'])
def test_fused_mlp_policy_vs_torch_fp32(pkg, variant, kernel, policy_kernel_choice):
    """The hand-written policy kernels -- tcgen05.mma with TMEM accumulators (kernel '1', the default) and
    warp-level mma.sync (kernel '0') -- against the plain PyTorch fp32 evaluation of the same network on
    the same observations (bf16 inputs / weights / activations, fp32 accumulation, MUFU tanh; the
    tcgen05 kernel evaluates a quarter of the hidden tanh as a polynomial on the FMA pipe).
    Tolerance: bf16 rounding of inputs, weights and two layers of activations (2^-9 relative
    each) plus tanh.approx (2^-11) on outputs in [-1, 1]."""
    policy_kernel_choice(kernel)
    n = 4099 if kernel == '0' else 4099 + 128 * 1500         # the tcgen05 kernel: more tiles (1533) than resident CTAs (148 x 7), so tiles are taken over by cluster launch control; ragged tail
    env = pkg.CopterVecEnv(variant, n, seed=3)
    env.reset()
    g = torch.Generator(device='cuda').manual_seed(0)
    for t in range(30):          # spread the states out
        env.step(0.0166 * (1 + 0.3 * torch.randn((n, env.action_size), device='cuda', generator=g)))
    pol = pkg.mlp_policy(env.obs_size, env.action_size, dtype=torch.float32, seed=5)
    for p in pol.net.parameters():
        p.data.mul_(3.0)         # push the activations into the curved part of tanh
    fused = pkg.FusedMLPPolicy(env, pol.net, out_scale=0.5, out_offset=0.25)
    got = fused()
    with torch.no_grad():
        ref = 0.25 + 0.5 * pol.net(env.obs)
    err = (got - ref).abs()
    assert got.shape == (n, env.action_size)
    assert err.max().item() <= 2e-2 and err.mean().item() <= 3e-3, (err.max().item(), err.mean().item())
    assert ref.std().item() > 0.01       # the comparison is not vacuous
    if kernel == '1':                    # and the two kernels agree with each other more closely than either with fp32
        policy_kernel_choice('0')
        other = pkg.FusedMLPPolicy(env, pol.net, out_scale=0.5, out_offset=0.25)()
        policy_kernel_choice('1')
        assert (got - other).abs().max().item() <= 1.5e-2 and (got - other).abs().mean().item() <= 1e-3
    # in the loop: same trajectories as the torch policy up to the policy's own rounding
    ro = pkg.PolicyRollout(env, fused, 4, planar=True, use_cuda_graph=True)
    r, d, _ = ro.run()
    assert r.shape == (4, n) and torch.isfinite(r).all()


@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('variant,n', [('Lander3D', 4099), ('Lander2D', 1000), ('Hover3D', 257), ('Lander1D', 31), ('Takeoff', 129),
                                       ('Hover2D', 517), ('Hover1D', 33), ('Lander3D', 128 * 148 * 8 + 77)])
def test_fused_policy_rollout_equals_policy_kernel_plus_step(pkg, variant, n, kernel, policy_kernel_choice):
    """copter_policy_rollout_f32 (policy + env step for T steps in one launch, state in
    registers) against the same network evaluated by copter_policy_mlp_f32 and stepped by
    copter_step_f32, launch by launch: done flags, recorded actions / observations, final state
    and counters are bit-identical, rewards agree to a few ulp (ragged n covers partly filled warps
    and tiles; the last size holds more tiles than the tcgen05 kernel has resident CTAs (148 x 6), so its CTAs take
    further tiles over by cluster launch control).
    Both implementations of the network exist fused and standalone -- '1': tcgen05 / TMEM
    (copter_policy_rollout_tc_kernel vs copter_mlp_policy_tc_kernel), '0': warp-level MMAs -- and each
    fused kernel is pinned to the standalone kernel of its own kind (the two kinds round differently:
    hi + lo bf16 biases and a quarter of the tanh as polynomials in the tcgen05 kernels)."""
    policy_kernel_choice(kernel)
    T = 150 if n < 10000 else 40
    kw = dict(initial_altitude=0.0, initial_random_force=0.0, max_steps=60) if variant == 'Takeoff' else {}
    envs = [pkg.CopterVecEnv(variant, n, seed=11, track_returns=True, **kw) for _ in range(2)]
    pol = pkg.mlp_policy(envs[0].obs_size, envs[0].action_size, dtype=torch.float32, seed=2)
    for p in pol.net.parameters():
        p.data.mul_(2.0)
    # commands around hover so that episodes end inside the horizon in several ways
    scale, offset = 0.03, 0.0166
    for e in envs:
        e.reset()
    fused = pkg.FusedPolicyRollout(envs[0], pol.net, T, out_scale=scale, out_offset=offset, store_obs=True, store_actions=True)
    r1, d1, last1 = fused.run()
    two = pkg.FusedMLPPolicy(envs[1], pol.net, out_scale=scale, out_offset=offset)
    rewards, dones, actions, obs = [], [], [], []
    for t in range(T):
        obs.append(envs[1].obs.clone())
        a = two()
        actions.append(a.clone())
        o, r, d, _, _ = envs[1].step(a)
        rewards.append(r.clone()); dones.append(d.clone())
    assert torch.equal(torch.stack(actions), fused.actions)
    assert torch.equal(torch.stack(obs), fused.obs)
    # same device arithmetic, but the compiler may contract the reward's FMAs differently in the
    # two kernels: rewards at a few ulp; everything that feeds back into the loop bit for bit
    assert merr(r1.cpu().numpy(), torch.stack(rewards).cpu().numpy()) <= 1e-5
    assert torch.equal(torch.stack(dones), d1)
    assert torch.equal(envs[0].state, envs[1].state) and torch.equal(envs[0].meta, envs[1].meta)
    assert torch.equal(last1, envs[1].obs)
    s0, s1 = envs[0].stats(), envs[1].stats()
    assert s0['episodes'] == s1['episodes'] and s0['env_steps'] == s1['env_steps'] == n * T
    assert abs(s0['return_sum'] - s1['return_sum']) <= 1e-6 * max(1.0, abs(s1['return_sum']))
    if variant in ('Lander3D', 'Lander2D') and T >= 150:      # the variants that can tip over inside the horizon
        assert d1.any() and not d1.all()
    # a second horizon continues from where the first one stopped
    r2, _, _ = fused.run()
    assert torch.isfinite(r2).all()


def test_fused_policy_rollout_argument_errors(pkg):
    env = pkg.CopterVecEnv('Lander3D', 64)
    bad = torch.nn.Sequential(torch.nn.Linear(10, 32), torch.nn.Tanh(), torch.nn.Linear(32, 32), torch.nn.Tanh(),
                              torch.nn.Linear(32, 4), torch.nn.Tanh()).cuda()
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(env, bad, 4)
    good = pkg.mlp_policy(10, 4, dtype=torch.float32).net
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(env, good, 4).run()          # not reset
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(pkg.CopterVecEnv('Lander3D', 64, k_substeps=2), good, 4)


@pytest.mark.parametrize('kernel', ['1', '0'])
def test_fused_policy_rollout_exploration_noise(pkg, kernel, policy_kernel_choice):
    """action_std: the sampled command is policy(obs) + std * xi with xi the documented Philox
    stream (counter (env, step, 2), Box-Muller) -- checked against the oracle's restatement of
    the stream and the policy kernel's own output on the recorded observations (the standalone
    kernel of the same kind as the fused one: '1' tcgen05 / TMEM, '0' warp-MMA); the trajectory
    equals stepping the recorded commands; cutting the horizon differently changes nothing."""
    policy_kernel_choice(kernel)
    n, T, seed, off = 1031, 24, 0xABCDEF0123, 5000
    mk = lambda: pkg.CopterVecEnv('Lander3D', n, seed=seed, env_offset=off)          # noqa: E731
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=9)
    std = torch.tensor([0.004, 0.002, 0.001, 0.003], device='cuda')
    a_env, b_env, c_env = mk(), mk(), mk()
    for e in (a_env, b_env, c_env):
        e.reset()
    a_env.rollout_step = b_env.rollout_step = 2 ** 32 + 7
    ro = pkg.FusedPolicyRollout(a_env, pol.net, T, out_scale=0.01, out_offset=0.0166, store_obs=True, store_actions=True, action_std=std)
    r, d, _ = ro.run()
    ids = np.arange(n, dtype=np.uint64) + np.uint64(off)
    mean_k = pkg.FusedMLPPolicy(c_env, pol.net, out_scale=0.01, out_offset=0.0166)
    s32 = std.cpu().numpy()
    for t in range(T):
        xi, rad = noise_oracle.gaussian_variates(seed, ids, 2 ** 32 + 7 + t, 2)
        st = torch.zeros((n, 12), device='cuda')
        st[:, :10] = ro.obs[t]
        c_env.set_state(st)
        mean = mean_k().clone()
        a32 = ro.actions[t].cpu().numpy()
        got = (a32.astype(np.float64) - mean.cpu().numpy()) / s32
        # the action is fmaf(std, xi, mean): half an ulp of it over std, plus the device variate's own error
        bound = noise_oracle.SLACK * (np.spacing(np.abs(a32)) / (2.0 * s32) + noise_oracle.pair_bound(rad, 4))
        assert np.all(np.abs(got - xi) <= bound), (t, float(np.max(np.abs(got - xi) / bound)))
        # replay of the recorded commands through the step kernel
        o, r2, d2, _, _ = b_env.step(ro.actions[t])
        assert torch.equal(d2, d[t]) and merr(r[t].cpu().numpy(), r2.cpu().numpy()) <= 1e-5
    assert torch.equal(a_env.state, b_env.state) and torch.equal(a_env.meta, b_env.meta)
    z = ((ro.actions - 0.0166).cpu().numpy())
    assert 0.5 * 0.001 < z[..., 2].std() < 0.02          # noise present, of the configured scale
    # same rollout cut into horizons of 5, 7 and 12 steps
    e2 = mk(); e2.reset(); e2.rollout_step = 2 ** 32 + 7
    for h in (5, 7, 12):
        pkg.FusedPolicyRollout(e2, pol.net, h, out_scale=0.01, out_offset=0.0166, action_std=std).run()
    assert torch.equal(e2.state, a_env.state) and torch.equal(e2.meta, a_env.meta) and e2.rollout_step == a_env.rollout_step
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(a_env, pol.net, 4, action_std=torch.ones(3, device='cuda'))
