"""CPU: the kernels' arithmetic (gym_copter_b200/csrc/copter_core.h, instantiated on the host) against the
reference-pinned numpy oracle at vehicle, world and task parameters away from the defaults (oracle/param_sets.py).

At the default DJI Phantom parameters Ix == Iy, the live model has no gyroscopic coupling and fps = 100, so a
header that divides the roll torque by Iy, swaps the two gyroscopic factors, drops the yaw Euler term or takes
dt from a hard-coded 100 computes the same bits as the right one, and every test at default parameters passes.
Here every variant x K in {1, 3, 16} x auto-reset on / off runs at every set: state and reward <= 1e-9, flags,
counters, causes, executed substeps and episode lengths exact, the statistics ledger's counts exact -- and each
run shows that it did what its set is for.  Then modified copies of the header, each with one such error, are
built and shown to fail at their set; those that compute the default constants unchanged are shown to pass at
the defaults, which is the blind spot this file closes.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle.copter_oracle import ALL_VARIANTS, EnvBatch, OracleParams
from oracle.host_restatement import CAUSE_STATS, HostEnvBatch
from oracle.param_sets import CASES, ENDINGS, SETS, hover_command, premises

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-9
DISCRETE = ('done', 'status', 'steps', 'episode', 'cause', 'executed', 'final_steps')


def streams(rng, n, t, a, hover, takeoff=False, saturating=True):
    """[t, n, a] float32 commands, four kinds interleaved over the envs: a constant per env between 0.6 and 1 of
    hover (descents that land gently or crash), hover with 10 % Gaussian and 20 % uniform noise, and U(-1, 1)
    (`saturating`; angle and bounds endings) or hover with 60 % uniform noise.  Takeoff (no angle limit: the
    Euler equations of an asymmetric vehicle blow up under saturating commands) gets hover x U(0.9, 1.2), with
    every fifth env's signs flipped (its commands are not clipped)."""
    act = np.empty((t, n, a))
    for i in range(4):
        m = len(range(i, n, 4))
        if takeoff:
            x = hover * rng.uniform(0.9, 1.2, (t, m, a))
        elif i == 0:
            x = np.broadcast_to(hover * rng.uniform(0.6, 1.0, (1, m, 1)), (t, m, a))
        elif i == 1:
            x = hover * (1 + 0.1 * rng.standard_normal((t, m, a)))
        elif i == 2:
            x = hover * (1 + 0.2 * rng.uniform(-1, 1, (t, m, a)))
        else:
            x = rng.uniform(-1, 1, (t, m, a)) if saturating else hover * (1 + 0.6 * rng.uniform(-1, 1, (t, m, a)))
        act[:, i::4] = x
    if takeoff:
        act[:, ::5] *= -1
    return act.astype(np.float32)


def compare(variant, params, k, auto_reset, lib=None, n=64, steps=384, seed=0):
    """The fp64 host instantiation (`lib`: another build of it) and the oracle on the same commands.  Returns the
    first discrete mismatch (name, launch) or None, the worst state / reward errors, both ledgers and what the
    run covered."""
    rng = np.random.default_rng(seed + 7 * k + sum(map(ord, variant)))
    A = ALL_VARIANTS[variant][2]
    T = steps // k
    act = streams(rng, n, T, A, hover_command(params), variant == 'Takeoff', auto_reset).astype(np.float64)
    h = HostEnvBatch(variant, n, params, dtype=np.float64, seed=11, env_offset=5 << 32, auto_reset=auto_reset,
                     track_returns=True, lib=lib)
    o = EnvBatch(variant, n, params, seed=11, env_offset=5 << 32, auto_reset=auto_reset)
    h.reset(); o.reset()
    out = dict(mismatch=None, state=0.0, reward=0.0, mid_angle=0, airborne=0)
    want = dict.fromkeys(('episodes', 'length_sum', 'env_steps') + tuple(c for c, _ in CAUSE_STATS), 0)
    for t in range(T):
        _, r, d, info = h.step(act[t], k)
        _, o_r, o_d, o_info = o.step(act[t], k)
        pairs = dict(done=(d, o_d), status=(h.status, o.dyn.status), steps=(h.steps, o.steps),
                     episode=(h.episode, o.episode), cause=(info['cause'], o_info['cause']),
                     executed=(info['executed'], o_info['steps_taken']),
                     final_steps=(info['final_steps'][o_d], o_info['final_steps'][o_d]))
        bad = [name for name in DISCRETE if not np.array_equal(*pairs[name])]
        if bad:
            out['mismatch'] = (bad[0], t)
            break
        x = o.dyn.x
        out['state'] = max(out['state'], float(np.max(np.abs(h.x - x) / np.maximum(np.abs(x), 1))))
        out['reward'] = max(out['reward'], float(np.max(np.abs(r - o_r) / np.maximum(np.abs(o_r), 1))))
        want['episodes'] += int(o_d.sum())
        want['length_sum'] += int((o_info['final_steps'][o_d] - 1).sum())
        want['env_steps'] += int(o_info['steps_taken'].sum())
        for name, bit in CAUSE_STATS:
            want[name] += int(((o_info['cause'][o_d] & bit) != 0).sum())
        ang = np.maximum(np.abs(x[:, 6]), np.abs(x[:, 8]))
        out['mid_angle'] += int((~o_d & (ang > np.pi / 4) & (ang < np.radians(params.max_angle_deg))).sum())
        out['airborne'] += int(((o.dyn.status == 3) & (x[:, 4] < -0.05)).sum())
    out['ledger'], out['want'] = h.stats(), {k_: float(v) for k_, v in want.items()}
    return out


def failed(out):
    """The run told the header from the oracle: a discrete mismatch, or a continuous error 10x the bound."""
    return out['mismatch'] is not None or max(out['state'], out['reward']) >= 10 * TOL


@pytest.mark.parametrize('name', list(SETS))
def test_parameter_sets_keep_their_premises(name):
    """Each set still tells roll, pitch and yaw apart, runs another frame rate and sits on the branch of
    calm_angle it is for (premises() raises otherwise); the defaults do not."""
    k = premises(name)
    assert k['kR'] != k['kP'] and k['gpsi'] != 0
    with pytest.raises(AssertionError):
        premises(name, OracleParams())


@pytest.mark.parametrize('auto_reset', [True, False], ids=['auto', 'noreset'])
@pytest.mark.parametrize('k', [1, 3, 16])
@pytest.mark.parametrize('name,variant', CASES, ids=['%s-%s' % c for c in CASES])
def test_fp64_instantiation_matches_the_oracle_at_the_parameter_set(name, variant, k, auto_reset):
    p = SETS[name]
    out = compare(variant, p, k, auto_reset)
    assert out['mismatch'] is None, out['mismatch']
    assert out['state'] <= TOL and out['reward'] <= TOL, (out['state'], out['reward'])
    s = out['ledger']
    assert {c: s[c] for c in out['want']} == out['want'], (s, out['want'])
    assert s['episodes'] >= 64 and s['timeout'] > 0
    if variant == 'Takeoff':
        assert out['airborne'] > 0                                # vehicles did leave the ground
        return
    # what the set is for: episodes end in at least two ways; at the asymmetric set's own landing limits Lander
    # envs both land and crash; above the polynomial range (60 degrees) envs fly on with roll or pitch past pi/4
    assert sum(s[c] > 0 for c, _ in CAUSE_STATS) >= 2, s
    if name == 'asymmetric' and variant.startswith('Lander'):
        assert s['landed'] > 0 and s['crashed'] > 0, s
    if name == 'asymmetric' and not variant.endswith('1D') and auto_reset and k < 16:
        assert out['mid_angle'] > 0


# modified copies of copter_core.h: (set the error shows at, variant, substitutions); every one except the landing
# limits computes the default parameters' constants unchanged
MUTANTS = {
    'kR-kP-inertia-swapped': ('asymmetric', 'Hover3D', [('k.kR = arm * b * w * w / p.Ix;', 'k.kR = arm * b * w * w / p.Iy;'),
                                                          ('k.kP = arm * b * w * w / p.Iy;', 'k.kP = arm * b * w * w / p.Ix;')]),
    'jx-jy-swapped': ('gyro', 'Hover3D', [('k.jx = (T)(p.Jr / p.Ix); k.jy = (T)(p.Jr / p.Iy);',
                                           'k.jx = (T)(p.Jr / p.Iy); k.jy = (T)(p.Jr / p.Ix);')]),
    'gpsi-zero': ('asymmetric', 'Hover3D', [('k.gpsi = (T)((p.Ix - p.Iy) / p.Iz);', 'k.gpsi = (T)0;')]),
    'lvx-lvy-swapped': ('asymmetric', 'Lander3D', [('k.lvx = (T)p.landing_vel_x; k.lvy = (T)p.landing_vel_y;',
                                                    'k.lvx = (T)p.landing_vel_y; k.lvy = (T)p.landing_vel_x;')]),
    'kOm-ignored': ('gyro', 'Hover3D', [('k.kOm = (p.dynamics_model & COPTER_MODEL_GYRO) ? w : 0.0;', 'k.kOm = 0.0;')]),
    'lift-torque-arm': ('mars-lift', 'Hover3D', [('const double arm = lift ? 1.0 : p.L;', 'const double arm = p.L;')]),
    'dt-from-100': ('asymmetric', 'Hover1D', [('k.dt = (T)((T)1 / (T)p.fps);', 'k.dt = (T)((T)1 / (T)100);')]),
}
VISIBLE_AT_DEFAULTS = {'lvx-lvy-swapped'}


@pytest.fixture(scope='module')
def mutant_libs(tmp_path_factory):
    """Each mutant's host instantiation, built from a copy of the sources with oracle/Makefile's own recipe."""
    core = open(os.path.join(ROOT, 'gym_copter_b200', 'csrc', 'copter_core.h')).read()
    jobs = {}
    for m, (_, _, subs) in MUTANTS.items():
        top = tmp_path_factory.mktemp(m)
        for rel in ('oracle/Makefile', 'oracle/copter_host.cpp', 'include/copter_b200.h'):
            os.makedirs(top / os.path.dirname(rel), exist_ok=True)
            shutil.copy(os.path.join(ROOT, rel), top / rel)
        src = core
        for old, new in subs:
            assert src.count(old) == 1, (m, old)
            src = src.replace(old, new)
        os.makedirs(top / 'gym_copter_b200' / 'csrc')
        (top / 'gym_copter_b200' / 'csrc' / 'copter_core.h').write_text(src)
        jobs[m] = (str(top / 'oracle' / 'libcopter_host.so'),
                   subprocess.Popen(['make', '-s', '-C', str(top / 'oracle'), 'libcopter_host.so']))
    for m, (_, proc) in jobs.items():
        assert proc.wait() == 0, m
    return {m: lib for m, (lib, _) in jobs.items()}


@pytest.mark.parametrize('mutant', list(MUTANTS))
def test_a_modified_header_fails_at_its_parameter_set(mutant, mutant_libs):
    name, variant, _ = MUTANTS[mutant]
    lib = mutant_libs[mutant]
    bad = compare(variant, SETS[name], 3, True, lib=lib)
    assert failed(bad), (mutant, bad['mismatch'], bad['state'], bad['reward'])
    assert not failed(compare(variant, SETS[name], 3, True))         # the real header passes the same run
    # at the default parameters the mutant computes the same constants: nothing at defaults can see it
    at_defaults = compare(variant, OracleParams(**ENDINGS), 3, True, lib=lib)
    if mutant in VISIBLE_AT_DEFAULTS:
        assert failed(at_defaults)
    else:
        assert not failed(at_defaults), (at_defaults['mismatch'], at_defaults['state'], at_defaults['reward'])
