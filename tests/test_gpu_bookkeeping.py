"""
GPU: the edges of the counter fields, on every kernel that keeps them -- the step kernel at K = 1 and K = 16,
the rollout kernel in fp32 and fp64, and both fused policy rollouts (tcgen05 / TMEM and warp-MMA).

The packed meta word holds an 11-bit step counter that saturates at 2047 and a 19-bit episode index that
wraps at 2^19; the wide layout holds a 30-bit counter (cap 2^30 - 1) and a 32-bit index in meta_hi.  Each
edge starts the envs next to a limit by writing the counters directly and checks two things after every
launch: equality with the host instantiation of copter_core.h (state bits, counters, flags and the
statistics' counts), and the values the edge must produce, written out here -- copter_core.h is shared with
the host, so a host comparison alone cannot see an error that lives there.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.host_restatement import STAT_NAMES, HostEnvBatch     # noqa: E402
from oracle.copter_oracle import OracleParams                    # noqa: E402

HOVER = 0.016560178212092172
TIMEOUT, OOB, AIRBORNE = 32, 4, 3
COUNTS = tuple(k for k in STAT_NAMES if k != 'return_sum')
PATHS = ['step-k1', 'step-k16', 'rollout-f32', 'rollout-f64', 'policy-tc', 'policy-mma']
N, SEED, OFF, H = 300, 41, 9 << 32, 16          # N: nine full warps and a partial one; H: steps per rollout launch


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


class Path:
    """One env on one kernel path, with its host twin.  launch() runs one launch (one step() of K substeps, or
    one rollout of H steps under the hover command), replays its commands on the host and checks the two
    against each other; it returns the launch's done flags and causes, [steps, N]."""

    def __init__(self, pkg, path, monkeypatch, wide=False, auto_reset=True, horizon=H, **params):
        self.path, self.horizon = path, horizon
        self.dtype = np.float64 if path == 'rollout-f64' else np.float32
        self.k = 16 if path == 'step-k16' else 1
        if path.startswith('policy'):
            monkeypatch.setenv('COPTER_B200_POLICY_ROLLOUT_TC', '1' if path == 'policy-tc' else '0')
        self.env = pkg.CopterVecEnv('Lander3D', N, dtype=torch.float64 if self.dtype == np.float64 else torch.float32,
                                    seed=SEED, env_offset=OFF, k_substeps=self.k, auto_reset=auto_reset,
                                    wide_counters=wide, track_returns=True, report_cause=True, **params)
        self.host = HostEnvBatch('Lander3D', N, OracleParams(**params), dtype=self.dtype, seed=SEED, env_offset=OFF,
                                 auto_reset=auto_reset, wide=wide, track_returns=True)
        self.env.reset(); self.host.reset()
        self.pro = None
        if path.startswith('policy'):          # a network whose every action is the hover command
            pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=1)
            self.pro = pkg.FusedPolicyRollout(self.env, pol.net, horizon, out_scale=0.0, out_offset=HOVER,
                                              store_actions=True, store_causes=True)

    def start(self, state, steps, episode, status=AIRBORNE):
        """Every env at `state` with the given counters, on the device and on the host."""
        env, host = self.env, self.host
        env.set_state(np.broadcast_to(state, (N, 12)), status=status, steps=steps)
        if env.wide:
            env.meta_hi.fill_(np.int64(episode).astype(np.uint32).astype(np.int32).item())
        else:
            m = (status | (steps << 2) | (episode << 13)) & 0xFFFFFFFF
            env.meta.fill_(m - (1 << 32) if m >= 1 << 31 else m)
        host.x[:] = np.asarray(state, self.dtype)
        host.status[:], host.steps[:], host.episode[:] = status, steps, episode
        assert (env.steps.cpu().numpy() == steps).all() and (env.episodes.cpu().numpy() == episode).all()
        assert (env.status.cpu().numpy() == status).all()

    def launch(self):
        env, host = self.env, self.host
        if self.path.startswith('step'):
            a = torch.full((N, 4), HOVER, dtype=env.dtype, device=env.device)
            _, _, term, _, info = env.step(a)
            acts, dones, causes = a[None], term[None], info['cause'][None]
        elif self.path.startswith('rollout'):
            out = env.rollout(self.horizon, source='const', offset=HOVER, record_actions=True, record_dones=True, record_causes=True)
            acts, dones, causes = out['actions'], out['dones'], out['causes']
        else:
            _, dones, _ = self.pro.run()
            acts, causes = self.pro.actions, self.pro.causes
        acts, dones, causes = acts.cpu().numpy(), dones.cpu().numpy(), causes.cpu().numpy()
        for t in range(len(acts)):
            _, _, h_done, h_info = host.step(acts[t], self.k)
            assert np.array_equal(dones[t], h_done) and np.array_equal(causes[t], h_info['cause']), t
        x = env.state.cpu().numpy()
        if self.dtype == np.float32:
            assert np.array_equal(bits(x), bits(host.x))
        else:
            assert float(np.max(np.abs(x - host.x) / np.maximum(np.abs(host.x), 1))) <= 1e-9
        assert np.array_equal(env.steps.cpu().numpy(), host.steps) and np.array_equal(env.status.cpu().numpy(), host.status)
        assert np.array_equal(env.episodes.cpu().numpy(), host.episode.astype(np.int64))
        s, h = env.stats(), host.stats()
        assert {k: s[k] for k in COUNTS} == {k: h[k] for k in COUNTS}, (s, h)
        return dones, causes

    def steps_per_launch(self):
        return self.k if self.path.startswith('step') else self.horizon


HOVER_STATE = np.array([0, 0, 0, 0, -5.0, 0, 0, 0, 0, 0, 0, 0])


@pytest.mark.parametrize('wide', [False, True], ids=['compact', 'wide'])
@pytest.mark.parametrize('path', PATHS)
def test_step_counter_saturates_at_its_cap(pkg, path, wide, monkeypatch):
    """No auto-reset, hovering AIRBORNE envs six steps short of the largest step limit of the layout: exactly one
    TIMEOUT ending, at step max_steps (length max_steps), then the counter stays at the cap on every later launch
    -- through the K = 16 calm streak too, which counts past the cap and clamps afterwards.  Status and episode
    index are untouched."""
    max_steps = 0x3FFFFFFE if wide else 2046
    cap, episode = max_steps + 1, (0xA5A5A5A5 if wide else 0x5A5A5)
    p = Path(pkg, path, monkeypatch, wide=wide, auto_reset=False, max_steps=max_steps)
    p.start(HOVER_STATE, max_steps - 6, episode)
    n_launch = 3 if p.steps_per_launch() > 1 else 12
    endings, executed = np.zeros(N, np.int64), 0
    for j in range(n_launch):
        dones, causes = p.launch()
        endings += dones.sum(0)
        assert set(np.unique(causes)) <= {0, TIMEOUT}
        if p.path == 'step-k16':               # the ending is the 7th substep; the env idles for the rest
            executed += 7 if j == 0 else 16
        else:
            executed += p.steps_per_launch()
        done_at = 6 - j * p.steps_per_launch()          # row of the ending within this launch, if it is in it
        if p.k == 1 and 0 <= done_at < len(dones):
            assert dones[done_at].all() and (causes[done_at] == TIMEOUT).all()
        steps = p.env.steps.cpu().numpy()
        assert (steps == min(max_steps - 6 + executed, cap)).all(), (j, np.unique(steps))
        assert (p.env.status.cpu().numpy() == AIRBORNE).all() and (p.env.episodes.cpu().numpy() == episode).all()
    assert (endings == 1).all()
    s = p.env.stats()
    assert s['episodes'] == N and s['timeout'] == N and s['length_sum'] == N * max_steps
    assert s['landed'] == s['bonus'] == s['oob'] == s['angle'] == s['crashed'] == 0
    assert s['env_steps'] == N * executed


@pytest.mark.parametrize('wide', [False, True], ids=['compact', 'wide'])
@pytest.mark.parametrize('path', PATHS)
def test_episode_index_wraps_to_zero(pkg, path, wide, monkeypatch):
    """Envs at the last episode index of the layout, out of bounds: the first step ends every episode, the index
    wraps to 0, and the next episode -- in the same launch on the rollout paths, where the index lives in a
    register -- runs exactly as episode 0 of a freshly reset env: the same Philox reset force."""
    last = 0xFFFFFFFF if wide else (1 << 19) - 1
    kw = dict(bounds=2.0)
    p = Path(pkg, path, monkeypatch, wide=wide, **kw)
    p.start(np.array([3.0, 0, 0, 0, -5.0, 0, 0, 0, 0, 0, 0, 0]), 5, last)
    dones, causes = p.launch()
    assert dones[0].all() and (causes[0] & OOB).all()
    assert (p.env.episodes.cpu().numpy() == 0).all()
    fresh = Path(pkg, path, monkeypatch, wide=wide, horizon=max(H - 1, 1), **kw)
    if p.k == 1 and not path.startswith('step'):
        fresh.launch()                              # the rest of the launch: H - 1 steps of episode 0
    else:
        p.launch(); fresh.launch()                 # the next launch: the first step(s) of episode 0
    assert np.array_equal(bits(p.env.state.cpu().numpy()), bits(fresh.env.state.cpu().numpy()))
    assert torch.equal(p.env.meta, fresh.env.meta) and (p.env.episodes.cpu().numpy() == 0).all()
    assert p.env.stats()['episodes'] == N + fresh.env.stats()['episodes']


@pytest.mark.parametrize('wide', [False, True], ids=['compact', 'wide'])
@pytest.mark.parametrize('dtype', ['f32', 'f64'])
def test_reset_keeping_the_episode_wraps_to_zero(pkg, wide, dtype, monkeypatch):
    """reset() after the first one moves every env to its next episode index: from the last index to 0, whose
    first step then draws the reset force of episode 0, as a freshly reset env does."""
    path = 'step-k1' if dtype == 'f32' else 'rollout-f64'
    last = 0xFFFFFFFF if wide else (1 << 19) - 1
    p = Path(pkg, path, monkeypatch, wide=wide)
    p.start(HOVER_STATE, 9, last)
    p.env.reset(); p.host.reset()
    assert (p.env.episodes.cpu().numpy() == 0).all() and (p.host.episode == 0).all()
    assert (p.env.steps.cpu().numpy() == 1).all() and not p.env.ep_return.cpu().numpy().any()
    fresh = Path(pkg, path, monkeypatch, wide=wide)
    p.launch(); fresh.launch()
    assert np.array_equal(bits(p.env.state.cpu().numpy()), bits(fresh.env.state.cpu().numpy()))
    assert torch.equal(p.env.meta, fresh.env.meta)


@pytest.mark.parametrize('path', PATHS)
def test_step_limit_of_one(pkg, path, monkeypatch):
    """max_steps = 1: every step is a TIMEOUT ending of length 1; a K = 16 launch executes one substep per env
    and credits N env-steps."""
    p = Path(pkg, path, monkeypatch, max_steps=1)
    rows = 0
    for j in range(3):
        dones, causes = p.launch()
        rows += len(dones)
        assert dones.all() and (causes == TIMEOUT).all(), j
        assert (p.env.steps.cpu().numpy() == 1).all() and (p.env.episodes.cpu().numpy() == rows).all()
    s = p.env.stats()
    assert s['episodes'] == s['timeout'] == s['length_sum'] == s['env_steps'] == N * rows
