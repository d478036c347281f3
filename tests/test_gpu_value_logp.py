"""The critic kernel (copter_value_mlp_f32 / FusedMLPValue), the log-probability kernel (copter_policy_logp_f32) and
FusedPolicyRollout's PPO batch (critic=..., store_log_probs=True):
  * values against oracle/value_oracle.py (the tcgen05 kernel's own rounding) within its ceiling on every shared case,
    and against a PyTorch fp32 critic relative to sum |W3| |h2| + |b3|;
  * launch edges, row layouts (packed, the env's stride-12 view, padded), untouched rows past m, selection;
  * log-probs against the float64 formula on the oracle's Philox restatement, against (action - mu) / std, and bit
    for bit across shard splits and horizon cuts;
  * every buffer of the rollout's PPO batch bit for bit against the standalone calls, advantages() == gae(), and the
    batch against a PyTorch fp32 critic + float64 GAE."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import value_oracle as vo                     # noqa: E402
from oracle import noise_oracle as no                     # noqa: E402

CASES = {c['name']: c for c in vo.critic_cases()}
SENTINEL = 0x7FC0DEAD


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    return gym_copter_b200


def make_critic(weights):
    W1 = weights[0]
    net = torch.nn.Sequential(torch.nn.Linear(W1.shape[1], 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                              torch.nn.Linear(64, 1))
    for p, w in zip(net.parameters(), weights):
        p.data = torch.from_numpy(np.ascontiguousarray(w, np.float32))
    return net.cuda()


def sentinel(shape):
    return torch.full(shape, SENTINEL, dtype=torch.int32, device='cuda').view(torch.float32)


def is_sentinel(x):
    return x.view(torch.int32) == SENTINEL


@pytest.mark.parametrize('name', list(CASES))
def test_value_kernel_vs_rounding_model(pkg, name):
    """Every row within the model's ceiling; the dense networks within REL_TO_NETWORK * scale of a PyTorch fp32
    critic (plus that critic's own fp32 error)."""
    c = CASES[name]
    net = make_critic(c['weights'])
    critic = pkg.FusedMLPValue(net, c['variant'])
    obs = torch.from_numpy(c['obs']).cuda()
    got = critic(obs).cpu().numpy().astype(np.float64)
    args = vo.case_args(c)
    ref, cei = vo.model(*args), vo.ceiling(*args)
    err = np.abs(got - ref)
    assert np.all(np.isfinite(got)) and np.all(err <= cei), (name, float(np.max(err / cei)))
    if not name.startswith('probe'):
        with torch.no_grad():
            t32 = net(obs)[:, 0].cpu().numpy().astype(np.float64)
        scale = vo.scale(*args)
        assert np.all(np.abs(got - t32) <= vo.REL_TO_NETWORK * scale + 2.0 ** -18 * scale), name


def _rows_in(layout, obs, first):
    """obs [m, O] as rows of the given layout: 'packed' (stride O), 'env' (the [m, 12] state rows, columns
    first .. first + O - 1) or 'padded' (stride O + 5)."""
    m, O = obs.shape
    if layout == 'packed':
        return obs.clone()
    width = 12 if layout == 'env' else O + 5
    off = first if layout == 'env' else 3
    big = torch.full((m, width), float('nan'), device='cuda')
    big[:, off:off + O] = obs
    return big[:, off:off + O]


@pytest.mark.parametrize('variant,first', [('Lander3D', 0), ('Lander2D', 2), ('Lander1D', 4), ('Hover3D', 0)])
def test_value_launch_edges_and_layouts(pkg, variant, first):
    """m in {1, 127, 128, 129} and more tiles than the resident CTAs hold (148 x 5 x 128 + 1, so cluster launch control
    hands tiles over inside the launch); packed, env-view and padded rows; an output of m + 200 rows prefilled with a
    sentinel keeps rows >= m.  Every value is the same bits on every layout and size."""
    from gym_copter_b200 import _lib
    O = {'Lander3D': 10, 'Lander2D': 6, 'Lander1D': 2, 'Hover3D': 12}[variant]
    big = 148 * 5 * 128 + 1
    rng = np.random.default_rng(3)
    obs = torch.from_numpy((rng.standard_normal((big, O)) * 2).astype(np.float32)).cuda()
    from oracle import policy_oracle as po
    W = po.dense_weights(variant, 3)
    W = W[:4] + (np.ascontiguousarray(W[4][:1]), np.ascontiguousarray(W[5][:1]))
    critic = pkg.FusedMLPValue(make_critic(W), variant)
    full = critic(obs)
    lib = _lib.load()
    for layout in ('packed', 'env', 'padded'):
        rows = _rows_in(layout, obs, first)
        for m in (1, 127, 128, 129, big):
            out = sentinel((m + 200,))
            r = rows[:m]
            rc = lib.copter_value_mlp_f32(r.data_ptr(), r.stride(0), m, _lib.VARIANT_IDS[variant], 64,
                                          *[p.data_ptr() for p in critic.params], None, 0, out.data_ptr(),
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
            torch.cuda.synchronize()
            assert torch.equal(out[:m], full[:m]), (layout, m)
            assert bool(is_sentinel(out[m:]).all()), (layout, m)
    ref = vo.model(obs.cpu().numpy(), variant, *W)
    assert np.all(np.abs(full.cpu().numpy() - ref) <= vo.ceiling(obs.cpu().numpy(), variant, *W))
    # [T, N, O] with a leading-dimension view, and a rows tensor whose leading dimensions do not flatten
    tn = obs[:128 * 6].view(6, 128, O)
    assert torch.equal(critic(tn), full[:128 * 6].view(6, 128))
    with pytest.raises(pkg.CopterError):
        critic(_rows_in('env', obs, first)[:128 * 6].view(6, 128, O).transpose(0, 1))
    with pytest.raises(pkg.CopterError):
        critic(obs[:, :O - 1] if O > 2 else obs[:, :1])


def test_value_selection(pkg):
    """Selected rows equal the unselected-mode values bit for bit; other rows, whole tiles without a selected row
    among them, keep their sentinel; a select byte counts only through the mask; an all-zero select writes nothing."""
    c = CASES['Hover3D_x3']
    critic = pkg.FusedMLPValue(make_critic(c['weights']), 'Hover3D')
    obs = torch.from_numpy(c['obs']).cuda()
    m = len(obs)
    full = critic(obs)
    rng = np.random.default_rng(5)
    sel = np.zeros(m, np.uint8)
    pick = rng.random(m) < 0.002                              # ~1/500 rows: most tiles have none
    sel[pick] = 32
    sel[rng.random(m) < 0.01] |= 4                            # bits outside the mask
    n_tiles = (m + 127) // 128
    empty = [k for k in range(n_tiles) if not pick[128 * k:128 * k + 128].any()]
    assert 0 < len(empty) < n_tiles
    select = torch.from_numpy(sel).cuda()
    out = sentinel((m,))
    critic(obs, select=select, mask=32, out=out)
    keep = torch.from_numpy(pick).cuda()
    assert torch.equal(out[keep], full[keep])
    assert bool(is_sentinel(out[~keep]).all())
    for k in empty[:50]:
        assert bool(is_sentinel(out[128 * k:128 * k + 128]).all())
    out = sentinel((m,))
    critic(obs, select=torch.zeros(m, dtype=torch.uint8, device='cuda'), out=out)
    assert bool(is_sentinel(out).all())
    out = sentinel((m,))
    critic(obs, select=torch.full((m,), 255, dtype=torch.uint8, device='cuda'), mask=1, out=out)
    assert torch.equal(out, full)


def test_log_probs_formula_and_cross_checks(pkg):
    """log_probs = -1/2 sum xi^2 - sum log std - A/2 log 2 pi on xi from the oracle's Philox restatement (float64);
    against (action - mu) / std with mu the standalone policy on the recorded observations; bit for bit across two
    shards of the envs and across horizons of 5 + 7 + 12 steps against one of 24."""
    from gym_copter_b200 import _lib
    n, T, seed, off = 1031, 24, 0xABCDEF0123, 5000
    mk = lambda o=off, k=n: pkg.CopterVecEnv('Lander3D', k, seed=seed, env_offset=o)      # noqa: E731
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=9)
    std = torch.tensor([0.004, 0.002, 0.001, 0.003], device='cuda')
    env = mk()
    env.reset()
    env.rollout_step = 2 ** 32 + 7
    ro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=0.01, out_offset=0.0166, store_obs=True, store_actions=True,
                                action_std=std, store_log_probs=True)
    ro.run()
    lp = ro.log_probs.cpu().numpy().astype(np.float64)
    ids = np.arange(n, dtype=np.uint64) + np.uint64(off)
    s64 = std.cpu().numpy().astype(np.float64)
    c = -np.log(s64).sum() - 2.0 * np.log(2 * np.pi)
    c_env = mk()
    mean_k = pkg.FusedMLPPolicy(c_env, pol.net, out_scale=0.01, out_offset=0.0166)
    s32 = std.cpu().numpy()
    for t in range(T):
        xi, rad = no.gaussian_variates(seed, ids, 2 ** 32 + 7 + t, 2)
        ref = -0.5 * (xi ** 2).sum(1) + c
        lpb = no.log_prob_bound(xi, s32, 4)
        assert np.all(np.abs(lp[t] - ref) <= lpb), (t, float(np.max(np.abs(lp[t] - ref) / lpb)))
        st = torch.zeros((n, 12), device='cuda')
        st[:, :10] = ro.obs[t]
        c_env.set_state(st)
        a32 = ro.actions[t].cpu().numpy()
        z = (a32.astype(np.float64) - mean_k().cpu().numpy()) / s64
        # (action - mu) / std is the device variate to half an ulp of the action over std, and that variate is the
        # reference to its own error: -1/2 z^2 moves from -1/2 xi^2 by |xi| eta + eta^2 / 2 per component
        eta = np.spacing(np.abs(a32)) / (2.0 * s64) + no.pair_bound(rad, 4)
        bound = no.SLACK * (np.abs(xi) * eta + 0.5 * eta ** 2).sum(1) + lpb
        assert np.all(np.abs(lp[t] - (-0.5 * (z ** 2).sum(1) + c)) <= bound), t
    # two shards
    lib = _lib.load()
    for lo, k in ((0, 500), (500, n - 500)):
        out = torch.empty((T, k), device='cuda')
        assert lib.copter_policy_logp_f32(seed, off + lo, k, 2 ** 32 + 7, T, 0, std.data_ptr(), out.data_ptr(),
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        assert torch.equal(out, ro.log_probs[:, lo:lo + k])
    # horizons 5 + 7 + 12
    e2 = mk()
    e2.reset()
    e2.rollout_step = 2 ** 32 + 7
    parts = []
    for h in (5, 7, 12):
        r = pkg.FusedPolicyRollout(e2, pol.net, h, out_scale=0.01, out_offset=0.0166, action_std=std, store_log_probs=True)
        r.run()
        parts.append(r.log_probs.clone())
    assert torch.equal(torch.cat(parts), ro.log_probs)


def gae64(r, v, last, causes, fv, gamma, lam):
    T = r.shape[0]
    adv = np.zeros_like(r)
    nxt, a = last.copy(), np.zeros_like(last)
    for t in range(T - 1, -1, -1):
        c = causes[t]
        boot = np.where(c == 0, nxt, np.where((c & 32) != 0, fv[t], 0.0))
        delta = r[t] + gamma * boot - v[t]
        a = delta + gamma * lam * np.where(c == 0, a, 0.0)
        adv[t] = a
        nxt = v[t]
    return adv


def test_rollout_ppo_batch(pkg):
    """On a workload with step-limit truncations: values, last_values and final_values are FusedMLPValue on obs,
    env.obs and final_obs (at truncations; 0 elsewhere) bit for bit; advantages() is gae() on those buffers; the
    batch is within bounds of a PyTorch fp32 critic + float64 GAE; the rollout's own outputs do not change when the
    critic and log-probs are asked for."""
    n, T, seed = 4099, 32, 21
    mk = lambda: pkg.CopterVecEnv('Lander3D', n, seed=seed, max_steps=20)       # noqa: E731
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32, seed=3)
    crit_net = make_critic(vo.critic_case(vo.po.dense_case('Lander3D', 1))['weights'])
    std = torch.tensor([0.02, 0.01, 0.01, 0.02], device='cuda')
    kw = dict(out_scale=0.01, out_offset=0.0166, store_obs=True, store_actions=True, action_std=std, store_causes=True,
              store_final_obs=True)
    a_env, b_env = mk(), mk()
    a_env.reset()
    b_env.reset()
    ro = pkg.FusedPolicyRollout(a_env, pol.net, T, critic=crit_net, store_log_probs=True, **kw)
    plain = pkg.FusedPolicyRollout(b_env, pol.net, T, **kw)
    for _ in range(2):                                   # the second run reuses (and re-zeroes) final_values
        ro.run()
        plain.run()
        for x, y in ((ro.rewards, plain.rewards), (ro.dones, plain.dones), (ro.obs, plain.obs), (ro.actions, plain.actions),
                     (ro.causes, plain.causes), (ro.final_obs, plain.final_obs), (a_env.state, b_env.state),
                     (a_env.meta, b_env.meta)):
            assert torch.equal(x, y)
    trunc = (ro.causes & 32) != 0
    assert int(trunc.sum()) > 0
    critic = pkg.FusedMLPValue(crit_net, a_env)
    assert torch.equal(ro.values, critic(ro.obs))
    assert torch.equal(ro.last_values, critic(a_env.obs))
    fv = torch.where(trunc, critic(ro.final_obs), torch.zeros_like(ro.values))
    assert torch.equal(ro.final_values, fv)
    adv, ret = ro.advantages(0.99, 0.95)
    adv2, ret2 = pkg.gae(ro.rewards, ro.values, ro.last_values, ro.causes, ro.final_values, 0.99, 0.95)
    assert torch.equal(adv, adv2) and torch.equal(ret, ret2)
    # against a PyTorch fp32 critic and float64 GAE
    with torch.no_grad():
        v32 = crit_net(ro.obs)[..., 0].double().cpu().numpy()
        l32 = crit_net(a_env.obs)[..., 0].double().cpu().numpy()
        f32 = crit_net(ro.final_obs)[..., 0].double().cpu().numpy()
    W = [p.detach().double().cpu().numpy() for p in crit_net.parameters()]

    def scale(x):
        h = np.tanh(np.tanh(x @ W[0].T + W[1]) @ W[2].T + W[3])
        return np.abs(h) @ np.abs(W[4][0]) + abs(W[5][0])
    bound = vo.REL_TO_NETWORK * 1.001
    obs64 = ro.obs.double().cpu().numpy()
    assert np.all(np.abs(ro.values.cpu().numpy() - v32) <= bound * scale(obs64))
    assert np.all(np.abs(ro.last_values.cpu().numpy() - l32) <= bound * scale(a_env.obs.double().cpu().numpy()))
    causes = ro.causes.cpu().numpy()
    f32 = np.where((causes & 32) != 0, f32, 0.0)
    ref = gae64(ro.rewards.double().cpu().numpy(), v32, l32, causes, f32, 0.99, 0.95)
    e_v = bound * max(scale(obs64).max(), scale(ro.final_obs.double().cpu().numpy()).max())
    r_abs = np.abs(ro.rewards.double().cpu().numpy()).max()
    tol = (1 + 0.99) / (1 - 0.99 * 0.95) * (e_v + 1e-6 * (1 + r_abs))
    assert np.max(np.abs(adv.double().cpu().numpy() - ref)) <= tol
    # without final_values truncations are terminations
    ro2 = pkg.FusedPolicyRollout(mk(), pol.net, T, critic=crit_net, out_scale=0.01, out_offset=0.0166, store_obs=True,
                                 store_causes=True)
    ro2.env.reset()
    ro2.run()
    assert ro2.final_values is None and ro2.log_probs is None
    adv3, _ = ro2.advantages()
    assert torch.equal(adv3, pkg.gae(ro2.rewards, ro2.values, ro2.last_values, ro2.causes, None)[0])


def test_rollout_construction_errors(pkg):
    env = pkg.CopterVecEnv('Lander3D', 256)
    pol = pkg.mlp_policy(10, 4, dtype=torch.float32).net
    crit = make_critic(vo.critic_case(vo.po.dense_case('Lander3D', 1))['weights'])
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(env, pol, 4, critic=crit)                      # no store_obs
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(env, pol, 4, store_log_probs=True)             # no action_std
    with pytest.raises(pkg.CopterError):
        pkg.FusedPolicyRollout(env, pol, 4, critic=make_critic(vo.critic_case(vo.po.dense_case('Lander2D', 1))['weights']),
                               store_obs=True)                                # O = 6 critic on a Lander3D env
    ro = pkg.FusedPolicyRollout(env, pol, 4, critic=crit, store_obs=True)
    with pytest.raises(pkg.CopterError):
        ro.advantages()                                                       # no store_causes
    ro = pkg.FusedPolicyRollout(env, pol, 4, store_causes=True)
    with pytest.raises(pkg.CopterError):
        ro.advantages()                                                       # no critic
