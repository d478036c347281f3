"""FusedPolicyRollout's PPO batch on every variant and both fused rollout kernels, against float64 references with
derived bounds (oracle/noise_oracle.py, policy_oracle.py, value_oracle.py):
  a. copter_policy_logp_f32 for A = 1, 2 and 4 on 2^20 envs x 4 steps, both high words of the env id and the step in
     play, every element within log_prob_bound of the float64 formula on the reference variates -- including the
     Gaussian's tails (c < 2^12), the tiny radii (u1 within 2^-20 of 1) and the edges of the folded angle;
  b. the exploration noise both fused rollout kernels draw, on all seven variants: (action - mu) / std within
     ulp(action) / (2 std) + variate_bound of the reference variate, and the rollout's log_probs within log_prob_bound;
  c. the whole PPO batch bit for bit against the standalone calls, the critic against its rounding model and the
     float64 network, the sampled actions' log-probabilities against the density of the float64 policy (the first
     PPO ratio), and advantages() against float64 GAE on float64 critic values;
  d. two shards at a split that is not a multiple of 128 (every env on another row of its tcgen05 tile) are the
     unsharded batch, bit for bit.

With COPTER_PPO_BATCH_REPORT=<path> the worst error / bound ratios per class, variant and kernel and the epoch-0
log-ratio deviations are written there as JSON."""
import ctypes as C
import functools
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import noise_oracle as no                      # noqa: E402
from oracle import policy_oracle as po                     # noqa: E402
from oracle import value_oracle as vo                      # noqa: E402

VARIANTS = list(po.VARIANTS)
KIND = {'1': 'tc', '0': 'mma'}
STD = {1: (0.013,), 2: (0.02, 0.0071), 4: (0.02, 0.01, 0.005, 0.015)}     # per component, different per j
OUT_SCALE, OUT_OFFSET = 0.01, 0.0166
REPORT = {}


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    yield gym_copter_b200
    path = os.environ.get('COPTER_PPO_BATCH_REPORT')
    if path:
        REPORT['device'] = torch.cuda.get_device_name()
        try:                                             # the power limit the numbers were taken at (a read-only query)
            import subprocess
            REPORT['power_limit'] = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                                                    str(torch.cuda.current_device())], capture_output=True, text=True,
                                                   timeout=30).stdout.strip()
        except (OSError, subprocess.SubprocessError):
            REPORT['power_limit'] = None
        with open(path, 'w') as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)


@pytest.fixture
def policy_kernel_choice():
    """COPTER_B200_POLICY_TC selects the standalone policy kernel per call -- '1' tcgen05 / TMEM (its default),
    '0' warp-level mma.sync -- and COPTER_B200_POLICY_ROLLOUT_TC the fused policy + step rollout kernel (the same
    values and default).  choose(v) sets both to the same kind."""
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


def report(*keys, **values):
    d = REPORT
    for k in keys:
        d = d.setdefault(k, {})
    d.update(values)


def worst(ratio):
    return float(np.max(ratio)) if np.size(ratio) else 0.0


def make_critic(weights):
    net = torch.nn.Sequential(torch.nn.Linear(weights[0].shape[1], 64), torch.nn.Tanh(), torch.nn.Linear(64, 64),
                              torch.nn.Tanh(), torch.nn.Linear(64, 1))
    for p, w in zip(net.parameters(), weights):
        p.data = torch.from_numpy(np.ascontiguousarray(w, np.float32))
    return net.cuda()


def critic_weights(variant):
    """The value_oracle critic of a variant: mlp_policy weights (policy_oracle.dense_weights), layer 3 = row 0."""
    W = po.dense_weights(variant, 1)
    return W[:4] + (np.ascontiguousarray(W[4][:1]), np.ascontiguousarray(W[5][:1]))


def state_rows(obs, variant):
    """[M, O] observations -> [M, 12] fp32 state rows holding them at columns first .. first + O - 1."""
    first, O, _ = po.VARIANTS[variant]
    st = torch.zeros((obs.shape[0], 12), dtype=torch.float32, device=obs.device)
    st[:, first:first + O] = obs
    return st


def standalone_means(pkg, variant, net, obs_tn):
    """mu [T, N, A] of the standalone policy kernel (the kind COPTER_B200_POLICY_TC selects) on recorded observations:
    bit-identical to the fused kernel's mean of the same kind (test_fused_policy_rollout_equals_policy_kernel_plus_step)."""
    T, n, _ = obs_tn.shape
    env = pkg.CopterVecEnv(variant, n)
    mean = pkg.FusedMLPPolicy(env, net, out_scale=OUT_SCALE, out_offset=OUT_OFFSET)
    out = []
    for t in range(T):
        env.set_state(state_rows(obs_tn[t], variant))
        out.append(mean().clone())
    return torch.stack(out)


def reference_variates(seed, env_offset, n, first_step, T):
    """xi [T, n, 4] and the pair radii [T, n, 2] of the exploration stream (tag 2)."""
    ids = np.arange(n, dtype=np.uint64) + np.uint64(env_offset)
    xr = [no.gaussian_variates(seed, ids, first_step + t, 2) for t in range(T)]
    return np.stack([x for x, _ in xr]), np.stack([r for _, r in xr])


def noise_slack(actions, std):
    """eta [.., A]: how far (action - mu) / std may be from the device variate -- the fmaf's rounding of the action,
    half an ulp of it, over std."""
    a32 = np.abs(np.asarray(actions, np.float32))
    return np.spacing(a32).astype(np.float64) / (2 * np.asarray(std, np.float64))


# ---- a. the log-prob kernel at the Gaussian's tails ----------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def sample_step(t):
    """Reference variates, pair radii and hard-class masks of step t of no.LOGP_SAMPLE."""
    s = no.LOGP_SAMPLE
    c = no.philox_counters(s['seed'], no.sample_ids(), s['first_step'] + t, 2)
    xi, r = no.variates_from_counters(c)
    return xi, r, no.pair_classes(c)


@pytest.mark.parametrize('A', [1, 2, 4])
def test_log_prob_kernel_vs_float64(pkg, A):
    from gym_copter_b200 import _lib
    s = no.LOGP_SAMPLE
    variant = no.LOGP_VARIANTS[A]
    std = torch.tensor(no.LOGP_STD[A], dtype=torch.float32, device='cuda')
    s32 = std.cpu().numpy()
    out = torch.full((s['T'], s['n']), float('nan'), device='cuda')
    rc = _lib.load().copter_policy_logp_f32(s['seed'], s['env_offset'], s['n'], s['first_step'], s['T'],
                                            _lib.VARIANT_IDS[variant], std.data_ptr(), out.data_ptr(),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    got = out.cpu().numpy().astype(np.float64)
    pairs = 1 if A < 4 else 2
    ratios = {k: [] for k in ('all', 'tail', 'u1_near_1', 'u2_edge')}
    counts = dict.fromkeys(ratios, 0)
    for t in range(s['T']):
        xi, r, cls = sample_step(t)
        ratio = np.abs(got[t] - no.log_prob(xi, s32, A)) / no.log_prob_bound(xi, s32, A)
        assert np.all(ratio <= 1.0), (t, float(np.nanmax(ratio)), int(np.argmax(np.nan_to_num(ratio, nan=np.inf))))
        ratios['all'].append(worst(ratio))
        counts['all'] += len(ratio)
        for k in ('tail', 'u1_near_1', 'u2_edge'):
            m = cls[k][:, :pairs].any(1)
            ratios[k].append(worst(ratio[m]))
            counts[k] += int(m.sum())
    assert all(counts.values()), counts                  # every hard class is in the sample
    report('log_prob_kernel', 'A=%d' % A, **{k: max(v) for k, v in ratios.items()},
           counts=counts, variant=variant)


# ---- b. exploration noise of both fused rollout kernels, every variant ----------------------------------------------

@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('variant', VARIANTS)
def test_rollout_exploration_noise_vs_float64(pkg, variant, kernel, policy_kernel_choice):
    """z = (action - mu) / std, with mu the standalone kernel of the same kind on the recorded observations, is the
    reference variate to within ulp(action) / (2 std) + variate_bound(r); the rollout's log_probs are the float64
    formula on the reference variates to within log_prob_bound."""
    policy_kernel_choice(kernel)
    n, T, seed, off, first_step = 2053, 16, 0xABCDEF0123, (7 << 32) + 3, 2 ** 32 + 7
    env = pkg.CopterVecEnv(variant, n, seed=seed, env_offset=off)
    A = env.action_size
    pol = pkg.mlp_policy(env.obs_size, A, dtype=torch.float32, seed=9)
    std = torch.tensor(STD[A], dtype=torch.float32, device='cuda')
    env.reset()
    env.rollout_step = first_step
    ro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=OUT_SCALE, out_offset=OUT_OFFSET, store_obs=True,
                                store_actions=True, action_std=std, store_log_probs=True)
    ro.run()
    mu = standalone_means(pkg, variant, pol.net, ro.obs).cpu().numpy().astype(np.float64)
    a32 = ro.actions.cpu().numpy()
    s32 = std.cpu().numpy()
    xi, r = reference_variates(seed, off, n, first_step, T)
    z = (a32.astype(np.float64) - mu) / s32.astype(np.float64)
    bound = no.SLACK * (noise_slack(a32, s32) + no.pair_bound(r.reshape(-1, 2), A).reshape(T, n, A))
    noise = np.abs(z - xi[..., :A]) / bound
    assert np.all(noise <= 1.0), (float(noise.max()), np.unravel_index(np.argmax(noise), noise.shape))
    assert 0.5 < np.std(z) < 2.0                          # the noise is there, at the configured scale
    lp = ro.log_probs.cpu().numpy().astype(np.float64).reshape(-1)
    xf = xi.reshape(-1, 4)
    lpr = np.abs(lp - no.log_prob(xf, s32, A)) / no.log_prob_bound(xf, s32, A)
    assert np.all(lpr <= 1.0), float(lpr.max())
    report('rollout_noise', variant, 'kernel=' + KIND[kernel], noise=worst(noise), log_probs=worst(lpr))


# ---- c. the PPO batch against float64 ----------------------------------------------------------------------------

def ppo_batch(pkg, variant, n, env_offset, seed=21, T=32):
    """The workload of parts c and d: max_steps = 20, so step-limit truncations fall inside the horizon; the tanh actor
    with per-component exploration noise, the value_oracle critic, log-probs; the rollout has run once."""
    env = pkg.CopterVecEnv(variant, n, seed=seed, env_offset=env_offset, max_steps=20, track_returns=True)
    pol = pkg.mlp_policy(env.obs_size, env.action_size, dtype=torch.float32, seed=3)
    std = torch.tensor(STD[env.action_size], dtype=torch.float32, device='cuda')
    crit = make_critic(critic_weights(variant))
    ro = pkg.FusedPolicyRollout(env, pol.net, T, out_scale=OUT_SCALE, out_offset=OUT_OFFSET, store_obs=True,
                                store_actions=True, action_std=std, store_causes=True, store_final_obs=True,
                                critic=crit, store_log_probs=True)
    env.reset()
    ro.run()
    return env, pol, std, crit, ro


def critic_check(values, obs, variant, Wc):
    """(|got - model| / ceiling, |got - float64 network| / (REL_TO_NETWORK * scale), model - network + ceiling) per row."""
    obs = np.asarray(obs, np.float32).reshape(-1, po.VARIANTS[variant][1])
    got = np.asarray(values, np.float64).reshape(-1)
    m, cei = vo.model(obs, variant, *Wc), vo.ceiling(obs, variant, *Wc)
    exact = vo.model(obs, variant, *Wc, exact=True)
    return np.abs(got - m) / cei, np.abs(got - exact) / (vo.REL_TO_NETWORK * vo.scale(obs, variant, *Wc)), \
        np.abs(m - exact) + cei, exact


def gae64(r, v, last, causes, fv, gamma, lam):
    T = r.shape[0]
    adv = np.zeros_like(r)
    nxt, a = last.copy(), np.zeros_like(last)
    for t in range(T - 1, -1, -1):
        c = causes[t]
        boot = np.where(c == 0, nxt, np.where((c & 32) != 0, fv[t], 0.0))
        a = r[t] + gamma * boot - v[t] + gamma * lam * np.where(c == 0, a, 0.0)
        adv[t] = a
        nxt = v[t]
    return adv


@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('variant', VARIANTS)
def test_ppo_batch_vs_float64(pkg, variant, kernel, policy_kernel_choice):
    """n = 4099 (a ragged last tile), T = 32.
      * bit for bit: values = FusedMLPValue(obs); last_values = FusedMLPValue(env.obs), the stride-12 view from column
        `first`; final_values = the critic on final_obs where the step limit fired, 0 elsewhere; log_probs =
        policy_log_probs; advantages() = gae() on those buffers;
      * the critic within value_oracle's ceiling of its rounding model and within REL_TO_NETWORK * scale of the float64
        network, on obs, env.obs and the truncations' final_obs;
      * the first PPO ratio: with e = |mu_dev - mu64| (mu64 the float64 policy on the recorded obs), e <= |model - mu64|
        + ceiling, and |log_probs - log N(action; mu64, std^2)| <= sum_j (|z_j| + e_j / (2 std_j)) e_j / std_j, the
        step from z = (action - mu_dev) / std to the reference variate, and log_prob_bound;
      * advantages() within the propagated bound of float64 GAE on the float64 critic's values."""
    from gym_copter_b200.rollout import policy_log_probs
    policy_kernel_choice(kernel)
    n, T, gamma, lam = 4099, 32, 0.99, 0.95
    env, pol, std, crit, ro = ppo_batch(pkg, variant, n, 0)
    first, O, A = po.VARIANTS[variant]
    assert tuple(env.obs.stride()) == (12, 1) and env.obs.storage_offset() == first
    trunc = (ro.causes & 32) != 0
    assert int(trunc.sum()) > 0
    critic = pkg.FusedMLPValue(crit, env)
    assert torch.equal(ro.values, critic(ro.obs))
    assert torch.equal(ro.last_values, critic(env.obs))
    assert torch.equal(ro.final_values, torch.where(trunc, critic(ro.final_obs), torch.zeros_like(ro.values)))
    assert torch.equal(ro.log_probs, policy_log_probs(env, std, env.rollout_step - T, T))
    adv, ret = ro.advantages(gamma, lam)
    adv2, ret2 = pkg.gae(ro.rewards, ro.values, ro.last_values, ro.causes, ro.final_values, gamma, lam)
    assert torch.equal(adv, adv2) and torch.equal(ret, ret2)

    # the critic against float64
    Wc = critic_weights(variant)
    tr = trunc.cpu().numpy()
    rep, exact = {}, {}
    e_v = 0.0                                        # bound on |device value - float64 value| over every value GAE reads
    for name, vals, obs in (('values', ro.values, ro.obs), ('last_values', ro.last_values, env.obs),
                            ('final_values', ro.final_values[trunc], ro.final_obs[trunc])):
        to_model, to_net, err, exact[name] = critic_check(vals.cpu().numpy(), obs.cpu().numpy(), variant, Wc)
        assert np.all(to_model <= 1.0) and np.all(to_net <= 1.0), (name, worst(to_model), worst(to_net))
        rep['critic_%s_to_ceiling' % name], rep['critic_%s_to_network' % name] = worst(to_model), worst(to_net)
        e_v = max(e_v, float(err.max()))
    v64, l64 = exact['values'].reshape(T, n), exact['last_values']
    f64 = np.zeros((T, n))
    f64[tr] = exact['final_values']

    # the first PPO ratio against the float64 policy
    W = [p.detach().cpu().numpy() for p in pol.net.parameters()]
    rows = state_rows(ro.obs.reshape(-1, O), variant).cpu().numpy()
    args = (rows, variant) + tuple(W) + (OUT_SCALE, OUT_OFFSET)
    mu_dev = standalone_means(pkg, variant, pol.net, ro.obs).cpu().numpy().astype(np.float64).reshape(-1, A)
    mu_model, mu_cei = po.model(KIND[kernel], *args), po.ceiling(KIND[kernel], *args)
    mu64 = po.model(KIND[kernel], *args, exact=True)
    e = np.abs(mu_dev - mu64)
    mu_ratio = e / (np.abs(mu_model - mu64) + mu_cei)
    assert np.all(mu_ratio <= 1.0), worst(mu_ratio)
    a32 = ro.actions.cpu().numpy().reshape(-1, A)
    s32 = std.cpu().numpy()
    s64 = s32.astype(np.float64)
    a64 = a32.astype(np.float64)
    xi, r = reference_variates(21, 0, n, env.rollout_step - T, T)
    xi, r = xi.reshape(-1, 4), r.reshape(-1, 2)
    logn64 = -0.5 * (((a64 - mu64) / s64) ** 2).sum(1) - np.log(s64).sum() - 0.5 * A * no.LOG_2PI
    lp = ro.log_probs.cpu().numpy().astype(np.float64).reshape(-1)
    z = (a64 - mu_dev) / s64
    eta = noise_slack(a32, s32) + no.pair_bound(r, A)              # |z - xi| (part b)
    bound = ((np.abs(z) + e / (2 * s64)) * e / s64).sum(1) + (np.abs(xi[:, :A]) * eta + 0.5 * eta ** 2).sum(1) \
        + no.log_prob_bound(xi, s32, A)
    dev = np.abs(lp - logn64)
    ratio = dev / (no.SLACK * bound)
    assert np.all(ratio <= 1.0), (worst(ratio), float(dev.max()))

    # GAE against float64 GAE on the float64 critic's values
    rew = ro.rewards.cpu().numpy().astype(np.float64)
    causes = ro.causes.cpu().numpy()
    ref = gae64(rew, v64, l64, causes, f64, float(np.float32(gamma)), float(np.float32(lam)))
    tol = (1 + gamma) / (1 - gamma * lam) * (e_v + 1e-6 * (1 + np.abs(rew).max()))
    gae_ratio = np.abs(adv.cpu().numpy().astype(np.float64) - ref) / tol
    assert np.all(gae_ratio <= 1.0), worst(gae_ratio)
    ret_ratio = np.abs(ret.cpu().numpy().astype(np.float64) - (ref + v64)) / (tol + e_v)
    assert np.all(ret_ratio <= 1.0), worst(ret_ratio)
    report('ppo_batch', variant, 'kernel=' + KIND[kernel], mean_to_model_and_ceiling=worst(mu_ratio),
           epoch0_log_ratio_to_bound=worst(ratio), epoch0_log_ratio_max=float(dev.max()),
           epoch0_log_ratio_mean=float(dev.mean()), advantages_to_bound=worst(gae_ratio),
           returns_to_bound=worst(ret_ratio), truncations=int(tr.sum()), **rep)


# ---- d. split shards are the unsharded batch ----------------------------------------------------------------------

@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('variant', VARIANTS)
def test_split_shards_are_the_unsharded_batch(pkg, variant, kernel, policy_kernel_choice):
    """Two envs with env_offset 0 and 1000 (sizes 1000 and 3099: the split is not a multiple of 128, so every env of
    the second shard sits on another row of its tcgen05 tile) and the same seed, critic and log-probs: every [T, N]
    and [T, N, .] buffer, concatenated along N, is the unsharded batch bit for bit, and so are last_values, the final
    state and meta; the statistics' counts add up and the return sums agree to their last bits."""
    from gym_copter_b200._lib import STAT_NAMES
    policy_kernel_choice(kernel)
    whole = ppo_batch(pkg, variant, 4099, 0)
    parts = [ppo_batch(pkg, variant, k, lo) for lo, k in ((0, 1000), (1000, 3099))]
    wenv, wro = whole[0], whole[-1]

    def cat(get, dim=1):
        return torch.cat([get(p[-1]) for p in parts], dim)
    adv_w, ret_w = wro.advantages()
    for name in ('rewards', 'dones', 'obs', 'actions', 'causes', 'final_obs', 'values', 'final_values', 'log_probs'):
        assert torch.equal(cat(lambda ro: getattr(ro, name)), getattr(wro, name)), name
    assert torch.equal(cat(lambda ro: ro.advantages()[0]), adv_w)
    assert torch.equal(cat(lambda ro: ro.advantages()[1]), ret_w)
    assert torch.equal(cat(lambda ro: ro.last_values, 0), wro.last_values)
    assert torch.equal(torch.cat([p[0].state for p in parts]), wenv.state)
    assert torch.equal(torch.cat([p[0].meta for p in parts]), wenv.meta)
    assert int(((wro.causes & 32) != 0).sum()) > 0
    sa = sum(p[0]._stats.sum(0) for p in parts)
    sb = wenv._stats.sum(0)
    ret = STAT_NAMES.index('return_sum')
    keep = [j for j in range(sa.numel()) if j != ret]
    assert torch.equal(sa[keep], sb[keep])
    assert abs(sa[ret].item() - sb[ret].item()) <= 1e-12 * max(1.0, abs(sb[ret].item()))
