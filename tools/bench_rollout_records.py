#!/usr/bin/env python3
"""
Cost of the rollouts' ending records and speed of the on-device GAE (run on the GPU box; one JSON line per
measurement, the first naming the card and its power limit):

  (a) FusedPolicyRollout on bench.py's policy workload (Lander3D fp32, 2^23 envs, T = 16, write_obs=False):
      records off vs store_causes + store_final_obs, alternating, REPS repetitions of 10 launches each.
  (b) env.rollout(source='randn'), Lander3D fp32, 2^24 envs, T = 16: records off, causes only, causes + terminal
      observations (the call allocates and zero-fills its [T,N,O] final_obs, so that arm includes the fill),
      alternating.
  (c) copter_gae_f32 at T = 32, N = 2^23 on the causes of a real rollout (uniform commands and a 25-step limit:
      terminations and truncations), with final values, against a plain torch backward loop computing the same
      thing.  GB/s from the algorithmic bytes (17 per element + 4 per truncation read) and the fraction of a
      device-to-device copy's rate measured in the same run (4 GiB buffers, far beyond the 126 MB L2).
"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gym_copter_b200 as g      # noqa: E402

REPS = 7


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def summary(ms):
    ms = sorted(ms)
    med = ms[len(ms) // 2]
    return {'median_ms': med, 'min_ms': ms[0], 'max_ms': ms[-1], 'spread': (ms[-1] - ms[0]) / med, 'samples_ms': ms}


def alternate(arms, reps, launches):
    """arms: {name: fn}; every repetition times each arm once (launches calls), in turn."""
    for fn in arms.values():
        fn(); fn()
    out = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            out[k].append(timed(fn, launches))
    return {k: summary(v) for k, v in out.items()}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().split('\n')[0]
    print(json.dumps({'card': torch.cuda.get_device_name(0), 'nvidia_smi': q}), flush=True)


def fused_policy():
    n, T = 1 << 23, 16
    env = g.CopterVecEnv('Lander3D', n, seed=2026, write_obs=False)
    env.reset()
    pol = g.mlp_policy(10, 4, dtype=torch.float32, seed=5)
    kw = dict(out_scale=0.2 * 0.0166, out_offset=0.0166)
    off = g.FusedPolicyRollout(env, pol.net, T, **kw)
    on = g.FusedPolicyRollout(env, pol.net, T, store_causes=True, store_final_obs=True, **kw)
    res = alternate({'records_off': off.run, 'records_on': on.run}, REPS, 10)
    for k, v in res.items():
        v['env_steps_per_s'] = n * T / (v['median_ms'] * 1e-3)
    print(json.dumps({'bench': '(a) FusedPolicyRollout Lander3D fp32 2^23 envs T=16 write_obs=False (bench.py policy_rollout workload)',
                      'ms_per_launch': res, 'on_over_off': res['records_on']['median_ms'] / res['records_off']['median_ms']}), flush=True)
    del off, on, env


def env_rollout():
    n, T = 1 << 24, 16
    env = g.CopterVecEnv('Lander3D', n, seed=2)
    env.reset()
    arms = {'records_off': lambda: env.rollout(T, source='randn'),
            'causes': lambda: env.rollout(T, source='randn', record_causes=True),
            'causes_and_final_obs': lambda: env.rollout(T, source='randn', record_causes=True, record_final_obs=True)}
    res = alternate(arms, REPS, 5)
    for k, v in res.items():
        v['env_steps_per_s'] = n * T / (v['median_ms'] * 1e-3)
    print(json.dumps({'bench': "(b) env.rollout(source='randn') Lander3D fp32 2^24 envs T=16", 'ms_per_launch': res,
                      'causes_over_off': res['causes']['median_ms'] / res['records_off']['median_ms'],
                      'causes_and_final_obs_over_off': res['causes_and_final_obs']['median_ms'] / res['records_off']['median_ms']}),
          flush=True)
    del env
    torch.cuda.empty_cache()


def torch_gae(r, v, last, c, fv, gamma, lam):
    adv = torch.empty_like(r)
    run, trunc = c == 0, (c & g._lib.CAUSE_TIMEOUT) != 0
    a, nxt, zero = torch.zeros_like(last), last, torch.zeros_like(last)
    for t in range(r.shape[0] - 1, -1, -1):
        boot = torch.where(run[t], nxt, torch.where(trunc[t], fv[t], zero))
        a = r[t] + gamma * boot - v[t] + gamma * lam * torch.where(run[t], a, zero)
        adv[t] = a
        nxt = v[t]
    return adv, adv + v


def gae():
    n, T = 1 << 23, 32
    env = g.CopterVecEnv('Lander3D', n, seed=3, max_steps=25)
    env.reset()
    out = env.rollout(T, source='uniform', record_rewards=True, record_causes=True)
    r, c = out['rewards'], out['causes']
    gen = torch.Generator(device='cuda').manual_seed(0)
    v = torch.randn((T, n), device='cuda', generator=gen)
    fv = torch.randn((T, n), device='cuda', generator=gen)
    last = torch.randn(n, device='cuda', generator=gen)
    del env
    trunc = int(((c & g._lib.CAUSE_TIMEOUT) != 0).sum())
    term = int(((c != 0) & ((c & g._lib.CAUSE_TIMEOUT) == 0)).sum())
    nbytes = 17 * T * n + 4 * trunc
    adv, ret = g.gae(r, v, last, c, fv)
    ref_adv, ref_ret = torch_gae(r, v, last, c, fv, 0.99, 0.95)
    err = ((adv - ref_adv).abs() / ref_adv.abs().clamp_min(1)).max().item()
    ms_k = [timed(lambda: g.gae(r, v, last, c, fv), 20) for _ in range(REPS)]
    ms_t = [timed(lambda: torch_gae(r, v, last, c, fv, 0.99, 0.95), 3) for _ in range(3)]
    src = torch.empty(1 << 30, dtype=torch.float32, device='cuda')
    dst = torch.empty_like(src)
    ms_c = [timed(lambda: dst.copy_(src), 20) for _ in range(REPS)]
    copy_gbs = 2 * src.numel() * 4 / (sorted(ms_c)[REPS // 2] * 1e-3) / 1e9
    k = summary(ms_k)
    gbs = nbytes / (k['median_ms'] * 1e-3) / 1e9
    print(json.dumps({'bench': '(c) copter_gae_f32 T=32 N=2^23, causes of a Lander3D uniform-command rollout with a 25-step limit, '
                               'final values given', 'steps_terminated': term, 'steps_truncated': trunc,
                      'algorithmic_bytes': nbytes, 'kernel': k, 'gb_per_s': gbs,
                      'copy_gb_per_s': copy_gbs, 'copy': summary(ms_c), 'frac_of_copy': gbs / copy_gbs,
                      'torch_loop': summary(ms_t), 'speedup_over_torch_loop': sorted(ms_t)[1] / k['median_ms'],
                      'max_rel_diff_vs_torch_loop': err}), flush=True)


if __name__ == '__main__':
    torch.cuda.set_device(0)
    card()
    fused_policy()
    env_rollout()
    gae()
