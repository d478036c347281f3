#!/usr/bin/env python3
"""
Cost of a PPO batch on the device (run on the GPU box): Lander3D fp32, N = 2^23 envs, T = 16, exploration noise on,
the critic Linear(10,64) -> tanh -> Linear(64,64) -> tanh -> Linear(64,1).  Writes ONE JSON record (appended to
--out, default profiles/ppo_batch_bench.jsonl) with the card's name and power limit read in the same run:

  kernels        the tcgen05 policy kernel at M = N, the critic kernel at M = N (the env's stride-12 observation view)
                 and at M = T N (the rollout's packed obs), the critic with selection on final_obs at the ~1/1000
                 truncation density of a 1000-step limit, and the log-prob kernel over [T, N]
  ppo_batch      the whole batch -- rollout + values + last / final values + log-probs + GAE -- on the new path
                 (FusedPolicyRollout(critic=..., store_log_probs=True) + advantages()), against the rollout followed
                 by a PyTorch critic (fp32 and bf16) on obs / final_obs / the last observation, PyTorch log-probs
                 from the recorded actions (the actor re-evaluated in the same precision) and gae()
  logp_deviation the epoch-0 mean and max |log pi_torch-fp32(a|s) - log_probs|: what a learner whose fp32 actor
                 rounds differently from the bf16 / fp16 kernel that sampled the action sees at its first ratio

Every time is the median over REPS repetitions of CUDA-event-timed launches after a warm-up; the buffers of the
timed work (GBs at this size) are far larger than the 126 MB L2.
"""
import argparse
import copy
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gym_copter_b200 as g      # noqa: E402

REPS = 7
OUT_SCALE, OUT_OFFSET = 0.01, 0.0166


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def median_ms(fn, launches):
    fn(); fn()
    ms = sorted(timed(fn, launches) for _ in range(REPS))
    return {'median_ms': ms[REPS // 2], 'min_ms': ms[0], 'max_ms': ms[-1]}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().split('\n')[0]
    return {'card': torch.cuda.get_device_name(0), 'nvidia_smi_name_power_limit_max_sm_clock': q}


def critic_net(seed=11):
    gen = torch.Generator(device='cpu').manual_seed(seed)
    net = torch.nn.Sequential(torch.nn.Linear(10, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                              torch.nn.Linear(64, 1))
    for p in net.parameters():
        p.data = torch.randn(p.shape, generator=gen) * (0.5 / max(1, p.shape[-1]) ** 0.5)
    return net.cuda()


def torch_log_prob(actor, obs_t, act_t, std):
    mu = OUT_OFFSET + OUT_SCALE * actor(obs_t.to(next(actor.parameters()).dtype)).float()
    z = (act_t - mu) / std
    return -0.5 * (z * z).sum(-1) - torch.log(std).sum() - 0.5 * act_t.shape[-1] * math.log(2 * math.pi)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=1 << 23)
    ap.add_argument('--horizon', type=int, default=16)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'ppo_batch_bench.jsonl'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_ppo_batch.py measures on the GPU: no CUDA device')
    n, T = args.n, args.horizon
    rec = dict(card(), workload='Lander3D fp32, N = %d, T = %d, action_std = [0.02, 0.01, 0.01, 0.02]' % (n, T))
    pol = g.mlp_policy(10, 4, dtype=torch.float32, seed=5)
    crit = critic_net()
    std = torch.tensor([0.02, 0.01, 0.01, 0.02], device='cuda')
    env = g.CopterVecEnv('Lander3D', n, seed=2026)
    env.reset()
    kw = dict(out_scale=OUT_SCALE, out_offset=OUT_OFFSET, store_obs=True, store_actions=True, action_std=std,
              store_causes=True, store_final_obs=True)
    ro = g.FusedPolicyRollout(env, pol.net, T, critic=crit, store_log_probs=True, **kw)
    snap = env.state_dict()
    ro.run()
    torch.cuda.synchronize()

    # ---- kernels alone
    value = g.FusedMLPValue(crit, env)
    policy = g.FusedMLPPolicy(env, pol.net, out_scale=OUT_SCALE, out_offset=OUT_OFFSET)
    vN = torch.empty(n, device='cuda')
    vTN = torch.empty((T, n), device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(1)
    sel = ((torch.rand((T, n), device='cuda', generator=gen) < 1e-3).to(torch.uint8) * g._lib.CAUSE_TIMEOUT)
    live_tiles = float((sel.view(-1)[:(T * n) // 128 * 128].view(-1, 128) != 0).any(1).float().mean())
    fv = torch.zeros((T, n), device='cuda')
    lp = torch.empty((T, n), device='cuda')
    from gym_copter_b200.rollout import policy_log_probs
    rec['kernels'] = {
        'policy_tc_M=N': median_ms(policy, 20),
        'critic_M=N_env_view': median_ms(lambda: value(env.obs, out=vN), 20),
        'critic_M=TN_packed_obs': median_ms(lambda: value(ro.obs, out=vTN), 5),
        'critic_final_obs_selected': dict(median_ms(lambda: value(ro.final_obs, select=sel, out=fv), 10),
                                          selected_rows=int((sel != 0).sum()), live_tile_fraction=live_tiles),
        'logp_TxN': median_ms(lambda: policy_log_probs(env, std, 0, T, out=lp), 10),
    }
    k = rec['kernels']
    k['critic_M=TN_ms_per_row_block_of_N'] = k['critic_M=TN_packed_obs']['median_ms'] / T

    # ---- the whole batch
    plain = g.FusedPolicyRollout(env, pol.net, T, **kw)
    actor16, crit16 = copy.deepcopy(pol.net).to(torch.bfloat16), copy.deepcopy(crit).to(torch.bfloat16)

    def new_path():
        ro.run()
        ro.advantages(0.99, 0.95)

    def torch_path(actor, critic_t):
        dt = next(critic_t.parameters()).dtype

        def run():
            plain.run()
            with torch.no_grad():
                vals = torch.empty((T, n), device='cuda')
                fvals = torch.zeros((T, n), device='cuda')
                logp = torch.empty((T, n), device='cuda')
                trunc = (plain.causes & g._lib.CAUSE_TIMEOUT) != 0
                for t in range(T):
                    vals[t] = critic_t(plain.obs[t].to(dt))[:, 0].float()
                    fvals[t] = torch.where(trunc[t], critic_t(plain.final_obs[t].to(dt))[:, 0].float(), fvals[t])
                    logp[t] = torch_log_prob(actor, plain.obs[t], plain.actions[t], std)
                last = critic_t(env.obs.to(dt))[:, 0].float()
            g.gae(plain.rewards, vals, last, plain.causes, fvals, 0.99, 0.95)
        return run
    res = {'new_path': median_ms(new_path, 3),
           'rollout_only': median_ms(plain.run, 3),
           'torch_fp32': median_ms(torch_path(pol.net, crit), 1),
           'torch_bf16': median_ms(torch_path(actor16, crit16), 1)}
    res['new_over_torch_fp32'] = res['new_path']['median_ms'] / res['torch_fp32']['median_ms']
    res['new_over_torch_bf16'] = res['new_path']['median_ms'] / res['torch_bf16']['median_ms']
    res['note'] = ('the env runs on from arm to arm (auto-reset); the torch arms run the critic and actor per row t of '
                   '[T, N] (N rows at a time)')
    rec['ppo_batch'] = res

    # ---- epoch-0 log-prob deviation and value agreement
    env.load_state_dict(snap)
    ro.run()
    with torch.no_grad():
        dev_sum, dev_max, vdev = 0.0, 0.0, 0.0
        for t in range(T):
            d = (torch_log_prob(pol.net, ro.obs[t], ro.actions[t], std) - ro.log_probs[t]).abs()
            dev_sum += float(d.double().sum())
            dev_max = max(dev_max, float(d.max()))
            vdev = max(vdev, float((crit(ro.obs[t])[:, 0] - ro.values[t]).abs().max()))
    rec['logp_deviation'] = {'mean_abs': dev_sum / (T * n), 'max_abs': dev_max,
                             'what': '|log pi_torch-fp32(a|s) - log_probs| over the [T, N] batch, epoch 0'}
    rec['value_max_abs_diff_vs_torch_fp32'] = vdev
    rec['truncations_in_batch'] = int(((ro.causes & g._lib.CAUSE_TIMEOUT) != 0).sum())
    line = json.dumps(rec)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'a') as f:
        f.write(line + '\n')


if __name__ == '__main__':
    main()
