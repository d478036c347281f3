#!/usr/bin/env python3
"""
Developer tool: times builds of the library against each other.  `build` cross-compiles the current
sources here (no GPU needed) into tools/variants/lib_current.so; `run` times it and every hand-built
tools/variants/lib_v*.so on the GPU box (one subprocess per build) and prints achieved GB/s and the
policy kernel's time and error.

    python tools/sweep.py build
    gpurun -- python tools/sweep.py run [--envs N] [--k K]
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VDIR = os.path.join(ROOT, 'tools', 'variants')
SRC = os.path.join(ROOT, 'gym_copter_b200', 'csrc', 'copter_kernels.cu')

sys.path.insert(0, ROOT)
from gym_copter_b200.build import NVCC_FLAGS          # noqa: E402  (the product's own flags: -fmad=false etc.)

VARIANTS = {}
VARIANTS['current'] = []
if os.environ.get('COPTER_SWEEP_ONLY'):
    VARIANTS = {k: v for k, v in VARIANTS.items() if k.startswith(tuple(os.environ['COPTER_SWEEP_ONLY'].split(',')))}


def build():
    os.makedirs(VDIR, exist_ok=True)
    procs = []
    for name, flags in VARIANTS.items():
        out = os.path.join(VDIR, 'lib_%s.so' % name)
        cmd = ['nvcc'] + NVCC_FLAGS + flags + ['-o', out, SRC]
        procs.append((name, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        if len(procs) >= 8:
            for n, p in procs:
                o, _ = p.communicate()
                print(n, 'rc', p.returncode, o[-200:] if p.returncode else '')
            procs = []
    for n, p in procs:
        o, _ = p.communicate()
        print(n, 'rc', p.returncode, o[-200:] if p.returncode else '')


def time_one(envs, k, steps, stats):
    import torch
    sys.path.insert(0, ROOT)
    import gym_copter_b200 as g
    env = g.LanderVec(envs, seed=1, k_substeps=k, track_stats=bool(stats))
    env.reset()
    acts = [1.625e-2 * torch.randn((envs, 4), device='cuda') for _ in range(4)]
    for i in range(20):
        env.step(acts[i % 4])
    best = 1e9
    for rep in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(steps):
            env.step(acts[i % 4])
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps)
    out = {'ms': best, 'gbs': 165 * envs / best / 1e6, 'steps_per_s': envs * k / best * 1e3}
    try:        # the policy kernel of this build: speed and error against the PyTorch fp32 network
        pol = g.mlp_policy(10, 4, dtype=torch.float32, seed=5)
        for p in pol.net.parameters():
            p.data.mul_(3.0)
        fused = g.FusedMLPPolicy(env, pol.net)
        got = fused()
        with torch.no_grad():
            ref = pol.net(env.obs)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(20):
            fused()
        e1.record(); torch.cuda.synchronize()
        out.update(policy_ms=e0.elapsed_time(e1) / 20, policy_max_err=(got - ref).abs().max().item(),
                   policy_mean_err=(got - ref).abs().mean().item())
    except Exception as e:
        out['policy'] = repr(e)[:100]
    print(json.dumps(out))


def copy_peak():
    """This box's own copy bandwidth, measured the way MEASURED_PEAKS.json's hbm_gbs was
    (torch b.copy_(a) over 1 Gi bf16 elements, read + write bytes): burst best-of-10, then a
    0.5 s back-to-back loop."""
    import torch
    a = torch.empty(1 << 30, dtype=torch.bfloat16, device='cuda')
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    best = 1e9
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); b.copy_(a); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(800):
        b.copy_(a)
    e1.record(); torch.cuda.synchronize()
    gb = 2 * a.numel() * 2 / 1e9
    print(json.dumps({'copy_burst_gbs': gb / best * 1e3, 'copy_sustained_gbs': gb * 800 / e0.elapsed_time(e1) * 1e3}), flush=True)


def run(envs, k, stats):
    if k == 1:
        copy_peak()
    extra = sorted(f[4:-3] for f in os.listdir(VDIR) if f.startswith('lib_v') and f.endswith('.so'))
    for name in list(VARIANTS) + extra:
        lib = os.path.join(VDIR, 'lib_%s.so' % name)
        if not os.path.exists(lib):
            continue
        env = dict(os.environ, COPTER_B200_LIB=lib)
        r = subprocess.run([sys.executable, __file__, 'one', str(envs), str(k), str(stats)], env=env, capture_output=True, text=True)
        print('%-16s %s' % (name, r.stdout.strip() or r.stderr[-300:]), flush=True)


if __name__ == '__main__':
    a = sys.argv[1:]
    if a[0] == 'build':
        build()
    elif a[0] == 'one':
        time_one(int(a[1]), int(a[2]), 200 if int(a[2]) == 1 else 40, int(a[3]))
    else:
        envs = int(a[a.index('--envs') + 1]) if '--envs' in a else 1 << 24
        k = int(a[a.index('--k') + 1]) if '--k' in a else 1
        stats = int(a[a.index('--stats') + 1]) if '--stats' in a else 0
        run(envs, k, stats)
