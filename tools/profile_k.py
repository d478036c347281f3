"""Developer tool: a few K-fused step launches on a desynchronised batch, for `ncu -k regex:copter_step`.
    python tools/profile_k.py [k] [envs]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gym_copter_b200 as g  # noqa: E402

k = int(sys.argv[1]) if len(sys.argv) > 1 else 16
n = int(sys.argv[2]) if len(sys.argv) > 2 else 1 << 24
env = g.LanderVec(n, seed=1, k_substeps=k)
env.reset()
env.rollout(997, source='randn')
a = 1.625e-2 * torch.randn((n, 4), device='cuda')
for _ in range(4):
    env.step(a)
torch.cuda.synchronize()
