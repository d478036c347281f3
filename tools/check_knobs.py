#!/usr/bin/env python3
"""
Developer tool: cross-compiles the library once per A/B knob combination of the policy kernels
(no GPU needed) so that the alternative shapes kept for measurements -- tcgen05 slots and splits,
polynomial tanh, cluster launch control, the warp-MMA kernel -- do not rot.  Runs the builds in
parallel; prints one line per combination.

    python tools/check_knobs.py
"""
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gym_copter_b200.build import NVCC_FLAGS          # noqa: E402
SRC = os.path.join(ROOT, 'gym_copter_b200', 'csrc', 'copter_kernels.cu')
COMBOS = [
    ['-DCOPTER_POLICY_POLY_MASK=0x88', '-DCOPTER_POLICY_MT=1'],
    ['-DCOPTER_POLICY_POLY_MASK=0xff', '-DCOPTER_POLICY_POLY_F32X2=0', '-DCOPTER_POLICY_TANH_BF16X2=1'],
    ['-DCOPTER_POLICY_TC_SLOTS=2', '-DCOPTER_POLICY_TC_SPLIT=2', '-DCOPTER_POLICY_TC_POLY=0'],        # (no tcgen05 fused rollout in these shapes)
    ['-DCOPTER_POLICY_TC_POLY=8', '-DCOPTER_POLICY_ROLLOUT_TC_CTAS_PER_SM=3', '-DCOPTER_POLICY_TC=0'],
    ['-DCOPTER_POLICY_TC_CLC=0', '-DCOPTER_POLICY_TC_ONES_ROWS=128', '-DCOPTER_POLICY_TC_CTAS_PER_SM=5', '-DCOPTER_POLICY_ROLLOUT_TC=0'],
    ['-DCOPTER_POLICY_TC_WAIT=2'],
    ['-DCOPTER_POLICY_TC_F16=2', '-DCOPTER_POLICY_TC_POLY=6'],
]


def main():
    with tempfile.TemporaryDirectory() as tmp:
        procs = []
        for i, flags in enumerate(COMBOS):
            cmd = ['nvcc'] + NVCC_FLAGS + flags + ['-o', os.path.join(tmp, 'lib_%d.so' % i), SRC]
            procs.append((flags, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        bad = 0
        for flags, p in procs:
            out, _ = p.communicate()
            errors = [line for line in out.splitlines() if 'error' in line.lower()]
            print('%-90s %s' % (' '.join(flags), 'ok' if p.returncode == 0 else 'FAILED: ' + ' | '.join(errors[:3])))
            bad += p.returncode != 0
    sys.exit(1 if bad else 0)


if __name__ == '__main__':
    main()
