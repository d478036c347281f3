"""CPU tests of oracle/noise_oracle.py, the float64 reference for the device's Gaussian variates and log-probabilities
that tests/test_gpu_ppo_batch.py holds the kernels to: it is source_actions' float64 restatement where that one is
exact, it bounds a float32 evaluation of the same transform, its constants are the kernel's, and -- the point of it --
each modelled kernel bug (mutant) misses its bounds by at least 2x on the sample the GPU test uses."""
import functools
import os
import re

import numpy as np
import pytest

from oracle import noise_oracle as no
from oracle.copter_oracle import source_actions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = os.path.join(ROOT, 'gym_copter_b200', 'csrc', 'copter_kernels.cu')
S = no.LOGP_SAMPLE


@functools.lru_cache(maxsize=None)
def counters(t):
    return no.philox_counters(S['seed'], no.sample_ids(), S['first_step'] + t, 2)


@functools.lru_cache(maxsize=None)
def variates(t, mutant=None):
    return no.variates_from_counters(counters(t), mutant)


def test_counters_are_the_philox_stream_of_the_action_sources():
    """The 'uniform' action source of tag 2 is c 2^-31 - 1, exactly: the same four words."""
    ids = no.sample_ids()[:4096]
    c = no.philox_counters(S['seed'], ids, S['first_step'], 2)
    u = source_actions(S['seed'], ids, S['first_step'], 'uniform', 1.0, 0.0, 4, np.float64, tag=2)
    assert np.array_equal(np.stack([x.astype(np.float64) * 2.0 ** -31 - 1.0 for x in c], -1), u)


def test_equals_float64_source_actions_where_the_uniforms_are_exact():
    """Where c + 1 < 2^24 and c' < 2^24 the fp32 rounding of both uniforms is the identity, so the reference is
    source_actions' float64 Box-Muller (which skips that rounding) -- to float64 rounding."""
    seen = 0
    for t in range(S['T']):
        c = [np.asarray(x, np.uint64) for x in counters(t)]
        exact = np.stack([(c[0] + np.uint64(1) < (1 << 24)) & (c[1] < (1 << 24)),
                          (c[2] + np.uint64(1) < (1 << 24)) & (c[3] < (1 << 24))], -1)
        rows = np.nonzero(exact.any(1))[0]
        xi, r = variates(t)
        ref = source_actions(S['seed'], no.sample_ids()[rows], S['first_step'] + t, 'randn', 1.0, 0.0, 4, np.float64, tag=2)
        for h in range(2):
            k = exact[rows, h]
            d = np.abs(xi[rows][k][:, 2 * h:2 * h + 2] - ref[k][:, 2 * h:2 * h + 2])
            assert np.all(d <= 1e-14 * r[rows, h][k][:, None]), d.max()
            seen += int(k.sum())
    assert seen >= 64, seen


def test_float32_evaluation_is_within_variate_bound():
    """numpy's float32 log / sqrt / sin / cos of the same uniforms stand in for a device-like evaluation of the
    transform (unfolded angle, library functions): within variate_bound of the reference everywhere, and not far
    inside it -- the bound is of the size of an fp32 evaluation's error."""
    worst = 0.0
    for t in range(S['T']):
        xi, r = variates(t)
        x32 = source_actions(S['seed'], no.sample_ids(), S['first_step'] + t, 'randn', 1.0, 0.0, 4, np.float32, tag=2)
        ratio = np.abs(x32.astype(np.float64) - xi) / no.pair_bound(r, 4)
        ok = np.where(np.isnan(ratio), True, ratio <= 1.0)       # r = 0 (u1 = 1): both give 0
        assert ok.all(), float(np.nanmax(ratio))
        worst = max(worst, float(np.nanmax(ratio)))
    assert worst > 0.1, worst


def test_constants_are_the_kernels():
    src = open(KERNELS).read()
    body = src[src.index('void draw_variates('):src.index('// Command vector of (env, step)')]
    assert '6.283185307179586f * (u2 - 0.5f)' in body
    assert '__ull2float_rn((unsigned long long)c[2 * h] + 1ull) * 0x1p-32f' in body
    assert '__uint2float_rn(c[2 * h + 1]) * 0x1p-32f' in body
    assert 'sqrt.approx.f32' in body and '-2.0f * logf(u1)' in body
    assert 'xi[2 * h] = -r * __cosf(ang); xi[2 * h + 1] = -r * __sinf(ang);' in body
    lit = re.search(r'float c = -0\.5f \* \(float\)A \* ([0-9.]+)f;', src).group(1)
    assert float(np.float32(lit)) == no.LOG_2PI_F32 and abs(float(lit) - no.LOG_2PI) < 1e-15
    # the kernel comment's claim -- 5e-7 on the direction, <= 4e-6 on a variate at 6.7 sigma -- lies inside the bound
    assert 5e-7 < no.DIR_ABS < 1e-6 and 4e-6 < no.variate_bound(6.7) < 8e-6


def test_log_prob_bound_covers_an_fp32_evaluation():
    """The log-prob kernel's arithmetic replayed in numpy float32 (its constant, logf of each std, the fmaf chain
    rounded per step) on the float32 variates: within log_prob_bound of the float64 formula on the reference."""
    for A, std in no.LOGP_STD.items():
        s32 = np.asarray(std, np.float32)
        c = np.float32(-0.5) * np.float32(A) * np.float32(no.LOG_2PI_F32)
        for j in range(A):
            c = np.float32(c - np.log(s32[j]))
        for t in range(S['T']):
            xi, r = variates(t)
            x32 = source_actions(S['seed'], no.sample_ids(), S['first_step'] + t, 'randn', 1.0, 0.0, 4, np.float32, tag=2)
            q = np.zeros(len(x32), np.float32)
            for j in range(A):
                q = (x32[:, j].astype(np.float64) ** 2 + q).astype(np.float32)
            got = (-0.5 * q.astype(np.float64) + float(c)).astype(np.float32).astype(np.float64)
            ratio = np.abs(got - no.log_prob(xi, s32, A)) / no.log_prob_bound(xi, s32, A)
            assert ratio.max() <= 1.0, (A, t, float(ratio.max()))


# Which check must catch each mutant: ('noise', A) -- the variates a rollout of action size A draws; ('logp', A) -- the
# log-prob kernel of action size A.  The swap keeps xi0^2 + xi1^2 and so only the A = 1 log-prob sees it.
SEPARATED_BY = {'u1_half_open': [('noise', 1), ('noise', 2), ('noise', 4), ('logp', 1), ('logp', 2), ('logp', 4)],
                'sincos_swapped': [('noise', 1), ('noise', 2), ('noise', 4), ('logp', 1)],
                'a2_pairs': [('noise', 2), ('logp', 2)],
                'logp_const_a4': [('logp', 1), ('logp', 2)],
                'log2pi_5_digits': [('logp', 1), ('logp', 2), ('logp', 4)]}


def mutant_ratio(mutant, what, A):
    """max over the sample of |mutant - reference| / bound (inf where the bound is 0 and the mutant differs)."""
    worst = 0.0
    std = np.asarray(no.LOGP_STD[A], np.float32)
    for t in range(S['T']):
        xi, r = variates(t)
        xm = variates(t, mutant)[0] if mutant in no.NOISE_MUTANTS else xi
        if what == 'noise':
            d, b = np.abs(xm[:, :A] - xi[:, :A]), no.pair_bound(r, A)
        else:
            lm = no.log_prob(xm, std, A, None if mutant in no.NOISE_MUTANTS else mutant)
            d, b = np.abs(lm - no.log_prob(xi, std, A)), no.log_prob_bound(xi, std, A)
        with np.errstate(divide='ignore', invalid='ignore'):
            ratio = np.where(d == 0, 0.0, np.where(np.isfinite(d), d / b, np.inf))
        worst = max(worst, float(np.max(ratio)))
    return worst


@pytest.mark.parametrize('mutant', list(no.MUTANTS))
def test_every_mutant_misses_its_bound_by_two(mutant):
    """|mutant - reference| >= 3 x bound somewhere in the GPU test's sample, for every check that SEPARATED_BY
    assigns to the mutant: a kernel with that bug, itself within one bound of the mutant, misses the bound by at
    least 2x (triangle inequality)."""
    for what, A in SEPARATED_BY[mutant]:
        r = mutant_ratio(mutant, what, A)
        print('%s %s A=%d: misses the bound by %.3g x' % (mutant, what, A, r - 1))
        assert r >= 3, (mutant, what, A, r)


def test_sample_holds_every_hard_class():
    """The seed of LOGP_SAMPLE is chosen so that every action size sees each hard class of pair at least once."""
    for A in (1, 2, 4):
        pairs = 1 if A < 4 else 2
        for k in ('tail', 'u1_near_1', 'u2_edge'):
            assert sum(int(no.pair_classes(counters(t))[k][:, :pairs].sum()) for t in range(S['T'])) > 0, (A, k)
