"""
TEST INFRASTRUCTURE ONLY -- a float64 reference for the device's Gaussian variates and the log-probabilities built
on them (CPU, numpy): draw_variates<float> of csrc/copter_kernels.cu (the fused policy rollouts' exploration noise,
stream tag 2) and copter_policy_logp_kernel<A>.

The reference evaluates the documented definition exactly where the device is exact and in float64 where it is
not: Philox4x32-10 on counter (env_lo, env_hi, step, tag), key (seed_lo ^ step_hi, seed_hi); the uniforms rounded
to fp32 as the device rounds them, u1 = RN((c + 1) 2^-32) in (0, 1] and u2 = RN(c' 2^-32) in [0, 1]; then
r = sqrt(-2 ln u1), xi = (r cos 2 pi u2, r sin 2 pi u2) in float64.  The fp32 rounding of u1 is part of the
definition: near u1 -> 1 it alone moves xi by up to sqrt(2 2^-25) ~ 2.4e-4, far more than the device's transform
error, so a reference that skipped it could not hold the device to a tight bound.

    gaussian_variates(seed, env_ids, step, tag)   -> xi [n, 4] float64, r [n, 2] (the radius of pairs (0,1), (2,3))
    variate_bound(r)                              -> bound on |xi_device - xi| for a variate of a pair of radius r
    log_prob_bound(xi, std, A)                    -> bound on |logp_device - log_prob(xi, std, A)|
    log_prob(xi, std, A)                          -> -1/2 sum xi^2 - sum log std - A/2 log 2 pi in float64

A mutant (`mutant=`) models one plausible kernel bug; see MUTANTS.  tests/test_noise_oracle_cpu.py shows that each
misses these bounds by at least 2x on LOGP_SAMPLE, the sample tests/test_gpu_ppo_batch.py holds the device to.
"""
import numpy as np

from .copter_oracle import _U32, philox4x32_10

# ---- the device's error, per operation of draw_variates<float> ---------------------------------------------------
# __cosf / __sinf: absolute error 2^-21.41 on [-pi, pi] (CUDA C++ Programming Guide, "Intrinsic Functions", the
# single-precision table).  The folded angle reaches pi_f32 = pi + 8.7e-8 at u2 = 0 and u2 = 1, outside that range by
# less than the angle's own rounding; the GPU test holds the pairs with u2 at those edges to the bound separately.
SINCOS_ABS = 2.0 ** -21.41
# The folded angle RN(RN(2 pi)_f32 * RN(u2 - 1/2)) against 2 pi (u2 - 1/2): u2 - 1/2 is exact for u2 >= 1/4 and
# rounded to within 2^-26 below; the fp32 constant 6.2831855 is off 2 pi by 1.75e-7 (times |u2 - 1/2| <= 1/2); the
# product's rounding is within half an ulp of |angle| < 4, 2^-23.
TWO_PI_F32_ERR = abs(float(np.float32(2 * np.pi)) - 2 * np.pi)
ANGLE_ABS = 2 * np.pi * 2.0 ** -26 + 0.5 * TWO_PI_F32_ERR + 2.0 ** -23
DIR_ABS = SINCOS_ABS + ANGLE_ABS                 # |(cos, sin) device - (cos, sin) exact| per component: 6.6e-7
# logf: 1 ulp (CUDA C++ Programming Guide, "Mathematical Functions", maximum ulp error of logf over the full range).
# One ulp of ln u1 is at most 2^-23 of it, and -2 * logf is exact, so the radius sqrt(-2 L) moves by half that.
LOGF_ULPS = 1
# sqrt.approx.f32: 1 ulp, so at most 2^-23 relative (the same Guide's sqrtf entry for -prec-sqrt=false, which is
# what nvcc emits sqrt.approx.f32 for).
SQRT_REL = 2.0 ** -23
R_REL = 0.5 * LOGF_ULPS * 2.0 ** -23 + SQRT_REL  # relative error of the device radius
# The final product -r * cos: one fp32 rounding, half an ulp of the result, at most 2^-24 of it.
PRODUCT_REL = 2.0 ** -24

# ---- copter_policy_logp_kernel<A>'s own rounding ------------------------------------------------------------------
LOG_2PI = float(np.log(2 * np.pi))
LOG_2PI_F32 = float(np.float32(1.8378770664093453))    # the kernel's literal, an fp32 constant
HALF_ULP_REL = 2.0 ** -24                        # one fp32 rounding: at most half an ulp, 2^-24 of the value
SLACK = 1.0 + 2.0 ** -20                         # for "of the value" meaning the rounded value, and float64 evaluation

MUTANTS = {
    'u1_half_open': 'u1 = RN(c 2^-32) in [0, 1) instead of RN((c + 1) 2^-32) in (0, 1]',
    'sincos_swapped': 'cos and sin exchanged within a pair',
    'a2_pairs': 'the A = 2 variates taken as (xi0, xi2) instead of (xi0, xi1)',
    'logp_const_a4': 'the log-prob constant -(A/2) log 2 pi with A = 4 for every action size',
    'log2pi_5_digits': 'log 2 pi rounded to 1.8379 in the log-prob constant',
}
NOISE_MUTANTS = ('u1_half_open', 'sincos_swapped', 'a2_pairs')


def philox_counters(seed, env_ids, step, tag):
    """The four Philox4x32-10 words of (seed, env, step, tag) as the device draws them: uint32 arrays [n] each."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    n = env_ids.shape[0]
    seed, step = int(seed), int(step)
    return philox4x32_10(env_ids & _U32, env_ids >> np.uint64(32), np.full(n, step & 0xFFFFFFFF, np.uint64),
                         np.full(n, tag, np.uint64), (seed & 0xFFFFFFFF) ^ (step >> 32), (seed >> 32) & 0xFFFFFFFF)


def uniforms(c, mutant=None):
    """(u1, u2) [n, 2] float64 of the pairs (c0, c1), (c2, c3): u1 = RN_f32((c + 1) 2^-32), u2 = RN_f32(c' 2^-32).
    The integer is rounded to fp32 and scaled by a power of two, as __ull2float_rn / __uint2float_rn and 0x1p-32f do:
    one rounding of the exact value."""
    c = [np.asarray(x, np.uint64) for x in c]
    add = 0 if mutant == 'u1_half_open' else 1
    u1 = np.stack([(c[0] + np.uint64(add)).astype(np.float64), (c[2] + np.uint64(add)).astype(np.float64)], -1)
    u2 = np.stack([c[1].astype(np.float64), c[3].astype(np.float64)], -1)
    # (uint64 -> float64 is exact below 2^53; the scaling is exact; then one rounding to fp32)
    f = lambda x: (x * 2.0 ** -32).astype(np.float32).astype(np.float64)     # noqa: E731
    return f(u1), f(u2)


def gaussian_variates(seed, env_ids, step, tag=2, mutant=None):
    """xi [n, 4] float64 of (seed, env_ids, step, tag) by the device's definition, and r [n, 2], the radius of the
    pairs (xi0, xi1) and (xi2, xi3).  `mutant` one of NOISE_MUTANTS (or None)."""
    return variates_from_counters(philox_counters(seed, env_ids, step, tag), mutant)


def variates_from_counters(c, mutant=None):
    """gaussian_variates on the four Philox words c (philox_counters)."""
    u1, u2 = uniforms(c, mutant)
    with np.errstate(divide='ignore'):
        r = np.sqrt(-2.0 * np.log(u1))
    ang = 2 * np.pi * u2
    cs, sn = np.cos(ang), np.sin(ang)
    if mutant == 'sincos_swapped':
        cs, sn = sn, cs
    xi = np.empty((len(r), 4))
    xi[:, 0::2], xi[:, 1::2] = r * cs, r * sn
    if mutant == 'a2_pairs':
        xi = xi[:, [0, 2, 1, 3]]
    return xi, r


def variate_bound(r):
    """Upper bound on |xi_device - xi| for either variate of a pair of radius r (float64 array): the radius off by
    R_REL of itself, the direction by DIR_ABS, and the product's rounding.  About r * 9e-7: at the 6.7-sigma end of
    the range 6e-6, of which the kernel comment's 5e-7 on the direction (4e-6 there) is the larger part."""
    r = np.asarray(r, np.float64)
    r_dev = r * (1 + R_REL)
    return SLACK * (r * R_REL * (1 + DIR_ABS) + r * DIR_ABS + PRODUCT_REL * r_dev * (1 + DIR_ABS))


def pair_bound(r, A):
    """variate_bound of each of the first A variates [n, A] from the pair radii r [n, 2]."""
    return variate_bound(np.asarray(r)[:, [0, 0, 1, 1][:A]])


def log_prob(xi, std, A, mutant=None):
    """-1/2 sum_{j<A} xi_j^2 - sum log std_j - (A/2) log 2 pi in float64 [n] (std: the fp32 values, [A])."""
    xi = np.asarray(xi, np.float64)[:, :A]
    s = np.asarray(std, np.float32).astype(np.float64)[:A]
    a_const = 4 if mutant == 'logp_const_a4' else A
    l2p = 1.8379 if mutant == 'log2pi_5_digits' else LOG_2PI
    return -0.5 * (xi ** 2).sum(1) - np.log(s).sum() - 0.5 * a_const * l2p


def log_prob_bound(xi, std, A):
    """Upper bound [n] on |copter_policy_logp_kernel<A> - log_prob(xi, std, A)| with xi [n, 4] the reference
    variates (all four: the radius of each pair is hypot of its two):
      * the variates: sum_j |xi_j| d_j + d_j^2 / 2 with d_j = variate_bound of its pair;
      * q = sum xi_j^2 by an fmaf chain: A roundings of at most 2^-24 of q, halved by the -1/2;
      * c = -(A/2) RN(log 2 pi) - sum logf(std_j): the fp32 constant's error, 1 ulp of each logf (CUDA C++
        Programming Guide), A roundings of the running sum;
      * the final fmaf(-0.5, q, c): one rounding of the result."""
    xi = np.asarray(xi, np.float64)
    if xi.ndim != 2 or xi.shape[1] != 4:
        raise ValueError('xi must be the reference variates [n, 4]')
    r = np.stack([np.hypot(xi[:, 0], xi[:, 1]), np.hypot(xi[:, 2], xi[:, 3])], -1)
    xi = xi[:, :A]
    s = np.asarray(std, np.float32).astype(np.float64)[:A]
    d = pair_bound(r, A)
    var = (np.abs(xi) * d + 0.5 * d * d).sum(1)
    Q = ((np.abs(xi) + d) ** 2).sum(1)                           # bounds every partial sum of q on the device
    log_s = np.abs(np.log(s))
    S = 0.5 * A * LOG_2PI_F32 + log_s.sum()                      # bounds every partial sum of c
    q_round = 0.5 * A * HALF_ULP_REL * Q
    c_round = 0.5 * A * abs(LOG_2PI_F32 - LOG_2PI) + LOGF_ULPS * 2.0 ** -23 * log_s.sum() + A * HALF_ULP_REL * S
    out_round = HALF_ULP_REL * (0.5 * Q + S)
    return var + SLACK * (q_round + c_round + out_round)


# ---- the sample the log-prob kernel is held to (tests/test_gpu_ppo_batch.py) -------------------------------------
# 2^20 envs x 4 steps, an env offset and a first step above 2^32 (both high words in play), the seed chosen so that
# every action size sees each hard class of pair at least once (CLASSES).
LOGP_SAMPLE = dict(seed=0x5EED0000000000 + 25, env_offset=(3 << 32) + 12345, first_step=(5 << 32) + 77, n=1 << 20, T=4)
LOGP_STD = {1: (0.013,), 2: (0.02, 0.0071), 4: (0.004, 0.002, 0.001, 0.003)}   # per-component, different per j
LOGP_VARIANTS = {1: 'Lander1D', 2: 'Lander2D', 4: 'Lander3D'}
EDGE = 2.0 ** -20


def pair_classes(c):
    """[n, 2] bool masks of the hard pairs of the Philox words c (philox_counters): 'tail' (c < 2^12, r > 5.1),
    'u1_near_1' (u1 within 2^-20 of 1: tiny radii, where the fp32 rounding of u1 decides xi) and 'u2_edge' (u2 within
    2^-20 of 0, 1/2 or 1: the edges of the folded angle)."""
    u1, u2 = uniforms(c)
    c_first = np.stack([np.asarray(c[0], np.uint64), np.asarray(c[2], np.uint64)], -1)
    return {'tail': c_first < (1 << 12), 'u1_near_1': (1.0 - u1) <= EDGE,
            'u2_edge': (u2 <= EDGE) | (np.abs(u2 - 0.5) <= EDGE) | (1.0 - u2 <= EDGE)}


def sample_ids(sample=None):
    s = LOGP_SAMPLE if sample is None else sample
    return np.arange(s['n'], dtype=np.uint64) + np.uint64(s['env_offset'])
