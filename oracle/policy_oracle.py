"""
TEST INFRASTRUCTURE ONLY -- a float64 model of the two policy kernels' own rounding (CPU, numpy):
csrc/copter_policy.cuh (warp-level mma.sync, kind 'mma') and csrc/copter_policy_tc.cuh (tcgen05 / TMEM,
kind 'tc').  Both evaluate the tanh MLP O -> 64 -> 64 -> A of FusedMLPPolicy from the fp32 state.

The model rounds exactly where a kernel rounds and nowhere else: operands to bf16 / fp16 (round to nearest
even, from the fp32 value the kernel holds), hidden activations to 16 bits after the tanh, and the polynomial
tanh of the tcgen05 kernel as its fp32 Horner chain.  Sums are exact (float64) and tanh is exact, so what is
left between a kernel and its model is the fp32 accumulation inside the MMAs and the error of MUFU.TANH
(tanh.approx.f32), which `ceiling` bounds per element and `noisy_model` draws at random.

    model(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset, mutant=None) -> [N, A]
    ceiling(...)       per-element upper bound on |kernel - model| (first-order propagation through |W|)
    noisy_model(...)   the model with every MUFU tanh multiplied by 1 + u, u ~ U(-2^-11, 2^-11) (seeded)
    tolerance(kind, case)   2 x the worst dist(noisy_model, model) over a few noise seeds
    cases()            the deterministic inputs shared by tests/test_policy_oracle_cpu.py and
                       tests/test_gpu_policy_numerics.py

A mutant (`mutant=`) models one plausible kernel bug; see MUTANTS.
"""
import numpy as np

# Variant<> of csrc/copter_core.h: first observation component, O, A
VARIANTS = {'Lander3D': (0, 10, 4), 'Lander2D': (2, 6, 2), 'Lander1D': (4, 2, 1), 'Hover3D': (0, 12, 4),
            'Hover2D': (2, 6, 2), 'Hover1D': (4, 2, 1), 'Takeoff': (0, 10, 4)}
HIDDEN = 64

# csrc/copter_policy_tc.cuh: kPolyLanes, kTanhClamp, tanh_poly_coef (tests/test_policy_oracle_cpu.py checks
# that these are the header's values)
K_POLY_LANES = 4
K_TANH_CLAMP = np.float32(3.25)
TANH_POLY_COEF = tuple(np.float32(c) for c in (9.977270291e-01, -3.117916466e-01, 9.229137325e-02, -1.838625564e-02,
                                               2.184749761e-03, -1.380842544e-04, 3.552717362e-06))

MUFU_REL = 2.0 ** -11          # relative error bound of tanh.approx.f32 (PTX ISA); the one constant the B200 confirms
ACC_REL = 2.0 ** -22           # per accumulated term, times the sum of |terms|: generous for the MMAs' fp32 adders
POLY_EVAL = 2.0 ** -19         # absolute bound of the fp32 rounding inside the Horner chain

MUTANTS = {
    'bf16_hidden': 'tc: hidden activations rounded to bf16 instead of fp16',
    'no_bias_lo1': 'tc: layer-1 bias without its bf16 lo half',
    'no_bias_lo2': 'tc: layer-2 bias without its fp16 lo half',
    'no_bias_lo3': 'tc: layer-3 bias without its fp16 lo half',
    'poly_cols_shifted': 'tc: the polynomial on columns j % 4 == 1 instead of j % 4 == 0',
    'poly_none': 'tc: MUFU tanh on every hidden column',
    'no_clamp': 'tc: the polynomial without its clamp to +-kTanhClamp',
    'obs_shift': 'both: observation read from component first + 1',
    'rounded_bias': 'mma: biases rounded to bf16 instead of exact fp32 accumulator values',
    'hidden_chunk_swap': 'both: columns 0-7 and 8-15 of the first K chunk of layer 2 exchanged (a wrong LBO)',
}
MUTANT_KINDS = {'bf16_hidden': ('tc',), 'no_bias_lo1': ('tc',), 'no_bias_lo2': ('tc',), 'no_bias_lo3': ('tc',),
                'poly_cols_shifted': ('tc',), 'poly_none': ('tc',), 'no_clamp': ('tc',), 'obs_shift': ('tc', 'mma'),
                'rounded_bias': ('mma',), 'hidden_chunk_swap': ('tc', 'mma')}


# ---- rounding (round to nearest even) -------------------------------------------------------------------------

def f32(x):
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float64)


def bf16(x):
    """fp32 -> bf16 -> float64 (the input is first rounded to fp32, as the kernel holds it)."""
    x32 = np.asarray(x, np.float64).astype(np.float32)
    u = x32.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000).astype(np.uint32)
    out = r.view(np.float32).astype(np.float64)
    return np.where(np.isnan(x32), np.nan, out)


def f16(x):
    """fp32 -> fp16 -> float64."""
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float16).astype(np.float64)


def _ulp(v, fmt):
    """ulp of a 16-bit value of magnitude v (array, >= 0)."""
    mant, emin = (10, -14) if fmt == 'f16' else (7, -126)
    e = np.floor(np.log2(np.maximum(v, 2.0 ** (emin - 1))))
    return 2.0 ** (np.maximum(e, emin) - mant)


def fmaf(a, b, c):
    """fp32 fmaf(a, b, c), exactly: the product of two fp32 values is exact in float64, so the float64 sum is off
    only by its own rounding; where it lands exactly halfway between two fp32 values, the sign of that rounding
    error (TwoSum) decides the fp32 result."""
    a, b, c = (np.asarray(v, np.float64) for v in (a, b, c))
    s = a * b
    hi = s + c
    tie = (hi.view(np.int64) & 0x1FFFFFFF) == 0x10000000
    if tie.any():
        bb = hi - s
        lo = (s - (hi - bb)) + (c - bb)
        hi = np.where(tie & (lo != 0), np.nextafter(hi, np.where(lo > 0, np.inf, -np.inf)), hi)
    return f32(hi)


def tanh_poly(x, clamp=True):
    """tanh_fma of copter_policy_tc.cuh on the fp32 value x: clamp, u = x * x, Horner with fmaf, times x."""
    x = f32(x)
    if clamp:
        x = np.minimum(np.maximum(x, -float(K_TANH_CLAMP)), float(K_TANH_CLAMP))
    u = f32(x * x)
    p = np.full_like(x, float(TANH_POLY_COEF[6]))
    for k in range(5, -1, -1):
        p = fmaf(p, u, float(TANH_POLY_COEF[k]))
    return f32(p * x)


def poly_columns(n=HIDDEN, shift=0):
    j = (np.arange(n) - shift) % 16
    return (j * K_POLY_LANES) % 16 < K_POLY_LANES


# ---- the model --------------------------------------------------------------------------------------------------

def _split(b, rnd):
    hi = rnd(b)
    return hi + rnd(f32(f32(b) - hi))


def _forward(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset, mutant=None, rng=None,
             exact=False):
    if kind not in ('tc', 'mma'):
        raise ValueError(kind)
    if mutant is not None and kind not in MUTANT_KINDS[mutant]:
        raise ValueError('mutant %s does not apply to kind %s' % (mutant, kind))
    first, O, A = VARIANTS[variant]
    if mutant == 'obs_shift' and first + O + 1 <= 12:
        first += 1
    W1, b1, W2, b2, W3, b3 = (np.asarray(v, np.float64) for v in (W1, b1, W2, b2, W3, b3))
    x = np.asarray(state_rows, np.float64)[:, first:first + O]
    ident = lambda v: v                     # noqa: E731
    if exact:
        r_in = r_w1 = r_w = r_hid = r32 = ident
        b1q, b2q, b3q = b1, b2, b3
    elif kind == 'mma':
        r_in = r_w1 = r_w = r_hid = bf16
        r32 = f32
        rb = bf16 if mutant == 'rounded_bias' else f32
        b1q, b2q, b3q = rb(b1), rb(b2), rb(b3)
    else:
        r_in = r_w1 = bf16
        r_w = f16
        r_hid = bf16 if mutant == 'bf16_hidden' else f16
        r32 = f32
        b1q = bf16(b1) if mutant == 'no_bias_lo1' else _split(b1, bf16)
        b2q = f16(b2) if mutant == 'no_bias_lo2' else _split(b2, f16)
        b3q = f16(b3) if mutant == 'no_bias_lo3' else _split(b3, f16)
    if exact or kind == 'mma' or mutant == 'poly_none':
        poly = np.zeros(HIDDEN, bool)
    else:
        poly = poly_columns(shift=1 if mutant == 'poly_cols_shifted' else 0)

    def mufu(z):
        t = np.tanh(z)
        if rng is not None:
            t = t * (1.0 + rng.uniform(-MUFU_REL, MUFU_REL, t.shape))
        return r32(t)

    def act(z):
        t = mufu(z)
        if poly.any():
            t[:, poly] = tanh_poly(z[:, poly], clamp=mutant != 'no_clamp')
        return t

    tr = {'poly': poly, 'kind': kind, 'exact': exact}
    xq = r_in(r32(x))
    W1q, W2q, W3q = r_w1(W1), r_w(W2), r_w(W3)
    z1 = xq @ W1q.T + b1q
    t1 = act(z1)
    h1 = r_hid(t1)
    if mutant == 'hidden_chunk_swap':
        h1 = h1[:, np.r_[8:16, 0:8, 16:HIDDEN]]
    z2 = h1 @ W2q.T + b2q
    t2 = act(z2)
    h2 = r_hid(t2)
    z3 = h2 @ W3q.T + b3q
    t3 = mufu(z3)
    out = (out_offset + out_scale * t3) if exact else fmaf(np.float32(out_scale), t3, np.float32(out_offset))
    tr.update(xq=xq, W=(W1q, W2q, W3q), b=(b1q, b2q, b3q), z=(z1, z2, z3), t=(t1, t2, t3), h=(h1, h2), out=out)
    return out, tr


def _forward_quiet(*a, **k):
    with np.errstate(over='ignore', invalid='ignore'):      # the no_clamp mutant overflows
        return _forward(*a, **k)


def model(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset, mutant=None, exact=False):
    """The kernel of `kind` ('tc' or 'mma') on fp32 state rows [N, 12]: actions [N, A], float64.
    exact=True: no rounding anywhere and exact tanh on every column (the float64 network)."""
    return _forward_quiet(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset, mutant, exact=exact)[0]


def noisy_model(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset, seed=0, mutant=None):
    """The model with each MUFU tanh (every tanh of the 'mma' kernel, the non-polynomial hidden columns and the
    output of the 'tc' kernel) multiplied by 1 + u, u uniform in +-2^-11 from a seeded generator."""
    rng = np.random.default_rng(seed)
    return _forward_quiet(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset, mutant, rng=rng)[0]


def _poly_slope_excess():
    """max |P'(x) - tanh'(x)| on [0, kTanhClamp] (float64 derivative of the polynomial), with a margin."""
    x = np.linspace(0, float(K_TANH_CLAMP), 200001)
    u = x * x
    c = [float(v) for v in TANH_POLY_COEF]
    dp = sum((2 * k + 1) * c[k] * u ** k for k in range(7))
    return 1.25 * float(np.max(np.abs(dp - 1.0 / np.cosh(x) ** 2)))


POLY_SLOPE_EXCESS = _poly_slope_excess()


def _sech2_bound(z, e):
    """max of tanh' over [|z| - e, |z| + e]"""
    return 1.0 / np.cosh(np.clip(np.abs(z) - e, 0.0, 300.0)) ** 2


def ceiling(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset):
    """Per-element upper bound on |kernel - model| [N, A], from first-order propagation through |W|:
      * fp32 accumulation of the k terms of a pre-activation adds at most k * 2^-22 * sum |terms|;
      * a pre-activation off by e moves tanh by at most e * max tanh' on [|z| - e, |z| + e], the polynomial by
        that plus its slope excess and its own fp32 rounding -- or not at all where both ends are clamped;
      * MUFU.TANH adds 2^-11 of the value;
      * the 16-bit rounding after it passes that on and may flip by one ulp (not where nothing moved)."""
    out, tr = _forward(kind, state_rows, variant, W1, b1, W2, b2, W3, b3, out_scale, out_offset)
    W1q, W2q, W3q = tr['W']
    b1q, b2q, b3q = tr['b']
    z1, z2, z3 = tr['z']
    h1, h2 = tr['h']
    poly = tr['poly']
    fmt = 'f16' if kind == 'tc' else 'bf16'
    clamp = float(K_TANH_CLAMP)
    nb = 2 if kind == 'tc' else 1           # bias terms of a pre-activation (hi + lo, or the accumulator's start)

    def acc(a_abs, W, b, k):
        return k * ACC_REL * (a_abs @ np.abs(W).T + nb * np.abs(b))

    def hidden(z, e_z):
        t = np.tanh(z)
        L = _sech2_bound(z, e_z)
        e_t = L * e_z + MUFU_REL * (np.abs(t) + L * e_z) + 2.0 ** -24 * np.abs(t)
        if poly.any():
            zp, ep = z[:, poly], e_z[:, poly]
            ep_t = (L[:, poly] + POLY_SLOPE_EXCESS) * ep + 2 * POLY_EVAL
            both_clamped = (np.abs(zp) - ep > clamp)
            e_t[:, poly] = np.where(both_clamped, 0.0, ep_t)
        return np.where(e_t > 0, e_t + _ulp(np.abs(t) + e_t + 2.5e-3, fmt), 0.0)

    xa = np.abs(tr['xq'])
    e_z1 = acc(xa, W1q, b1q, W1q.shape[1] + nb)
    e_h1 = hidden(z1, e_z1)
    e_z2 = np.abs(W2q) @ e_h1.T
    e_z2 = e_z2.T + acc(np.abs(h1) + e_h1, W2q, b2q, HIDDEN + nb)
    e_h2 = hidden(z2, e_z2)
    e_z3 = (np.abs(W3q) @ e_h2.T).T + acc(np.abs(h2) + e_h2, W3q, b3q, HIDDEN + nb)
    t3 = np.tanh(z3)
    L3 = _sech2_bound(z3, e_z3)
    e_t3 = L3 * e_z3 + MUFU_REL * (np.abs(t3) + L3 * e_z3) + 2.0 ** -24 * np.abs(t3)
    big = np.maximum(np.abs(out), abs(out_offset)) + abs(out_scale)
    return abs(out_scale) * e_t3 + 2.0 ** -22 * big


# ---- statistics and tolerances ----------------------------------------------------------------------------------

def dist(a, b):
    """(mean, 99.9th percentile) of |a - b| per output column: two arrays [A]."""
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
    return d.mean(0), np.percentile(d, 99.9, axis=0)


def case_args(case):
    return (case['state'], case['variant']) + tuple(case['weights']) + (case['out_scale'], case['out_offset'])


def tolerance(kind, case, seeds=(0, 1, 2, 3)):
    """tol = 2 x the worst dist(noisy_model, model) over the noise seeds: (mean [A], p99.9 [A])."""
    ref = model(kind, *case_args(case))
    worst_m, worst_p = None, None
    for s in seeds:
        m, p = dist(noisy_model(kind, *case_args(case), seed=s), ref)
        worst_m = m if worst_m is None else np.maximum(worst_m, m)
        worst_p = p if worst_p is None else np.maximum(worst_p, p)
    return 2 * worst_m, 2 * worst_p


def ratio(d, tol):
    """The worst of dist / tol over both statistics and all columns (inf where a distance is not finite)."""
    r = np.concatenate([d[0] / tol[0], d[1] / tol[1]])
    return float(np.max(np.where(np.isfinite(r), r, np.inf)))


def applies(mutant, kind, case):
    """Whether `case` is one that must separate `mutant` of `kind` from the model (SEPARATED_BY)."""
    if kind not in MUTANT_KINDS[mutant]:
        return False
    first, O, _ = VARIANTS[case['variant']]
    if mutant == 'obs_shift' and first + O + 1 > 12:
        return False
    return case['probe'] in SEPARATED_BY[mutant]


# The cases that separate each mutant: None = the dense networks, 0..3 = the probe designs.  The subtle mutants move
# a dense network's outputs by less than the MUFU error does (a 16-bit rounding of a bias, the polynomial's 2e-3 on a
# quarter of the columns); the probes single out the path they change.
SEPARATED_BY = {'bf16_hidden': (1, 2), 'no_bias_lo1': (0,), 'no_bias_lo2': (1,), 'no_bias_lo3': (2,),
                'poly_cols_shifted': (1, 2), 'poly_none': (1, 2), 'no_clamp': (None, 0, 1, 2, 3),
                'obs_shift': (None,), 'rounded_bias': (1, 2), 'hidden_chunk_swap': (None,)}


def case_model(kind, case, mutant=None):
    return model(kind, *case_args(case), mutant=mutant)


def case_ceiling(kind, case):
    return ceiling(kind, *case_args(case))


# ---- shared inputs ----------------------------------------------------------------------------------------------

# per-component scales of the dense state rows (X, dX, Y, dY, Z, dZ, Phi, dPhi, Theta, dTheta, Psi, dPsi): the ranges
# of policy rollouts, a little wider
_STATE_SCALE = np.array([4.0, 3.0, 4.0, 3.0, 4.0, 3.0, 0.6, 2.0, 0.6, 2.0, 1.5, 2.0])
_STATE_SHIFT = np.array([0.0, 0.0, 0.0, 0.0, -5.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0])
DENSE_ROWS = 1 << 16


def dense_states(n, seed):
    """[n + 80, 12] fp32: n rows from a seeded distribution over rollout ranges, then 64 rows with a component
    at +-1e4 and 16 rows of exact zeros."""
    rng = np.random.default_rng(seed)
    s = rng.standard_normal((n, 12)) * _STATE_SCALE + _STATE_SHIFT
    big = rng.standard_normal((64, 12)) * _STATE_SCALE
    big[np.arange(64), np.arange(64) % 12] = np.where(np.arange(64) % 2 == 0, 1e4, -1e4)
    return np.concatenate([s, big, np.zeros((16, 12))]).astype(np.float32)


def dense_weights(variant, mult, seed=5):
    """mlp_policy(O, A, seed) weights times `mult`, fp32 numpy (W1, b1, W2, b2, W3, b3)."""
    import torch
    from gym_copter_b200.rollout import mlp_policy
    _, O, A = VARIANTS[variant]
    net = mlp_policy(O, A, dtype=torch.float32, device='cpu', seed=seed).net
    return tuple((p.detach() * mult).numpy().astype(np.float32) for p in net.parameters())


# Probe networks (Lander3D, 4 actions).  W1 one-hot (hidden j reads observation component j mod O), W2 the identity,
# W3 one-hot with weight 0.5 (output a of probe m reads hidden column 4 m + a), every observation component of row r
# equal to x_r, x_r swept over [-6, 6].  Each output then depends on ONE path through both hidden layers, and output
# 0 of every probe on a polynomial column (j % 4 == 0) in both layers: deterministic up to the output's MUFU tanh.
# The 16 groups of 4 hidden columns (probe m reads group m) have one of four bias designs (m % 4):
#   0  layer-1 bias in [4, 8) with a large bf16 lo half: layer 1 swept across the clamp; the other layers mild
#   1  layer-1 bias +-10 (layer 1 saturated: h1 = +-f16(P(3.25)) on every row), layer-2 bias just under 1.25 in
#      magnitude with a large fp16 lo half, layer 3 cancelling layer 2 to |z3| ~ 0.01 (MUFU error ~ 0)
#   2  layer 2 saturated through a bias of +-5, layer-3 bias just under 0.5 in magnitude with a large fp16 lo half,
#      cancelling to |z3| ~ 0.01: output 0 pins P(3.25) and the layer-3 lo half
#   3  mild biases with lo halves in all layers: a plain sweep of every layer
PROBE_ROWS = 4096


def _with_lo(hi, frac, ulp):
    return np.float32(hi + frac * ulp)


def probe_bias():
    """(b1 [64], b2 [64]) shared by the probes, fp32."""
    b1 = np.zeros(HIDDEN, np.float32)
    b2 = np.zeros(HIDDEN, np.float32)
    for j in range(HIDDEN):
        g, a = j // 4, j % 4
        sg = 1.0 if (g // 4 + a) % 2 == 0 else -1.0
        mode = g % 4
        if mode == 0:
            b1[j] = sg * _with_lo(4.0 + 0.75 * a, 0.45, 2.0 ** -5)
            b2[j] = -sg * _with_lo(0.25, 0.4, 2.0 ** -12)
        elif mode == 1:
            b1[j] = sg * 10.0
            b2[j] = -sg * _with_lo(1.25 - 2.0 ** -9 * (g // 4), 0.45, 2.0 ** -10)
        elif mode == 2:
            b1[j] = sg * _with_lo(0.5 + 0.25 * a, 0.4, 2.0 ** -8)
            b2[j] = sg * 5.0
        else:
            b1[j] = -sg * _with_lo(1.0 + 0.5 * a, 0.45, 2.0 ** -7)
            b2[j] = sg * _with_lo(0.5, 0.45, 2.0 ** -11)
    return b1, b2


def probe_states():
    x = np.linspace(-6.0, 6.0, PROBE_ROWS)
    return np.repeat(x[:, None], 12, axis=1).astype(np.float32)


def probe_case(m):
    """Probe network m (0..15): reads hidden columns 4 m .. 4 m + 3."""
    _, O, A = VARIANTS['Lander3D']
    W1 = np.zeros((HIDDEN, O), np.float32)
    W1[np.arange(HIDDEN), np.arange(HIDDEN) % O] = 1.0
    W2 = np.eye(HIDDEN, dtype=np.float32)
    W3 = np.zeros((A, HIDDEN), np.float32)
    W3[np.arange(A), 4 * m + np.arange(A)] = 0.5
    b1, b2 = probe_bias()
    b3 = np.zeros(A, np.float32)
    if m % 4 in (1, 2):
        # cancel layer 2 (constant on every row in these designs) to |z3| ~ 0.01, with the lo half of b3 large
        # where it is the design's target
        h2 = _forward('tc', probe_states()[:1], 'Lander3D', W1, b1, W2, b2, W3, b3, 1.0, 0.0)[1]['h'][1][0, 4 * m:4 * m + A]
        for a in range(A):
            target = -0.5 * h2[a] + (0.01 if a % 2 == 0 else -0.01)
            if m % 4 == 2:
                hi = float(f16(target))
                ulp = float(_ulp(np.array([abs(hi)]), 'f16')[0])
                b3[a] = np.float32(hi - np.sign(hi) * 0.45 * ulp)
            else:
                b3[a] = np.float32(target)
    elif m % 4 == 0:
        b3[:] = [0.02, -0.03, 0.05, -0.07]
    return dict(name='probe%02d' % m, variant='Lander3D', weights=(W1, b1, W2, b2, W3, b3),
                state=probe_states(), out_scale=1.0, out_offset=0.0, probe=m % 4)


def dense_case(variant, mult):
    return dict(name='%s_x%d' % (variant, mult), variant=variant, weights=dense_weights(variant, mult),
                state=dense_states(DENSE_ROWS, seed=100 + 10 * list(VARIANTS).index(variant) + mult),
                out_scale=0.5, out_offset=0.25, probe=None)


def cases():
    """Every shared case: the dense networks (all 7 variants, mlp_policy weights x1 and x3) and the 16 probes."""
    for variant in VARIANTS:
        for mult in (1, 3):
            yield dense_case(variant, mult)
    for m in range(16):
        yield probe_case(m)
