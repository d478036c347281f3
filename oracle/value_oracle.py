"""
TEST INFRASTRUCTURE ONLY -- the value head of the tcgen05 kernel (copter_value_mlp_f32: csrc/copter_policy_tc.cuh with
ObsRows and ValueHead) in the float64 rounding model of policy_oracle.py (CPU, numpy).

The critic O -> 64 -> 64 -> 1 rounds exactly as the tcgen05 policy kernel does up to layer 3 (bf16 observation and
layer-1 weights, biases as 16-bit hi + lo, tanh.approx / the FMA polynomial on the same hidden columns, fp16 hidden
activations and layer-2 / -3 weights); its output is layer 3's fp32 accumulator -- no tanh, scale or offset.  So the
model's value is the exact layer-3 pre-activation of the rounded operands, and what is left between the kernel and
the model is the fp32 accumulation and the hidden layers' MUFU.TANH error, which `ceiling` bounds per row.

    model(obs, variant, W1, b1, W2, b2, W3, b3, exact=False) -> [N]   (W3 [1][64], b3 [1]; obs [N, O] fp32)
    ceiling(...)                                              -> [N]   upper bound on |kernel - model|
    scale(...)                                                -> [N]   sum_j |W3_j| |h2_j| + |b3| of the float64 network
    REL_TO_NETWORK     |model - float64 network| <= REL_TO_NETWORK * scale on the dense cases (mlp_policy weights; the
                       probes are built to single out one rounding path each and cancel layer 3 to |z3| ~ 0.01)
    critic_cases()     the shared policy cases (policy_oracle.cases()) with the critic weights of each: layer 3 is
                       the policy's output row 0 (for a probe: the path through the polynomial columns)
"""
import numpy as np

from . import policy_oracle as po

# The rounded network against the float64 one, relative to sum |W3| |h2| + |b3|: bf16 rows and layer-1 weights
# (2^-9 each) and the polynomial's 2e-3 on a quarter of the hidden columns dominate (worst dense case: 6.9e-3).
# tests/test_value_oracle_cpu.py shows every dense case within it; the GPU tests hold the kernel to it against a
# PyTorch fp32 critic.
REL_TO_NETWORK = 2.0 ** -5


def _state(obs, variant):
    """[N, O] observation rows -> the [N, 12] state rows policy_oracle's model reads them from."""
    first, O, _ = po.VARIANTS[variant]
    obs = np.asarray(obs, np.float64)
    if obs.shape[1] != O:
        raise ValueError('obs must be [N, %d] for %s' % (O, variant))
    s = np.zeros((obs.shape[0], 12))
    s[:, first:first + O] = obs
    return s


def _trace(obs, variant, W1, b1, W2, b2, W3, b3, exact=False):
    if np.asarray(W3).shape[0] != 1 or np.asarray(b3).shape != (1,):
        raise ValueError('the value head has one output: W3 [1][64], b3 [1]')
    return po._forward_quiet('tc', _state(obs, variant), variant, W1, b1, W2, b2, W3, b3, 1.0, 0.0, exact=exact)[1]


def model(obs, variant, W1, b1, W2, b2, W3, b3, exact=False):
    """values [N] float64: the layer-3 pre-activation of the kernel's rounded operands (exact=True: of the float64
    network, no rounding anywhere)."""
    return _trace(obs, variant, W1, b1, W2, b2, W3, b3, exact=exact)['z'][2][:, 0]


def ceiling(obs, variant, W1, b1, W2, b2, W3, b3):
    """Per-row upper bound on |kernel - model| [N]: the first-order propagation of policy_oracle.ceiling up to layer
    3's pre-activation (fp32 accumulation, MUFU.TANH, the polynomial's fp32 chain, a 16-bit flip), plus the
    accumulator's own fp32 rounding."""
    tr = _trace(obs, variant, W1, b1, W2, b2, W3, b3)
    W1q, W2q, W3q = tr['W']
    b1q, b2q, b3q = tr['b']
    z1, z2, z3 = tr['z']
    h1, h2 = tr['h']
    poly = tr['poly']
    clamp = float(po.K_TANH_CLAMP)
    nb = 2

    def acc(a_abs, W, b, k):
        return k * po.ACC_REL * (a_abs @ np.abs(W).T + nb * np.abs(b))

    def hidden(z, e_z):
        t = np.tanh(z)
        L = po._sech2_bound(z, e_z)
        e_t = L * e_z + po.MUFU_REL * (np.abs(t) + L * e_z) + 2.0 ** -24 * np.abs(t)
        zp, ep = z[:, poly], e_z[:, poly]
        ep_t = (L[:, poly] + po.POLY_SLOPE_EXCESS) * ep + 2 * po.POLY_EVAL
        e_t[:, poly] = np.where(np.abs(zp) - ep > clamp, 0.0, ep_t)
        return np.where(e_t > 0, e_t + po._ulp(np.abs(t) + e_t + 2.5e-3, 'f16'), 0.0)

    e_z1 = acc(np.abs(tr['xq']), W1q, b1q, W1q.shape[1] + nb)
    e_h1 = hidden(z1, e_z1)
    e_z2 = (np.abs(W2q) @ e_h1.T).T + acc(np.abs(h1) + e_h1, W2q, b2q, po.HIDDEN + nb)
    e_h2 = hidden(z2, e_z2)
    e_z3 = (np.abs(W3q) @ e_h2.T).T + acc(np.abs(h2) + e_h2, W3q, b3q, po.HIDDEN + nb)
    return e_z3[:, 0] + 2.0 ** -23 * np.abs(z3[:, 0])


def scale(obs, variant, W1, b1, W2, b2, W3, b3):
    """sum_j |W3_j| |h2_j| + |b3| [N] of the float64 network: the size of the sum the value is."""
    tr = _trace(obs, variant, W1, b1, W2, b2, W3, b3, exact=True)
    return np.abs(tr['h'][1]) @ np.abs(np.asarray(W3, np.float64))[0] + abs(float(np.asarray(b3)[0]))


def critic_case(case):
    """A shared policy case as a critic case: its observation rows [N, O] and weights with layer 3 = output row 0."""
    first, O, _ = po.VARIANTS[case['variant']]
    W1, b1, W2, b2, W3, b3 = case['weights']
    return dict(name=case['name'], variant=case['variant'], obs=np.ascontiguousarray(case['state'][:, first:first + O]),
                weights=(W1, b1, W2, b2, np.ascontiguousarray(W3[:1]), np.ascontiguousarray(b3[:1])))


def critic_cases():
    for case in po.cases():
        yield critic_case(case)


def case_args(c):
    return (c['obs'], c['variant']) + tuple(c['weights'])
