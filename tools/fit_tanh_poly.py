#!/usr/bin/env python3
"""
Developer tool (CPU only): the polynomial tanh of the policy kernels' FMA-pipe route
(gym_copter_b200/csrc/copter_policy_tc.cuh: tanh_poly_coef / kTanhClamp, used by tanh_fma there).

    tanh(x) ~ x * P(x^2),  P of degree 6 (odd polynomial of degree 13), |x| clamped to 3.25

The fit minimises the maximum of the error weighted by 1 / max(|tanh x|, 2^-4) over [0, 3.25] -- i.e. a
relative criterion where tanh is not tiny, because the value is rounded to bf16 (2^-9 relative) right
after -- by Lawson's iteratively reweighted least squares on a dense grid.  The script prints the fitted
coefficients, and the absolute / relative error of both the fresh fit and the coefficients shipped in
the header, including the clamp's own error tanh(inf) - tanh(3.25) = 3.0e-3 * ... at the top end.

    python tools/fit_tanh_poly.py
"""
import numpy as np

CLAMP = 3.25
SHIPPED = [9.977270291e-01, -3.117916466e-01, 9.229137325e-02, -1.838625564e-02,
           2.184749761e-03, -1.380842544e-04, 3.552717362e-06]


def evaluate(c, x):
    xc = np.clip(x, -CLAMP, CLAMP).astype(np.float32)
    u = xc * xc
    p = np.float32(c[6])
    for k in range(5, -1, -1):
        p = p * u + np.float32(c[k])            # (fp32 like the kernel; fma vs mul+add is below the fit error)
    return p * xc


def report(name, c):
    x = np.linspace(-8, 8, 400001)
    err = evaluate(c, x).astype(np.float64) - np.tanh(x)
    rel = np.abs(err) / np.maximum(np.abs(np.tanh(x)), 2.0 ** -4)
    print('%-8s max |err| %.3e   max |err| / max(|tanh|, 2^-4) %.3e   (bf16 half-ulp: 2^-9 = %.2e)'
          % (name, np.abs(err).max(), rel.max(), 2.0 ** -9))


def fit(iters=200):
    x = np.linspace(1e-4, CLAMP, 20001)
    t = np.tanh(x)
    w_err = 1.0 / np.maximum(t, 2.0 ** -4)                  # the error weight of the criterion
    A = np.stack([x ** (2 * k + 1) for k in range(7)], axis=1)
    lam = np.ones_like(x)
    c = None
    for _ in range(iters):                                  # Lawson: reweight by the current weighted error
        sw = np.sqrt(lam) * w_err
        c, *_ = np.linalg.lstsq(A * sw[:, None], t * sw, rcond=None)
        e = np.abs(A @ c - t) * w_err
        lam = lam * e
        lam /= lam.sum()
    return c


def main():
    c = fit()
    print('fitted  :', ', '.join('%.9e' % v for v in c))
    print('shipped :', ', '.join('%.9e' % v for v in SHIPPED))
    report('fitted', c)
    report('shipped', SHIPPED)


if __name__ == '__main__':
    main()
