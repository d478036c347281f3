"""CPU tests of oracle/policy_oracle.py, the float64 model of the two policy kernels' rounding that
tests/test_gpu_policy_numerics.py holds the kernels to: its rounding helpers, its agreement with the float64
network when rounding is switched off, its constants against the header, and -- the point of it -- that the
tolerance it derives would catch each modelled kernel bug (mutant) with a 3x margin."""
import functools
import os
import re

import numpy as np
import pytest
import torch

from oracle import policy_oracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TC_HEADER = os.path.join(ROOT, 'gym_copter_b200', 'csrc', 'copter_policy_tc.cuh')


@functools.lru_cache(maxsize=None)
def all_cases():
    return tuple(po.cases())


@functools.lru_cache(maxsize=None)
def tol_and_ref(kind, name):
    case = next(c for c in all_cases() if c['name'] == name)
    return po.tolerance(kind, case), po.case_model(kind, case)


def _edge_values():
    f = np.float32
    v = [0.0, -0.0, 1.0, -1.0, np.finfo(f).max, -np.finfo(f).max, np.finfo(f).tiny, -np.finfo(f).tiny,
         np.finfo(f).smallest_subnormal, 3 * np.finfo(f).smallest_subnormal, 65504.0, -65504.0, 65519.0, 65520.0,
         2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -25, 2.0 ** -14, 2.0 ** -15 + 2.0 ** -25, 1e-30, -1e-40, 3.0e38]
    for e in (-130, -20, -1, 0, 3, 100):           # exact ties of bf16 (bit 15 set, bits 0-14 zero), both parities
        for m in (0x3F800000, 0x3F810000):
            u = np.uint32(m + (e << 23)) | np.uint32(0x8000) if -126 < e < 128 else np.uint32(0x8000 | (m & 0x7F0000))
            v += [float(np.array(u, np.uint32).view(f)), -float(np.array(u, np.uint32).view(f))]
    for m in (1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 0.5 + 2.0 ** -12, 2.0 ** -14 * (1 + 2.0 ** -11)):  # fp16 ties
        v += [m, -m]
    rng = np.random.default_rng(0)
    v += list(rng.standard_normal(2000) * 10.0 ** rng.integers(-8, 8, 2000))
    return np.array(v, np.float32)


def test_bf16_and_fp16_helpers_round_like_torch_and_numpy():
    x = _edge_values()
    want_bf = torch.from_numpy(x).to(torch.bfloat16).to(torch.float64).numpy()
    got_bf = po.bf16(x)
    assert np.array_equal(got_bf, want_bf)
    assert np.array_equal(np.signbit(got_bf), np.signbit(want_bf))            # -0 stays -0
    with np.errstate(over='ignore'):
        want_h = x.astype(np.float16).astype(np.float64)
        got_h = po.f16(x)
    same = (got_h == want_h) | (np.isinf(got_h) & np.isinf(want_h) & (np.sign(got_h) == np.sign(want_h)))
    assert same.all() and np.array_equal(np.signbit(got_h), np.signbit(want_h))
    assert po.bf16(np.float32(np.nan)) != po.bf16(np.float32(np.nan))        # NaN stays NaN
    # both round to nearest EVEN on an exact tie
    assert po.bf16(np.float32(1.0 + 2.0 ** -8)) == 1.0 and po.bf16(np.float32(1.0 + 3 * 2.0 ** -8)) == 1.0 + 2.0 ** -6
    assert po.f16(1.0 + 2.0 ** -11) == 1.0 and po.f16(1.0 + 3 * 2.0 ** -11) == 1.0 + 2.0 ** -9


@pytest.mark.parametrize('kind', ['tc', 'mma'])
@pytest.mark.parametrize('variant', list(po.VARIANTS))
def test_unrounded_model_is_the_float64_network(kind, variant):
    first, O, A = po.VARIANTS[variant]
    W = po.dense_weights(variant, 3)
    st = po.dense_states(2000, seed=1)
    net = torch.nn.Sequential(torch.nn.Linear(O, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                              torch.nn.Linear(64, A), torch.nn.Tanh()).double()
    for p, w in zip(net.parameters(), W):
        p.data = torch.from_numpy(w.astype(np.float64))
    with torch.no_grad():
        ref = 0.25 + 0.5 * net(torch.from_numpy(st[:, first:first + O].astype(np.float64))).numpy()
    got = po.model(kind, st, variant, *W, 0.5, 0.25, exact=True)
    assert np.max(np.abs(got - ref)) <= 1e-12


def test_constants_are_the_headers():
    src = open(TC_HEADER).read()
    assert int(re.search(r'constexpr int kPolyLanes = (\d+);', src).group(1)) == po.K_POLY_LANES
    assert np.float32(re.search(r'constexpr float kTanhClamp = ([0-9.eE+-]+)f;', src).group(1)) == po.K_TANH_CLAMP
    body = re.search(r'constexpr float c\[7\] = \{([^}]*)\};', src).group(1)
    coef = [np.float32(t.strip().rstrip('f')) for t in body.split(',')]
    assert len(coef) == 7 and all(a == b for a, b in zip(coef, po.TANH_POLY_COEF))


def test_polynomial_tanh_error():
    x = np.linspace(-8, 8, 400001)
    err = np.abs(po.tanh_poly(x) - np.tanh(x))
    assert err.max() <= 2.0e-3
    # about 8 fp16 half-ulps on [0.5, 1) (2^-12 each) -- the comment in copter_policy_tc.cuh says so
    assert 7 * 2.0 ** -12 < err.max() < 9 * 2.0 ** -12
    assert abs(po.tanh_poly(3.25) - 0.99894) < 1e-5 and po.tanh_poly(100.0) == po.tanh_poly(3.25)
    assert np.array_equal(po.tanh_poly(-x), -po.tanh_poly(x))


def test_poly_columns_are_every_fourth():
    assert np.array_equal(np.nonzero(po.poly_columns())[0], np.arange(0, 64, 4))


@pytest.mark.parametrize('kind', ['tc', 'mma'])
def test_every_mutant_is_separated_by_three_tolerances(kind):
    """dist(mutant, model) >= 3 x tol on every case that SEPARATED_BY assigns to the mutant -- so a kernel with that
    bug misses tol by at least 2x (triangle inequality) -- and every mutant of this kind has such a case."""
    covered = {m: 0 for m, ks in po.MUTANT_KINDS.items() if kind in ks}
    for case in all_cases():
        tol, ref = tol_and_ref(kind, case['name'])
        for m in covered:
            if po.applies(m, kind, case):
                r = po.ratio(po.dist(po.case_model(kind, case, m), ref), tol)
                assert r >= 3, (case['name'], m, r)
                covered[m] += 1
    assert all(covered.values()), covered


@pytest.mark.parametrize('kind', ['tc', 'mma'])
def test_ceiling_bounds_the_noise_model(kind):
    """The hard per-element bound holds against the model with random MUFU errors at their bound, for many seeds."""
    picked = [c for c in all_cases() if c['probe'] is not None] + \
             [c for c in all_cases() if c['name'] in ('Lander3D_x3', 'Hover1D_x1', 'Lander2D_x3')]
    for case in picked:
        ref = po.case_model(kind, case)
        cei = po.case_ceiling(kind, case)
        assert np.all(np.isfinite(cei)) and np.all(cei > 0)
        seeds = range(100, 112) if case['probe'] is not None else range(100, 103)
        for s in seeds:
            d = np.abs(po.noisy_model(kind, *po.case_args(case), seed=s) - ref)
            assert np.all(d <= cei), (case['name'], s, float(np.max(d / cei)))


def test_probe_ceiling_is_a_few_ulps():
    """On a probe each output depends on one path, so the bound is tight: a few fp16 ulps of the output."""
    for case in all_cases():
        if case['probe'] is not None:
            assert po.case_ceiling('tc', case).max() < 16 * 2.0 ** -11, case['name']
