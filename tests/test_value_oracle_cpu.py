"""CPU checks of the critic's rounding model (oracle/value_oracle.py) and of the argument checks of the two new C-ABI
calls, copter_value_mlp_f32 and copter_policy_logp_f32, which return before anything touches the device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import value_oracle as vo

CASES = {c['name']: c for c in vo.critic_cases()}


def torch_f64(c):
    W1, b1, W2, b2, W3, b3 = (torch.from_numpy(np.asarray(w, np.float64)) for w in c['weights'])
    x = torch.from_numpy(np.asarray(c['obs'], np.float64))
    return ((torch.tanh(torch.tanh(x @ W1.T + b1) @ W2.T + b2) @ W3.T + b3)[:, 0]).numpy()


@pytest.mark.parametrize('name', list(CASES))
def test_value_model_against_float64_network(name):
    """exact=True is the float64 critic; the rounded model is within REL_TO_NETWORK * (sum |W3| |h2| + |b3|) of it on
    the dense networks; the ceiling is finite, positive and below that bound."""
    c = CASES[name]
    args = vo.case_args(c)
    net = torch_f64(c)
    exact = vo.model(*args, exact=True)
    assert np.allclose(exact, net, rtol=1e-12, atol=1e-12)
    got, scale, cei = vo.model(*args), vo.scale(*args), vo.ceiling(*args)
    assert got.shape == cei.shape == (len(c['obs']),)
    assert np.all(np.isfinite(cei)) and np.all(cei > 0)
    if name.startswith('probe'):
        return
    assert np.all(np.abs(got - net) <= vo.REL_TO_NETWORK * scale), np.max(np.abs(got - net) / scale)
    assert np.all(cei <= vo.REL_TO_NETWORK * scale)


def test_value_model_is_the_policy_models_layer3_preactivation():
    """The value is policy_oracle's layer-3 pre-activation (no tanh, scale or offset), and a rounding the policy
    model changes (the layer-3 bias lo half) moves it."""
    from oracle import policy_oracle as po
    c = CASES['Lander2D_x3']
    first, O, _ = po.VARIANTS['Lander2D']
    state = np.zeros((len(c['obs']), 12))
    state[:, first:first + O] = c['obs']
    tr = po._forward('tc', state, 'Lander2D', *c['weights'], 1.0, 0.0)[1]
    assert np.array_equal(vo.model(*vo.case_args(c)), tr['z'][2][:, 0])
    with pytest.raises(ValueError):
        vo.model(c['obs'], 'Lander2D', *po.dense_weights('Lander2D', 1))      # two outputs: not a value head


@pytest.fixture(scope='module')
def lib():
    from gym_copter_b200 import build, _lib
    build.build()
    return _lib.load()


def _value_call(lib, **over):
    a = dict(rows=4096, row_stride=10, m=5, variant=0, hidden=64, w=[8192, 8192, 8192, 8192, 8192, 8192], select=None,
             mask=32, value=12288)
    a.update(over)
    return lib.copter_value_mlp_f32(a['rows'], a['row_stride'], a['m'], a['variant'], a['hidden'], *a['w'], a['select'],
                                    a['mask'], a['value'], None)


def test_value_abi_errors(lib):
    """Each error code for its case (the pointers are never dereferenced: every check comes first); m == 0 is a
    no-op that returns 0 without a device."""
    from gym_copter_b200 import _lib
    E_ARG, E_VARIANT, E_ALIGN, E_RANGE = -1, -2, -3, -4
    assert _value_call(lib, rows=None) == E_ARG
    assert _value_call(lib, value=None) == E_ARG
    for k in range(6):
        w = [8192] * 6
        w[k] = None
        assert _value_call(lib, w=w) == E_ARG, k
    assert _value_call(lib, m=-1) == E_ARG
    assert _value_call(lib, variant=7) == E_VARIANT and _value_call(lib, variant=-1) == E_VARIANT
    assert _value_call(lib, row_stride=9) == E_RANGE                            # Lander3D: O = 10
    assert _value_call(lib, variant=_lib.VARIANT_IDS['Hover3D'], row_stride=11) == E_RANGE
    assert _value_call(lib, hidden=32) == E_RANGE
    assert _value_call(lib, rows=4098) == E_ALIGN and _value_call(lib, value=12290) == E_ALIGN
    assert _value_call(lib, w=[8192, 8192, 8193, 8192, 8192, 8192]) == E_ALIGN
    assert _value_call(lib, m=0) == 0 and _value_call(lib, m=0, rows=4100, row_stride=10) == 0


def _logp_call(lib, **over):
    a = dict(seed=1, env_offset=0, n=5, first_step=0, n_steps=3, variant=0, std=4096, out=8192)
    a.update(over)
    return lib.copter_policy_logp_f32(a['seed'], a['env_offset'], a['n'], a['first_step'], a['n_steps'], a['variant'],
                                      a['std'], a['out'], None)


def test_logp_abi_errors(lib):
    E_ARG, E_VARIANT, E_ALIGN, E_RANGE = -1, -2, -3, -4
    assert _logp_call(lib, std=None) == E_ARG and _logp_call(lib, out=None) == E_ARG
    assert _logp_call(lib, n=-1) == E_ARG and _logp_call(lib, n_steps=0) == E_ARG
    assert _logp_call(lib, variant=9) == E_VARIANT
    assert _logp_call(lib, env_offset=-1) == E_RANGE and _logp_call(lib, first_step=-1) == E_RANGE
    assert _logp_call(lib, std=4097) == E_ALIGN and _logp_call(lib, out=8194) == E_ALIGN
    assert _logp_call(lib, n=0) == 0


def test_fused_rollout_and_value_prerequisites_without_a_device():
    """FusedMLPValue rejects a network of the wrong shape before it looks at a device."""
    import gym_copter_b200 as g
    bad = torch.nn.Sequential(torch.nn.Linear(10, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                              torch.nn.Linear(64, 2))
    with pytest.raises(g.CopterError):
        g.FusedMLPValue(bad, 'Lander3D')
    good = torch.nn.Sequential(torch.nn.Linear(10, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                               torch.nn.Linear(64, 1))
    with pytest.raises(g.CopterError):
        g.FusedMLPValue(good, 'Lander2D')                                    # O = 6
    with pytest.raises(g.CopterError):
        g.FusedMLPValue(good, 'Lander3D')                                    # CPU parameters
    with pytest.raises(g.CopterError):
        g.FusedMLPValue(good, 'NoSuchEnv')
