"""CPU-side checks of the GAE entry point: copter_gae_f32 rejects bad arguments with COPTER_E_ARG before
anything reaches the device, and rollout.gae rejects bad tensors before it calls the library."""
import ctypes as C

import pytest
import torch


@pytest.fixture(scope='module')
def lib():
    from gym_copter_b200 import build, _lib
    build.build()
    return _lib.load()


def test_copter_gae_f32_argument_errors_without_a_gpu(lib):
    # non-null but never dereferenced: every call below must be refused before a launch
    p = C.c_void_p(16)
    ok = dict(reward=p, value=p, last=p, cause=p, final=None, n=64, steps=8, adv=p, ret=None)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.copter_gae_f32(a['reward'], a['value'], a['last'], a['cause'], a['final'], a['n'], a['steps'],
                                  C.c_float(0.99), C.c_float(0.95), a['adv'], a['ret'], None)
    for name in ('reward', 'value', 'last', 'cause', 'adv'):
        assert call(**{name: None}) == -1, name
    assert call(n=-1) == -1
    assert call(steps=0) == -1 and call(steps=-3) == -1
    assert call(n=0) == 0                       # nothing to do: returns before any launch


def test_gae_rejects_bad_tensors_before_the_library():
    from gym_copter_b200 import gae, CopterError
    T, n = 4, 8
    r, v, lv = torch.zeros(T, n), torch.zeros(T, n), torch.zeros(n)
    c = torch.zeros(T, n, dtype=torch.uint8)
    with pytest.raises(ValueError, match='float64'):
        gae(r.double(), v, lv, c)
    with pytest.raises(ValueError):
        gae(r, v, lv, c.bool())                 # causes must be the uint8 cause bits
    with pytest.raises(ValueError):
        gae(r, v[:3], lv, c)                    # T mismatch
    with pytest.raises(ValueError):
        gae(r, v, lv[:5], c)
    with pytest.raises(ValueError):
        gae(r[0], v, lv, c)                     # not [T, N]
    with pytest.raises(ValueError):
        gae(r, v, lv, c, final_values=torch.zeros(T, n + 1))
    with pytest.raises(CopterError):
        gae(r, v, lv, c)                        # host tensors: there is no CPU path
