"""The two policy kernels -- tcgen05 / TMEM (COPTER_B200_POLICY_TC=1, copter_policy_tc.cuh) and warp-level mma.sync
(=0, copter_policy.cuh) -- against oracle/policy_oracle.py, a float64 model of each kernel's own rounding:
  * every element within the model's hard ceiling (fp32 accumulation, MUFU.TANH at 2^-11, a 16-bit flip);
  * per output column, the mean and 99.9th percentile of |got - model| within the tolerance derived from the
    noise model -- a tolerance that tests/test_policy_oracle_cpu.py shows each modelled kernel bug would miss
    by at least 2x;
on dense networks of all variants, on per-column probe networks, at the launch edges, through the C ABI's
sub-range call, and after in-place weight updates.

With COPTER_POLICY_NUMERICS_REPORT=<path> the worst ratios per case and kernel, and the MUFU.TANH error implied
by the probes, are written there as JSON."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import policy_oracle as po      # noqa: E402

CASES = {c['name']: c for c in po.cases()}
REPORT = {}


@pytest.fixture(scope='module')
def pkg():
    import gym_copter_b200
    gym_copter_b200.load_library()
    yield gym_copter_b200
    path = os.environ.get('COPTER_POLICY_NUMERICS_REPORT')
    if path:
        with open(path, 'w') as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)


@pytest.fixture
def policy_kernel_choice():
    """COPTER_B200_POLICY_TC selects the standalone policy kernel per call -- '1' tcgen05 / TMEM (its default),
    '0' warp-level mma.sync -- and COPTER_B200_POLICY_ROLLOUT_TC the fused policy + step rollout kernel (the same
    values and default).  choose(v) sets both to the same kind."""
    names = ('COPTER_B200_POLICY_TC', 'COPTER_B200_POLICY_ROLLOUT_TC')
    old = {k: os.environ.get(k) for k in names}

    def choose(v):
        for k in names:
            os.environ[k] = v
    yield choose
    for k in names:
        if old[k] is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = old[k]


KIND = {'1': 'tc', '0': 'mma'}


def make_net(weights):
    W1, _, _, _, W3, _ = weights
    net = torch.nn.Sequential(torch.nn.Linear(W1.shape[1], 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                              torch.nn.Linear(64, W3.shape[0]), torch.nn.Tanh())
    for p, w in zip(net.parameters(), weights):
        p.data = torch.from_numpy(np.ascontiguousarray(w, np.float32))
    return net.cuda()


def set_planes(env, rows):
    """the fp32 state planes [3][n][4] of `env` <- state rows [n, 12]"""
    env.state_planes.copy_(torch.from_numpy(np.ascontiguousarray(rows.reshape(-1, 3, 4).transpose(1, 0, 2))).cuda())


def run_policy(pkg, variant, rows, net, out_scale, out_offset):
    env = pkg.CopterVecEnv(variant, len(rows), seed=0)
    set_planes(env, rows)
    return pkg.FusedMLPPolicy(env, net, out_scale=out_scale, out_offset=out_offset)().cpu().numpy().astype(np.float64)


def check_against_model(kind, case, got, tol=None, name=None):
    ref = po.case_model(kind, case)
    cei = po.case_ceiling(kind, case)
    assert got.shape == ref.shape and np.all(np.isfinite(got))
    err = np.abs(got - ref)
    worst = float(np.max(err / cei))
    assert np.all(err <= cei), (name, worst, np.unravel_index(np.argmax(err / cei), err.shape))
    if tol is None:
        return worst, None
    d = po.dist(got, ref)
    r = po.ratio(d, tol)
    assert np.all(d[0] <= tol[0]) and np.all(d[1] <= tol[1]), (name, d, tol)
    return worst, r


@pytest.mark.parametrize('kernel', ['1', '0'])
@pytest.mark.parametrize('name', list(CASES))
def test_policy_kernel_vs_rounding_model(pkg, name, kernel, policy_kernel_choice):
    """Dense networks (mlp_policy x1 / x3, all variants, 2^16 rows over rollout ranges plus +-1e4 and zero rows) and
    the 16 probe networks (one path per output, every hidden column of both layers)."""
    policy_kernel_choice(kernel)
    kind, case = KIND[kernel], CASES[name]
    got = run_policy(pkg, case['variant'], case['state'], make_net(case['weights']), case['out_scale'], case['out_offset'])
    tol = po.tolerance(kind, case, seeds=(0, 1, 2))
    worst, r = check_against_model(kind, case, got, tol, name)
    entry = {'ceiling_ratio': worst, 'tol_ratio': r}
    if kind == 'tc' and case['probe'] is not None:
        # output 0 of a probe reads the polynomial columns of both layers: its pre-activation is exact, so what is
        # left is the output's MUFU.TANH (and the final fp32 rounding)
        tr = po._forward(kind, *po.case_args(case))[1]
        t = np.tanh(tr['z'][2][:, 0])
        keep = np.abs(t) > 1e-3
        entry['mufu_rel'] = float(np.max(np.abs(got[keep, 0] - tr['out'][keep, 0]) / np.abs(t[keep])))
    REPORT['%s/%s' % (name, kind)] = entry


@pytest.mark.parametrize('kernel', ['1', '0'])
def test_launch_edges(pkg, kernel, policy_kernel_choice):
    """Partly filled warps and tiles, and one tile more than the resident tcgen05 CTAs hold (148 x 7 x 128 + 1: cluster
    launch control takes the ragged tail over): every row is the same as in one large launch, and within the ceiling."""
    policy_kernel_choice(kernel)
    kind = KIND[kernel]
    big = 148 * 7 * 128 + 1
    W = po.dense_weights('Lander3D', 3)
    rows = po.dense_states(big - 80, seed=7)
    net = make_net(W)
    full = run_policy(pkg, 'Lander3D', rows, net, 0.5, 0.25)
    case = dict(variant='Lander3D', weights=W, state=rows, out_scale=0.5, out_offset=0.25)
    check_against_model(kind, case, full)
    for n in (1, 31, 32, 33, 127, 128, 129, 4099):
        got = run_policy(pkg, 'Lander3D', rows[:n], net, 0.5, 0.25)
        assert np.array_equal(got, full[:n]), n


@pytest.mark.parametrize('kernel', ['1', '0'])
def test_c_abi_sub_range_and_untouched_action_rows(pkg, kernel, policy_kernel_choice):
    """copter_policy_mlp_f32 on rows [lo, lo + n) of a larger allocation (state + lo vectors, state_stride > n), the
    rows outside filled with NaN: the actions equal the model on exactly those rows; an action buffer of n + 64 rows
    prefilled with a NaN sentinel keeps rows >= n bit for bit."""
    from gym_copter_b200 import _lib
    policy_kernel_choice(kernel)
    kind = KIND[kernel]
    case = CASES['Lander2D_x3']
    S, lo, n = 1000, 203, 333
    rows = case['state'][:n]
    planes = torch.full((3, S, 4), float('nan'), device='cuda')
    planes[:, lo:lo + n] = torch.from_numpy(np.ascontiguousarray(rows.reshape(-1, 3, 4).transpose(1, 0, 2))).cuda()
    net = make_net(case['weights'])
    params = [p for p in net.parameters()]
    A = 2
    sentinel = np.array([0x7FC0DEAD], np.uint32).view(np.float32)[0]
    action = torch.full((n + 64, A), float(sentinel), device='cuda')
    action.view(torch.int32).fill_(0x7FC0DEAD)
    lib = _lib.load()
    rc = lib.copter_policy_mlp_f32(planes.data_ptr() + lo * 16, S, n, _lib.VARIANT_IDS['Lander2D'], 64,
                                   *[p.data_ptr() for p in params], C.c_float(case['out_scale']),
                                   C.c_float(case['out_offset']), action.data_ptr(),
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    got = action.cpu().numpy()
    assert np.all(got[n:].view(np.uint32) == 0x7FC0DEAD)
    compact = run_policy(pkg, 'Lander2D', rows, net, case['out_scale'], case['out_offset'])
    assert np.array_equal(got[:n].astype(np.float64), compact)
    check_against_model(kind, dict(case, state=rows), compact)


@pytest.mark.parametrize('kernel', ['1', '0'])
def test_weights_are_read_in_place(pkg, kernel, policy_kernel_choice):
    """After an in-place update of the fp32 parameters (as an optimizer step does), the next FusedMLPPolicy call, the
    next replay of a captured PolicyRollout graph and the next FusedPolicyRollout.run() all use the new weights."""
    policy_kernel_choice(kernel)
    kind = KIND[kernel]
    case = CASES['Lander3D_x1']
    n, T = 2000, 3
    rows = case['state'][:n]
    scale, offset = 0.03, 0.0166

    def fresh_env():
        e = pkg.CopterVecEnv('Lander3D', n, seed=4)
        e.reset()
        return e

    new_w = tuple(np.float32(w * np.float32(0.5)) for w in case['weights'])
    new_case = dict(case, state=rows, weights=new_w, out_scale=scale, out_offset=offset)
    # the standalone kernel
    env = pkg.CopterVecEnv('Lander3D', n, seed=0)
    set_planes(env, rows)
    net = make_net(case['weights'])
    pol = pkg.FusedMLPPolicy(env, net, out_scale=scale, out_offset=offset)
    before = pol().clone()
    for p in net.parameters():
        p.data.mul_(0.5)
    after = pol().cpu().numpy().astype(np.float64)
    assert not np.array_equal(after, before.cpu().numpy())
    assert np.array_equal(after, run_policy(pkg, 'Lander3D', rows, make_net(new_w), scale, offset))
    check_against_model(kind, new_case, after)

    # a captured PolicyRollout graph: replayed after the update == an eager loop with the new weights
    net = make_net(case['weights'])
    a_env, b_env = fresh_env(), fresh_env()
    a_pol = pkg.FusedMLPPolicy(a_env, net, out_scale=scale, out_offset=offset)
    ro = pkg.PolicyRollout(a_env, a_pol, T, planar=True, use_cuda_graph=True)
    ro.run()
    snap = a_env.state_dict()
    b_env.load_state_dict(snap)
    for p in net.parameters():
        p.data.mul_(0.5)
    r_graph = ro.run()[0].clone()
    b_pol = pkg.FusedMLPPolicy(b_env, make_net(new_w), out_scale=scale, out_offset=offset)
    for t in range(T):
        _, r, _, _, _ = b_env.step(b_pol())
        assert torch.equal(r, r_graph[t]), t
    assert torch.equal(a_env.state, b_env.state)

    # FusedPolicyRollout.run(): its recorded actions at t = 0 after the update
    net = make_net(case['weights'])
    c_env = fresh_env()
    set_planes(c_env, rows)
    snap = c_env.state_dict()
    fr = pkg.FusedPolicyRollout(c_env, net, 2, out_scale=scale, out_offset=offset, store_actions=True)
    fr.run()
    old0 = fr.actions[0].clone()
    c_env.load_state_dict(snap)
    for p in net.parameters():
        p.data.mul_(0.5)
    fr.run()
    got0 = fr.actions[0].cpu().numpy().astype(np.float64)
    assert not np.array_equal(got0, old0.cpu().numpy())
    assert np.array_equal(got0, after)
    check_against_model(kind, new_case, got0)
