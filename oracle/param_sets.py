"""
TEST INFRASTRUCTURE ONLY -- named vehicle / world / task parameter sets away from the reference's defaults.

The default DJI Phantom parameters are degenerate in ways that hide whole classes of error: Ix == Iy, so the
roll and pitch torque constants are equal, the two gyroscopic factors are equal and the yaw Euler term
(Ix - Iy) / Iz * dtheta * dphi is exactly zero; the live model has no rotor-gyroscopic coupling; max_angle_deg
= 45 rounds in fp32 to the polynomial range bound of sincos_poly, so calm_angle == max_angle; and every
landing limit, penalty and step length runs at one value.  A transposition of Ix and Iy, or of the two
landing limits, or a dt computed from a hard-coded frame rate, gives the same bits there.

Each set below names the premises it exists to exercise, and premises() checks them on the constants
make_kparams (gym_copter_b200/csrc/copter_core.h) derives, restated here in float64, so that a later edit of
a set cannot quietly make it degenerate again.  tests/test_params_cpu.py runs the header's host
instantiation against the numpy oracle at every set; tests/test_gpu_params.py runs every kernel that takes
CopterParams against the host instantiation and the oracle at the same sets.
"""
import numpy as np

from .copter_oracle import OracleParams

# sincos_poly's range: sincos3_t, airborne_hot and calm_angle all test against this fp32 constant
POLY_RANGE_F32 = np.float32(0.78539816)

# short episodes that end in every way within a few dozen steps (as ENDINGS in tests/test_gpu_host_exact.py); the
# start is low enough that a slow descent touches down gently, inside the landing limits, before the step limit
ENDINGS = dict(bounds=2.0, initial_altitude=0.3, max_steps=60)

SETS = {
    # asymmetric inertia, another vehicle and frame rate, an angle limit above the polynomial range, and every
    # landing limit, penalty and reward constant away from its default
    'asymmetric': OracleParams(
        B=6.0e-3, D=2.5e-6, M=1.2, L=0.3, Ix=1.7, Iy=2.3, Iz=3.1, Jr=45e-4, maxrpm=14000, fps=60,
        max_angle_deg=60, landing_vel_x=1.5, landing_vel_y=0.8, landing_angle=0.6, target_radius=0.7,
        yaw_penalty_factor=30, xyz_penalty_factor=15, dz_max=3.0, dz_penalty=40, inside_radius_bonus=70,
        out_of_bounds_penalty=60, initial_random_force=12.5, **ENDINGS),
    # the live rotor-gyroscopic coupling (Omega != 0) with Ix > Iy, and an angle limit below the polynomial range
    'gyro': OracleParams(
        Ix=2.4, Iy=1.6, Iz=2.9, Jr=0.05, fps=80, max_angle_deg=30, dynamics_model=2, initial_random_force=7.75,
        **ENDINGS),
    # attic/mars: rotor-lift thrust with the gyroscopic coupling, Mars gravity and air density
    'mars-lift': OracleParams(
        Ix=1.9, Iy=2.6, Iz=3.3, Jr=0.02, fps=48, G=3.721, rho=0.017, dynamics_model=3, initial_random_force=3.5,
        **ENDINGS),
    # the Takeoff shell's defaults (starts LANDED, no reset force) on an asymmetric vehicle at another frame
    # rate and target altitude; Takeoff has no angle limit, so its commands stay near hover (hover_command)
    'takeoff': OracleParams(
        Ix=2.2, Iy=1.5, Iz=2.7, Jr=0.01, fps=40, initial_altitude=0.0, initial_random_force=0.0,
        takeoff_target_altitude=3.0, max_steps=60),
}

# the variants each set runs: Takeoff has no landing, bounds or angle limit and runs at its own set
SET_VARIANTS = {'asymmetric': ('Lander3D', 'Lander2D', 'Lander1D', 'Hover3D', 'Hover2D', 'Hover1D'),
                'gyro': ('Lander3D', 'Lander2D', 'Lander1D', 'Hover3D', 'Hover2D', 'Hover1D'),
                'mars-lift': ('Lander3D', 'Lander2D', 'Lander1D', 'Hover3D', 'Hover2D', 'Hover1D'),
                'takeoff': ('Takeoff',)}
CASES = [(name, v) for name, vs in SET_VARIANTS.items() for v in vs]

MODEL_LIFT, MODEL_GYRO = 1, 2


def params_dict(p):
    """The set as keyword arguments of CopterVecEnv / make_params."""
    return {f: getattr(p, f) for f in p.__dataclass_fields__}


def kconstants(p):
    """make_kparams' constants in float64 (copter_core.h:95-132)."""
    w = p.maxrpm * np.pi / 30.0
    lift = bool(p.dynamics_model & MODEL_LIFT)
    b = 0.5 * p.rho * (0.05 * p.L * 4) * p.lift_coefficient * (p.L / 2) ** 2 if lift else p.B
    arm = 1.0 if lift else p.L
    max_angle = np.float32(p.max_angle_deg * np.pi / 180.0)
    return dict(kT=b * w * w / p.M, kR=arm * b * w * w / p.Ix, kP=arm * b * w * w / p.Iy, kY=p.D * w * w / p.Iz,
                kOm=w if p.dynamics_model & MODEL_GYRO else 0.0, jx=p.Jr / p.Ix, jy=p.Jr / p.Iy,
                gphi=(p.Iy - p.Iz) / p.Ix, gthe=(p.Iz - p.Ix) / p.Iy, gpsi=(p.Ix - p.Iy) / p.Iz, dt=1.0 / p.fps,
                max_angle_f32=max_angle, calm_angle_f32=min(max_angle, POLY_RANGE_F32), b=b)


def hover_command(p):
    """The motor command whose four rotors together carry the vehicle's weight: sqrt(M G / (4 B)) / w for the
    live model; for the lift model the rotor speed whose lift 0.5 rho S C_L (w L / 2)^2 is M G / 4."""
    w = p.maxrpm * np.pi / 30.0
    if p.dynamics_model & MODEL_LIFT:
        S = 0.05 * p.L * 4
        return float(np.sqrt(p.M * p.G / 4 / (0.5 * p.rho * S * p.lift_coefficient)) / (p.L / 2) / w)
    return float(np.sqrt(p.M * p.G / (4 * p.B)) / w)


def premises(name, p=None):
    """What makes set `name` worth running: assert it on the constants the kernels derive from it."""
    p = SETS[name] if p is None else p
    d = OracleParams()
    k, k0 = kconstants(p), kconstants(d)
    assert k['kR'] != k['kP'] and k['jx'] != k['jy'] and k['gpsi'] != 0, (name, k)      # roll, pitch and yaw told apart
    assert abs(k['gpsi']) > 0.1 and abs(k['kR'] / k['kP'] - 1) > 0.1, (name, k)
    assert k['dt'] != k0['dt'], name                                                    # another frame rate
    assert p.initial_random_force != d.initial_random_force or name == 'takeoff', name
    if name == 'asymmetric':
        assert k['calm_angle_f32'] == POLY_RANGE_F32 < k['max_angle_f32'], k          # the calm_angle clamp
        for f in ('B', 'D', 'M', 'L', 'Jr', 'maxrpm', 'landing_vel_x', 'landing_vel_y', 'landing_angle',
                  'target_radius', 'yaw_penalty_factor', 'xyz_penalty_factor', 'dz_max', 'dz_penalty',
                  'inside_radius_bonus', 'out_of_bounds_penalty'):
            assert getattr(p, f) != getattr(d, f), f
        assert p.landing_vel_x != p.landing_vel_y and p.dynamics_model == 0
    if name == 'gyro':
        assert p.dynamics_model == MODEL_GYRO and k['kOm'] != 0
        assert k['calm_angle_f32'] == k['max_angle_f32'] < POLY_RANGE_F32, k          # unclamped, below the range
    if name == 'mars-lift':
        assert p.dynamics_model == MODEL_LIFT | MODEL_GYRO and k['kOm'] != 0
        assert p.G != d.G and p.rho != d.rho
        assert k['kR'] != k['b'] * (p.maxrpm * np.pi / 30) ** 2 * p.L / p.Ix          # the lift model's unit arm
    if name == 'takeoff':
        assert p.initial_altitude == 0 and p.initial_random_force == 0
        assert p.takeoff_target_altitude != d.takeoff_target_altitude and p.fps != 50   # (50: the shell's default)
    if name != 'takeoff':
        assert p.bounds < d.bounds and p.initial_altitude < d.initial_altitude and p.max_steps <= 60
    return k
