// copter_core.h -- the arithmetic of one batched copter step, ONE source for the device and the host.
//
// Everything here compiles both as CUDA device code (included by copter_physics.cuh for the sm_100a
// kernels) and as plain C++ on the host (oracle/copter_host.cpp builds it with g++ into the fp32 / fp64
// CPU restatement the GPU tests compare the kernels with, bit for bit on the fp32 path).  To make
// "the same arithmetic" a statement about BITS and not about compilers:
//   * every fused multiply-add is written out (fma_), every other product and sum is a separate
//     IEEE operation: the .cu is built with -fmad=false and the host file with -ffp-contract=off
//     (COPTER_NO_CONTRACT is defined by both build recipes; without it this header refuses to compile);
//   * no libm function whose result depends on the library is used on the fp32 path: sin / cos are the
//     polynomials below behind an exact fp64 Cody-Waite reduction, sqrt is the IEEE one, and the two
//     approximate reward helpers of the DEVICE path (MUFU.RSQ / MUFU.RCP, reward_sqrt / reward_div below)
//     touch the reward only, never the state or a flag;
//   * the arithmetic is a template over a LANE type L (float or double): any type with the lane
//     operations below instantiates the same sequence of IEEE operations.
//
// What each function restates (paths relative to the reference root):
//   motor_forces()        gym_copter/dynamics/__init__.py:120-132, 231-247   (Eq. 6)
//   airborne_integrate()  gym_copter/dynamics/__init__.py:139-143, 180-187, 249-302   (Eq. 12, Euler)
//   dynamics_update()     gym_copter/dynamics/__init__.py:147-177, 194-197   (status machine)
//   lander_shaping()      gym_copter/envs/lander.py:48-56
//   env_advance()         gym_copter/envs/task.py:77-137 + gym_copter/envs/lander.py:58-72
//   reset_state()         gym_copter/envs/task.py:145-197, gym_copter/dynamics/__init__.py:210-217
//   Takeoff variant       attic/gym_copter/envs/takeoff.py:18-91
//
// Precision.  T = double restates the numpy arithmetic (<= 1e-12 against the reference over 1000
// steps).  T = float stores and integrates in fp32 but evaluates the motor -> thrust/torque stage in
// fp64: the squares of fp32 motor commands are exact in fp64, which removes the systematic
// thrust/torque bias that otherwise grows like t^2 (altitude) and t^4 (lateral position) and breaks
// the 1e-4 budget over 1000 steps (measured: 1.5e-3 all-fp32 vs 1.8e-5 mixed; DESIGN.md).

#pragma once

#include <stdint.h>
#include <math.h>

#include "../../include/copter_b200.h"

#ifndef COPTER_NO_CONTRACT
#error "build with -fmad=false (nvcc) / -ffp-contract=off (host) and -DCOPTER_NO_CONTRACT=1: the arithmetic below is bit-defined"
#endif

#if defined(__CUDACC__)
#define COPTER_HD __host__ __device__ __forceinline__
#else
#define COPTER_HD inline
#endif

namespace copter {

enum { ST_CRASHED = 0, ST_LANDED = 1, ST_LEVELING = 2, ST_AIRBORNE = 3 };
enum { CAUSE_LANDED = 1, CAUSE_BONUS = 2, CAUSE_OOB = 4, CAUSE_ANGLE = 8, CAUSE_CRASHED = 16, CAUSE_TIMEOUT = 32 };
enum { REWARD_LANDER = 0, REWARD_HOVER = 1, REWARD_TAKEOFF = 2 };

// ------------------------------------------------------------------------------------------
// compile-time description of the env variants (SURVEY.md 2.2)
//   clip    the action row is clipped to [0,1] before use (envs/task.py:91); the attic Takeoff env hands
//           it to setMotors as it is (attic/gym_copter/envs/takeoff.py:64)
//   direct  Dynamics is driven directly: a LANDED vehicle still reaches setMotors and can take off
//           (dynamics/__init__.py:147-149); through _Task.step it never does (task.py:86-94)
// ------------------------------------------------------------------------------------------
template <int VARIANT> struct Variant;
template <> struct Variant<COPTER_LANDER3D> { static constexpr int O = 10, A = 4, first = 0, reward = REWARD_LANDER;  static constexpr bool lander = true,  clip = true,  direct = false; };
template <> struct Variant<COPTER_LANDER2D> { static constexpr int O = 6,  A = 2, first = 2, reward = REWARD_LANDER;  static constexpr bool lander = true,  clip = true,  direct = false; };
template <> struct Variant<COPTER_LANDER1D> { static constexpr int O = 2,  A = 1, first = 4, reward = REWARD_LANDER;  static constexpr bool lander = true,  clip = true,  direct = false; };
template <> struct Variant<COPTER_HOVER3D>  { static constexpr int O = 12, A = 4, first = 0, reward = REWARD_HOVER;   static constexpr bool lander = false, clip = true,  direct = false; };
template <> struct Variant<COPTER_HOVER2D>  { static constexpr int O = 6,  A = 2, first = 2, reward = REWARD_HOVER;   static constexpr bool lander = false, clip = true,  direct = false; };
template <> struct Variant<COPTER_HOVER1D>  { static constexpr int O = 2,  A = 1, first = 4, reward = REWARD_HOVER;   static constexpr bool lander = false, clip = true,  direct = false; };
template <> struct Variant<COPTER_TAKEOFF>  { static constexpr int O = 10, A = 4, first = 0, reward = REWARD_TAKEOFF; static constexpr bool lander = false, clip = false, direct = true; };

// ------------------------------------------------------------------------------------------
// kernel-side constants, derived once on the host from CopterParams
// ------------------------------------------------------------------------------------------
template <typename T>
struct KParams {
    double kT, kR, kP, kY;        // B w^2/M, L B w^2/Ix, L B w^2/Iy, D w^2/Iz  (w = maxrpm*pi/30)
    double kOm;                   // w when the gyroscopic coupling is live (COPTER_MODEL_GYRO), else 0
    double force_scale, force_off; // u32 -> U(-F,F): u * 2F/2^32 - F
    T G, dt, gphi, gthe, gpsi;    // (Iy-Iz)/Ix, (Iz-Ix)/Iy, (Ix-Iy)/Iz
    T lvx, lvy, lang, invM;
    T jx, jy;                     // Jr/Ix, Jr/Iy
    T oob_penalty, max_angle, bounds, z0, target_radius;
    T calm_angle;            // min(max_angle, polynomial sin/cos range): below it a step neither ends over-angle nor leaves the fast path
    T yaw_pf, xyz_pf, dz_max, dz_penalty, bonus;
    T takeoff_alt;                // target altitude of the Takeoff variant (attic takeoff.py:20)
    int max_steps;
    int status0;                  // status right after reset (dynamics/__init__.py:215-217)
    int steps_cap;                // the step counter saturates here: 2047 (compact meta word) or 2^30 - 1 (wide counters)
    uint32_t ep_mask;             // episode index wraps here: 2^19 - 1 (compact) or 2^32 - 1 (wide)
};

constexpr double kPi = 3.14159265358979323846;

template <typename T>
inline KParams<T> make_kparams(const CopterParams& p, bool wide = false) {
    KParams<T> k;
    const double w = p.maxrpm * kPi / 30.0;
    // thrust per unit w^2 and the roll/pitch torque arm: live model B and L (dynamics/__init__.py:127-129),
    // lift model 0.5 rho S C_L (L/2)^2 and 1 (attic/mars/dynamics/__init__.py:101,146-158)
    const bool lift = (p.dynamics_model & COPTER_MODEL_LIFT) != 0;
    const double b = lift ? 0.5 * p.rho * (0.05 * p.L * 4) * p.lift_coefficient * (p.L / 2) * (p.L / 2) : p.B;
    const double arm = lift ? 1.0 : p.L;
    k.kT = b * w * w / p.M;
    k.kR = arm * b * w * w / p.Ix;
    k.kP = arm * b * w * w / p.Iy;
    k.kY = p.D * w * w / p.Iz;
    k.kOm = (p.dynamics_model & COPTER_MODEL_GYRO) ? w : 0.0;
    k.jx = (T)(p.Jr / p.Ix); k.jy = (T)(p.Jr / p.Iy);
    k.force_scale = 2.0 * p.initial_random_force / 4294967296.0;
    k.force_off = -p.initial_random_force;
    k.G = (T)p.G;
    k.dt = (T)((T)1 / (T)p.fps);
    k.gphi = (T)((p.Iy - p.Iz) / p.Ix);
    k.gthe = (T)((p.Iz - p.Ix) / p.Iy);
    k.gpsi = (T)((p.Ix - p.Iy) / p.Iz);
    k.lvx = (T)p.landing_vel_x; k.lvy = (T)p.landing_vel_y; k.lang = (T)p.landing_angle;
    k.invM = (T)(1.0 / p.M);
    k.oob_penalty = (T)p.out_of_bounds_penalty;
    k.max_angle = (T)(p.max_angle_deg * kPi / 180.0);
    k.calm_angle = (sizeof(T) == 4 && k.max_angle > (T)0.78539816f) ? (T)0.78539816f : k.max_angle;
    k.bounds = (T)p.bounds;
    k.z0 = (T)(-p.initial_altitude);
    k.target_radius = (T)p.target_radius;
    k.yaw_pf = (T)p.yaw_penalty_factor; k.xyz_pf = (T)p.xyz_penalty_factor;
    k.dz_max = (T)p.dz_max; k.dz_penalty = (T)p.dz_penalty; k.bonus = (T)p.inside_radius_bonus;
    k.takeoff_alt = (T)p.takeoff_target_altitude;
    k.max_steps = p.max_steps;
    k.status0 = (-p.initial_altitude < 0) ? ST_AIRBORNE : ST_LANDED;
    k.steps_cap = wide ? 0x3FFFFFFF : 2047;
    k.ep_mask = wide ? 0xFFFFFFFFu : 0x7FFFFu;
    return k;
}

// ------------------------------------------------------------------------------------------
// lane operations.  A lane type L supports L(scalar) (broadcast), unary minus, + - * as separate
// IEEE operations, and fma_ as ONE fused operation.  float and double are lanes as they are.
// ------------------------------------------------------------------------------------------
COPTER_HD float  fma_(float a, float b, float c)    { return fmaf(a, b, c); }
COPTER_HD double fma_(double a, double b, double c) { return fma(a, b, c); }
COPTER_HD float  abs_t(float a)  { return fabsf(a); }
COPTER_HD double abs_t(double a) { return fabs(a); }
COPTER_HD float  max_t(float a, float b)   { return fmaxf(a, b); }
COPTER_HD double max_t(double a, double b) { return fmax(a, b); }
COPTER_HD float  min_t(float a, float b)   { return fminf(a, b); }
COPTER_HD double min_t(double a, double b) { return fmin(a, b); }
COPTER_HD float  sqrt_t(float a)  { return sqrtf(a); }     // IEEE (correctly rounded) on both sides
COPTER_HD double sqrt_t(double a) { return sqrt(a); }

// fp32 sin/cos on [-pi/4 - eps, pi/4 + eps]: the degree-7 / degree-8 minimax polynomials an accurate
// sincosf evaluates after its range reduction (max rel. error 7e-8 / 9e-8 over the interval).
template <typename L>
COPTER_HD void sincos_poly(L a, L& s, L& c) {
    const L z = a * a;
    L ps = fma_(z, L(-1.95152959e-4f), L(8.33216087e-3f));
    ps = fma_(ps, z, L(-1.66666546e-1f));
    s = fma_(a * z, ps, a);
    L pc = fma_(z, L(2.44331571e-5f), L(-1.38873163e-3f));
    pc = fma_(pc, z, L(4.16666456e-2f));
    pc = fma_(pc, z, L(-0.5f));
    c = fma_(pc, z, L(1.0f));
}

// fp32 sin/cos of any angle.  |a| <= pi/4 needs no range reduction; anything larger (roll / pitch
// beyond pi/4 end the episode, task.py:116, so in practice only a large yaw angle) is reduced in fp64
// with a two-term pi/2 -- exact IEEE operations, the same bits on the host and on the device -- and
// handed to the same polynomials.  Never the SFU approximations (__sinf / __cosf).
COPTER_HD void sincos_t(float a, float& s, float& c) {
    if (fabsf(a) <= 0.78539816f) { sincos_poly<float>(a, s, c); return; }
    const double ad = (double)a;
    const double q = rint(ad * 0.63661977236758134308);             // nearest multiple of pi/2
    double r = fma(q, -1.57079632679489655800, ad);
    r = fma(q, -6.12323399573676603587e-17, r);
    float sr, cr;
    sincos_poly<float>((float)r, sr, cr);
    const double m = q - 4.0 * floor(q * 0.25);                     // quadrant 0..3 (exact while |q| < 2^51)
    const int n = (int)(m >= 0.5) + (int)(m >= 1.5) + (int)(m >= 2.5);
    s = (n & 1) ? cr : sr;  c = (n & 1) ? sr : cr;
    if (n == 1 || n == 2) c = -c;
    if (n >= 2) s = -s;
}
COPTER_HD void sincos_t(double a, double& s, double& c) {
#if defined(__CUDA_ARCH__)
    sincos(a, &s, &c);
#else
    s = sin(a); c = cos(a);
#endif
}

// sin/cos of roll, pitch and yaw together: ONE range test for the three angles on the fp32 path (all
// three are below pi/4 in every step that matters), then three polynomial pairs.
COPTER_HD void sincos3_t(float a, float b, float g, float& sa, float& ca, float& sb, float& cb, float& sg, float& cg) {
    if (fmaxf(fmaxf(fabsf(a), fabsf(b)), fabsf(g)) <= 0.78539816f) {
        sincos_poly<float>(a, sa, ca); sincos_poly<float>(b, sb, cb); sincos_poly<float>(g, sg, cg);
    } else {
        sincos_t(a, sa, ca); sincos_t(b, sb, cb); sincos_t(g, sg, cg);
    }
}
COPTER_HD void sincos3_t(double a, double b, double g, double& sa, double& ca, double& sb, double& cb, double& sg, double& cg) {
    sincos_t(a, sa, ca); sincos_t(b, sb, cb); sincos_t(g, sg, cg);
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11), counter-based: no per-env generator state in memory
// ------------------------------------------------------------------------------------------
COPTER_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}
COPTER_HD void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// Reset force for (global env id, episode): exact in fp64, ONE rounding to T.
template <typename T>
COPTER_HD void reset_force(const KParams<T>& kp, uint64_t seed, uint64_t env, uint32_t episode, T (&f)[3]) {
    uint32_t c[4] = {(uint32_t)env, (uint32_t)(env >> 32), episode, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    for (int j = 0; j < 3; ++j) f[j] = (T)fma((double)c[j], kp.force_scale, kp.force_off);
}

// ------------------------------------------------------------------------------------------
// dynamics
// ------------------------------------------------------------------------------------------
template <typename L> struct Forces { L bz, u2, u3, u4, jxom, jyom; };   // -U1/M, U2/Ix, U3/Iy, U4/Iz, Jr/Ix Omega, Jr/Iy Omega

// dynamics/__init__.py:120-132.  Always evaluated in fp64 (see header comment).
template <typename T>
COPTER_HD Forces<T> motor_forces(const KParams<T>& kp, T m0, T m1, T m2, T m3) {
    const double q0 = (double)m0 * (double)m0, q1 = (double)m1 * (double)m1;
    const double q2 = (double)m2 * (double)m2, q3 = (double)m3 * (double)m3;
    const double s01 = q0 + q1, s23 = q2 + q3;
    Forces<T> f;
    f.bz = (T)(-kp.kT * (s01 + s23));
    f.u2 = (T)(kp.kR * ((q1 + q2) - (q0 + q3)));      // roll right  (:231-235)
    f.u3 = (T)(kp.kP * ((q1 + q3) - (q0 + q2)));      // pitch forward (:237-241)
    f.u4 = (T)(kp.kY * (s01 - s23));                  // yaw cw (:243-247)
    // Omega: zero in the live model (:135); u4 of the UNSQUARED speeds in attic/mars (:143)
    // the rotor-gyroscopic terms of Eq. 12 as two per-launch products (Omega is fixed while the action is): the step
    // multiplies them by one body rate each instead of forming (Jr/I rate) Omega every substep.  Zero in the live model (:135).
    const T om = (T)(kp.kOm * (((double)m0 + (double)m1) - ((double)m2 + (double)m3)));
    f.jxom = kp.jx * om; f.jyom = kp.jy * om;
    return f;
}

// The AIRBORNE, not-touching-the-ground case of setMotors (:180-197): Eq. 12 and one forward Euler
// step from the sines / cosines of the current angles.  PERT: the reset perturbation `p` is added
// (twice, :263-287 and :183) to the first NP rate derivatives (NP = 3 on the env path: x,y,z only,
// envs/task.py:179-184; 6 for the Dynamics facade).  `na` / `nc` receive the shaping numerators
// sum_j inc_j (2 s_j + inc_j) over (x,dx,y,dy,z,dz) and (psi,dpsi), inc_j = dt*ds_j being the Euler
// increment BEFORE it is rounded into the state -- see shaping_delta.  Shared by dynamics_update and
// the straight-line substeps of the K-fused loop, which therefore produce the same bits.  Every
// operation below is one IEEE operation; the comments give the reference expression.
template <typename L, typename T, int NP, bool PERT>
COPTER_HD void airborne_integrate(const KParams<T>& kp, L (&s)[12], const Forces<L>& f, const L (&p)[NP],
                                  L sph, L cph, L sth, L cth, L sps, L cps, L& na, L& nc) {
    // third column of the body->inertial rotation times the body-Z thrust (:292-302)
    const L ux = fma_(cph * cps, sth, sph * sps);                 // sph sps + cph cps sth
    const L uy = fma_(cph * sps, sth, -(cps * sph));              // cph sps sth - cps sph
    L d1 = f.bz * ux, d3 = f.bz * uy;
    L d5 = fma_(f.bz, cph * cth, L(kp.G));                        // netz (:143)
    const L dphi = s[7], dthe = s[9], dpsi = s[11];
    // Eq. 12 (:257-290); the Omega terms are zero in the live model (:135)
    L d7 = fma_(dpsi * dthe, L(kp.gphi), fma_(-dthe, f.jxom, f.u2));
    L d9 = -fma_(dpsi * dphi, L(kp.gthe), fma_(dphi, f.jyom, f.u3));
    L d11 = fma_(dthe * dphi, L(kp.gpsi), f.u4);
    if constexpr (PERT) {                                         // added twice (:263-287, :183); 2 p is exact
        d1 = fma_(L((T)2), p[0], d1); d3 = fma_(L((T)2), p[1], d3); d5 = fma_(L((T)2), p[2], d5);
        if constexpr (NP == 6) { d7 = fma_(L((T)2), p[3], d7); d9 = fma_(L((T)2), p[4], d9); d11 = fma_(L((T)2), p[5], d11); }
    }
    // forward Euler, every derivative from the old state (:187), interleaved with the step's shaping numerators per
    // unit of dt:  a(new) - a(old) = sum_j inc_j (2 old_j + inc_j) with the Euler increment inc_j = dt ds_j taken BEFORE it
    // is rounded into the state (shaping_delta), and 2 old_j + inc_j = old_j + new_j up to that rounding (2^-25 of the
    // term), so each component adds ds_j old_j before and ds_j new_j after its in-place update -- two FMAs, no
    // temporaries; the factor dt is applied once by the consumer (shaping_delta, run_reward).  A position is updated
    // before its velocity, whose old value is its derivative.
    const L dt = L(kp.dt);
    L a = s[1] * s[0];  s[0] = fma_(dt, s[1], s[0]);  a = fma_(s[1], s[0], a);
    a = fma_(d1, s[1], a);  s[1] = fma_(dt, d1, s[1]);  a = fma_(d1, s[1], a);
    a = fma_(s[3], s[2], a);  s[2] = fma_(dt, s[3], s[2]);  a = fma_(s[3], s[2], a);
    a = fma_(d3, s[3], a);  s[3] = fma_(dt, d3, s[3]);  a = fma_(d3, s[3], a);
    a = fma_(s[5], s[4], a);  s[4] = fma_(dt, s[5], s[4]);  a = fma_(s[5], s[4], a);
    a = fma_(d5, s[5], a);  s[5] = fma_(dt, d5, s[5]);  na = fma_(d5, s[5], a);
    s[6] = fma_(dt, dphi, s[6]);   s[7] = fma_(dt, d7, s[7]);
    s[8] = fma_(dt, dthe, s[8]);   s[9] = fma_(dt, d9, s[9]);
    L c = dpsi * s[10];  s[10] = fma_(dt, dpsi, s[10]);  c = fma_(dpsi, s[10], c);
    c = fma_(d11, s[11], c);  s[11] = fma_(dt, d11, s[11]);  nc = fma_(d11, s[11], c);
}

// dynamics/__init__.py:139-197 for one env.  DIRECT enables the LANDED -> AIRBORNE take-off
// transition, unreachable through _Task.step (task.py:86-94).  Returns true when the call ran to
// the end of setMotors (perturbation cleared, ticks += 1), false on the ground-contact early
// return (:177).  The hot case (AIRBORNE, not touching the ground) is tested first.
template <typename T, int NP, bool DIRECT>
COPTER_HD bool dynamics_update(const KParams<T>& kp, T (&s)[12], int& st, const Forces<T>& f, const T (&p)[NP], T& na, T& nc) {
    na = (T)0; nc = (T)0;
    const bool touch = s[4] > (T)0 && s[5] > (T)0;                 // :162 (pre-step state)
    // (the sines / cosines are needed only by the take-off test and the airborne step: a vehicle on the ground,
    // touching it, levelling or crashed goes straight to the status machine)
    if ((DIRECT && st == ST_LANDED) || (st == ST_AIRBORNE && !touch)) {
        T sph, cph, sth, cth, sps, cps;
        sincos3_t(s[6], s[8], s[10], sph, cph, sth, cth, sps, cps);
        if (DIRECT && st == ST_LANDED) {                           // :147-149
            const T netz = fma_(f.bz, cph * cth, kp.G);            // :143
            if (netz < (T)0) st = ST_AIRBORNE;
        }
        if (st == ST_AIRBORNE && !touch) {                         // :159, :180-187
            airborne_integrate<T, T, NP, true>(kp, s, f, p, sph, cph, sth, cth, sps, cps, na, nc);
            return true;
        }
    }
    if (st == ST_LEVELING) {                                       // :152-156
        s[6] = (T)0; s[8] = (T)0; st = ST_LANDED;
        return true;
    }
    if (st == ST_AIRBORNE) {                                       // touched the ground (:162-177)
        // :165-171 -- "velx" is dy, "vely" is dz, only phi is angle-tested (sic)
        st = (s[5] > kp.lvy || abs_t(s[3]) > kp.lvx || abs_t(s[6]) > kp.lang) ? ST_CRASHED : ST_LEVELING;
        return false;                                              // :177
    }
    return true;
}

// envs/lander.py:48-56, kept as its ingredients: shaping = -(xyz_pf*sqrt(a) + yaw_pf*sqrt(c)) - pen.
template <typename T> struct Shaping { T ra, rc, pen; };

template <typename T>
COPTER_HD void shaping_sums(const T (&s)[12], T& spos, T& spsi) {
    spos = ((((s[0] * s[0] + s[1] * s[1]) + s[2] * s[2]) + s[3] * s[3]) + s[4] * s[4]) + s[5] * s[5];
    spsi = s[10] * s[10] + s[11] * s[11];
}

// Reward-only helpers (never used for the state).  On the fp32 DEVICE path sqrt and the quotient of
// shaping_delta go through MUFU.RSQ / MUFU.RCP (<= 2 ulp: a few 1e-7 of the reward against a 1e-4
// budget); the host restatement and the fp64 path use the IEEE operations, so fp32 rewards agree
// between device and host to ~1e-6 relative while states and flags agree bit for bit.
COPTER_HD float reward_sqrt(float a) {
#if defined(__CUDA_ARCH__)
    return a > 0.0f ? a * rsqrtf(a) : 0.0f;
#else
    return sqrtf(a);
#endif
}
COPTER_HD double reward_sqrt(double a) { return sqrt(a); }
COPTER_HD float reward_div(float n, float d) {
#if defined(__CUDA_ARCH__)
    return __fdividef(n, d);
#else
    return n / d;
#endif
}
COPTER_HD double reward_div(double n, double d) { return n / d; }

template <typename T>
COPTER_HD Shaping<T> lander_shaping(const KParams<T>& kp, const T (&s)[12]) {
    T spos, spsi;
    shaping_sums<T>(s, spos, spsi);
    Shaping<T> sh;
    sh.ra = reward_sqrt(spos);
    sh.rc = reward_sqrt(spsi);
    sh.pen = abs_t(s[5]) > kp.dz_max ? kp.dz_penalty : (T)0;
    return sh;
}

// reward = shaping(post) - shaping(pre) (envs/lander.py:58-62), evaluated without the
// cancellation of two O(250..1e4) numbers:  sqrt(a1) - sqrt(a0) = (a1 - a0) / (sqrt(a1) + sqrt(a0))
// with a1 - a0 = sum_j inc_j (2 pre_j + inc_j) = dt sum_j ds_j (pre_j + post_j) (`na`, `nc` from airborne_integrate,
// per unit of dt), where inc_j = dt*ds_j is the Euler increment BEFORE it is rounded into the stored state.  In fp32
// this keeps the reward error proportional to |reward| (1e-5 measured) instead of
// |shaping| * 2^-24 (literal subtraction, up to 1e-3) or ulp(state)/increment (differences of
// stored states, 3e-4 at |v| ~ 270 m/s); in fp64 it agrees with the reference's literal
// subtraction to ~1e-13.
template <typename T>
COPTER_HD T shaping_delta(const KParams<T>& kp, const Shaping<T>& pre, T na, T nc, const Shaping<T>& post) {
    const T da = post.ra + pre.ra, dc = post.rc + pre.rc;
    const T ga = da > (T)0 ? reward_div(kp.dt * na, da) : (T)0;      // (na, nc: numerators per unit of dt, airborne_integrate)
    const T gc = dc > (T)0 ? reward_div(kp.dt * nc, dc) : (T)0;
    return -(kp.xyz_pf * ga + kp.yaw_pf * gc) - (post.pen - pre.pen);
}

// attic/gym_copter/envs/takeoff.py:77-82: shaping = -|altitude - target|, altitude = -z
template <typename T>
COPTER_HD T takeoff_shaping(const KParams<T>& kp, const T (&s)[12]) { return -abs_t(-s[4] - kp.takeoff_alt); }

// One reference _Task.step (envs/task.py:77-137) for one env held in registers, WITHOUT the
// reward: advances the dynamics, the status machine and the step counter and reports whether
// the episode ended and why.  `na` / `nc` are the shaping numerators of this step (see
// airborne_integrate); the reward modifiers are encoded in `cause` (BONUS: + bonus, lander.py:69-72;
// OOB: - penalty, task.py:111-113; ANGLE: reward := - penalty, task.py:116-118; the two are
// exclusive because the reference tests them with if / elif).
// The Takeoff variant is the attic env's step (takeoff.py:57-88): setMotors whatever the status, no
// bounds, no angle limit, never done -- except by the step limit every batched variant has.
template <typename T, int VARIANT>
COPTER_HD void env_advance(const KParams<T>& kp, T (&s)[12], int& st, int& steps, const Forces<T>& f,
                           const T (&pert)[3], T& na, T& nc, bool& done, int& cause) {
    using V = Variant<VARIANT>;
    const int st0 = st;                                            // :81 stale status
    na = (T)0; nc = (T)0;
    if (V::direct || st0 != ST_LANDED)                             // :86-94
        dynamics_update<T, 3, V::direct>(kp, s, st, f, pert, na, nc);
    cause = 0;
    done = false;
    if constexpr (V::reward != REWARD_TAKEOFF) {
        if (V::lander && st0 == ST_LANDED) {                       // lander.py:64-72
            done = true; cause |= CAUSE_LANDED;
            if (sqrt_t(s[0] * s[0] + s[2] * s[2]) < kp.target_radius) cause |= CAUSE_BONUS;
        }
        if (abs_t(s[0]) >= kp.bounds || abs_t(s[2]) >= kp.bounds) {    // task.py:111
            done = true; cause |= CAUSE_OOB;
        } else if (abs_t(s[6]) >= kp.max_angle || abs_t(s[8]) >= kp.max_angle) {   // :116
            done = true; cause |= CAUSE_ANGLE;
        } else if (st0 == ST_CRASHED) {                            // :121
            done = true;
        }
        if (st0 == ST_CRASHED) cause |= CAUSE_CRASHED;
    }
    if (steps == kp.max_steps) { done = true; cause |= CAUSE_TIMEOUT; }          // :128
    steps = steps < kp.steps_cap ? steps + 1 : kp.steps_cap;       // :130 (saturating counter field)
    if (!done) cause = 0;
}

// The reward modifiers of task.py:111-118 and lander.py:69-72 applied to a base reward.
template <typename T>
COPTER_HD T apply_reward_modifiers(const KParams<T>& kp, T r, int cause) {
    if (cause & CAUSE_BONUS) r += kp.bonus;
    if (cause & CAUSE_OOB) r -= kp.oob_penalty;
    else if (cause & CAUSE_ANGLE) r = -kp.oob_penalty;
    return r;
}

// env_advance + the step's reward.  `pre_sh` is shaping(pre-step state) == prev_shaping (the
// priming step of _reset sets it to shaping(s0) and every later step stores the post-step
// value, task.py:197, lander.py:62), so it never has to live in memory; on return it holds
// shaping(post).
template <typename T, int VARIANT>
COPTER_HD void env_substep(const KParams<T>& kp, T (&s)[12], int& st, int& steps, const Forces<T>& f,
                           const T (&pert)[3], Shaping<T>& pre_sh, T& reward, bool& done, int& cause) {
    T na, nc;
    const T tk0 = Variant<VARIANT>::reward == REWARD_TAKEOFF ? takeoff_shaping<T>(kp, s) : (T)0;
    env_advance<T, VARIANT>(kp, s, st, steps, f, pert, na, nc, done, cause);
    if constexpr (Variant<VARIANT>::reward == REWARD_LANDER) {
        const Shaping<T> sh = lander_shaping<T>(kp, s);            // lander.py:48-56
        reward = shaping_delta<T>(kp, pre_sh, na, nc, sh);         // :58-62
        pre_sh = sh;
    } else if constexpr (Variant<VARIANT>::reward == REWARD_TAKEOFF) {
        reward = takeoff_shaping<T>(kp, s) - tk0;                  // takeoff.py:82-86
    } else {
        reward = (T)1;                                             // attic hover.py:18-21
    }
    reward = apply_reward_modifiers<T>(kp, reward, cause);
}

// ------------------------------------------------------------------------------------------
// Telescoped reward of a run of consecutive steps of ONE episode.  sum_k (shaping_k -
// shaping_{k-1}) = shaping_end - shaping_start, so a fused loop only accumulates the shaping
// numerators (two adds per step) and the square roots / quotients are evaluated once, by
// run_reward(), when the run ends (episode finished, or last step of the launch).
// An over-angle ending REPLACES its own step reward by the penalty (task.py:116-118): that
// step's numerators are then left out of the sums and the run ends at the state before it,
// recovered from a_prev = a_now - na, c_prev = c_now - nc and the previous dz.
// Hover variants: +1 per step (attic hover.py:18-21) with the same modifiers.  Takeoff: the
// difference of the two end shapings (no modifiers: the variant has no bounds or angle limit).
// ------------------------------------------------------------------------------------------
template <typename T> struct RewardRun { Shaping<T> start; T na, nc; int steps; };

template <typename T, int VARIANT>
COPTER_HD void run_begin(const KParams<T>& kp, RewardRun<T>& run, const T (&s)[12]) {
    if constexpr (Variant<VARIANT>::reward == REWARD_LANDER) run.start = lander_shaping<T>(kp, s);
    else if constexpr (Variant<VARIANT>::reward == REWARD_TAKEOFF) { run.start.ra = takeoff_shaping<T>(kp, s); run.start.rc = (T)0; run.start.pen = (T)0; }
    else { run.start.ra = (T)0; run.start.rc = (T)0; run.start.pen = (T)0; }
    run.na = (T)0; run.nc = (T)0; run.steps = 0;
}

// one executed step: `cause` is the step's ending cause (0 if the episode goes on)
template <typename T>
COPTER_HD void run_step(RewardRun<T>& run, T na, T nc, int cause) {
    ++run.steps;
    if (!(cause & CAUSE_ANGLE)) { run.na += na; run.nc += nc; }
}

// reward of the run; `s` is the state after its last step (before any auto-reset), `cause` /
// `na` / `nc` / `dz_prev` belong to that last step
template <typename T, int VARIANT>
COPTER_HD T run_reward(const KParams<T>& kp, const RewardRun<T>& run, const T (&s)[12], int cause, T na, T nc, T dz_prev) {
    const bool replaced = (cause & CAUSE_ANGLE) != 0;
    if constexpr (Variant<VARIANT>::reward == REWARD_LANDER) {
        Shaping<T> end = lander_shaping<T>(kp, s);
        if (replaced) {
            end.ra = reward_sqrt(max_t(end.ra * end.ra - kp.dt * na, (T)0));
            end.rc = reward_sqrt(max_t(end.rc * end.rc - kp.dt * nc, (T)0));
            end.pen = abs_t(dz_prev) > kp.dz_max ? kp.dz_penalty : (T)0;
        }
        const T total = shaping_delta<T>(kp, run.start, run.na, run.nc, end);
        return replaced ? total - kp.oob_penalty : apply_reward_modifiers<T>(kp, total, cause);
    } else if constexpr (Variant<VARIANT>::reward == REWARD_TAKEOFF) {
        return takeoff_shaping<T>(kp, s) - run.start.ra;
    } else {
        const T total = (T)run.steps;
        return replaced ? total - (T)1 - kp.oob_penalty : apply_reward_modifiers<T>(kp, total, cause);
    }
}

template <typename T>
COPTER_HD void reset_state(const KParams<T>& kp, T (&s)[12], int& st, int& steps) {
    // envs/task.py:149,164-171,191,197 and dynamics/__init__.py:215-217
    for (int j = 0; j < 12; ++j) s[j] = (T)0;
    s[4] = kp.z0;
    st = kp.status0;
    steps = 1;
}

// the action row of one env -> four motor commands: clip to [0,1] (task.py:91) and fan out (_get_motors)
template <typename T, int VARIANT>
COPTER_HD void motors_from_action(const T* act, T (&m)[4]) {
    constexpr int A = Variant<VARIANT>::A;
    T a[A];
    for (int j = 0; j < A; ++j) a[j] = Variant<VARIANT>::clip ? min_t(max_t(act[j], (T)0), (T)1) : act[j];
    if constexpr (A == 4) { m[0] = a[0]; m[1] = a[1]; m[2] = a[2]; m[3] = a[3]; }
    else if constexpr (A == 2) { m[0] = a[0]; m[1] = a[1]; m[2] = a[1]; m[3] = a[0]; }   // attic lander2d.py:49-51
    else { m[0] = m[1] = m[2] = m[3] = a[0]; }                                          // attic lander1d.py:47-49
}

// ------------------------------------------------------------------------------------------
// One launch of the step for ONE env, the plain way: k substeps under one action through the general
// env_advance, rewards telescoped per run exactly as the kernels do (K = 1 uses env_substep).  This is
// the definition the kernels' fast paths (straight-line substeps, calm streaks, warp votes) must
// reproduce; the host restatement (oracle/copter_host.cpp) is a loop over it.
// ------------------------------------------------------------------------------------------
template <typename T> struct EnvOut { T reward; bool done; int cause; int executed; int final_steps; bool has_final; T final_state[12]; };

template <typename T, int VARIANT>
COPTER_HD void env_launch(const KParams<T>& kp, T (&s)[12], int& st, int& steps, uint32_t& episode, const T (&m)[4],
                          const T (&pert0)[3], int k, bool auto_reset, EnvOut<T>& out) {
    const Forces<T> forces = motor_forces<T>(kp, m[0], m[1], m[2], m[3]);
    T pert[3] = {pert0[0], pert0[1], pert0[2]};
    out.done = false; out.cause = 0; out.executed = 0; out.final_steps = 0; out.has_final = false;
    if (k == 1) {
        Shaping<T> pre_sh = lander_shaping<T>(kp, s);
        T r; bool dn; int cause;
        env_substep<T, VARIANT>(kp, s, st, steps, forces, pert, pre_sh, r, dn, cause);
        out.reward = r; out.executed = 1;
        if (dn) {
            out.done = true; out.cause = cause; out.has_final = true; out.final_steps = steps;
            for (int j = 0; j < 12; ++j) out.final_state[j] = s[j];
            if (auto_reset) { reset_state<T>(kp, s, st, steps); episode = (episode + 1) & kp.ep_mask; }
        }
        return;
    }
    RewardRun<T> run;
    run_begin<T, VARIANT>(kp, run, s);
    T na = (T)0, nc = (T)0, dz_prev = s[5];
    for (int j = 0; j < k; ++j) {
        bool dn; int cause;
        dz_prev = s[5];
        env_advance<T, VARIANT>(kp, s, st, steps, forces, pert, na, nc, dn, cause);
        pert[0] = (T)0; pert[1] = (T)0; pert[2] = (T)0;
        run_step<T>(run, na, nc, cause);
        ++out.executed;
        if (dn) {
            out.done = true; out.cause = cause; out.has_final = true; out.final_steps = steps;
            out.reward = run_reward<T, VARIANT>(kp, run, s, cause, na, nc, dz_prev);
            for (int q = 0; q < 12; ++q) out.final_state[q] = s[q];
            if (auto_reset) { reset_state<T>(kp, s, st, steps); episode = (episode + 1) & kp.ep_mask; }
            return;                                                // idles for the rest of the launch
        }
    }
    out.reward = run_reward<T, VARIANT>(kp, run, s, 0, na, nc, dz_prev);
}

}  // namespace copter
