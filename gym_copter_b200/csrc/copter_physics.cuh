// copter_physics.cuh -- device-side glue around the shared arithmetic (copter_core.h): launch-shape
// constants, vector-plane state access, the straight-line / calm-streak substep pieces of the
// K-fused loop, and the observation staging.
// Included by copter_kernels.cu (kernels, launchers, C ABI).
//
// The arithmetic itself -- Eq. 6 / Eq. 12 dynamics with the flight-status machine, the lander
// reward, one reference env step, the reset state, Philox -- is in copter_core.h, which also
// compiles on the host: oracle/copter_host.cpp is the fp32 / fp64 CPU restatement the kernels are
// compared with (fp32: state, status, step counters, episode indices and done flags bit for bit).

#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "copter_core.h"

namespace copter {

#ifndef COPTER_F32_CTAS_PER_SM
#define COPTER_F32_CTAS_PER_SM 8  // x 128 threads: 1024 resident envs per SM at <= 64 registers (the drawn-command rollout kernels)
#endif
// The step kernel itself: 10 CTAs per SM (<= 48 registers, which the fp32 step kernels reach without spills since the
// two-FMA shaping numerators; at 8 the compiler took 56 and the hardware placed 9).  HBM-bound launches do not care
// (K = 1: 0.4135 vs 0.4134 ms); the issue-bound ones gain a little from the extra warps (K = 8 0.834 -> 0.818, K = 16
// 1.390 -> 1.359 ms, profiles/r2_ab_k_loop5.txt; 9: 1.373, 7: 1.404; 11+ spill).
#ifndef COPTER_STEP_CTAS_PER_SM
#define COPTER_STEP_CTAS_PER_SM 10
#endif

#ifndef COPTER_BLOCK
#define COPTER_BLOCK 128
#endif

constexpr int kBlock = COPTER_BLOCK;
constexpr int kWarpsPerBlock = kBlock / 32;

// ------------------------------------------------------------------------------------------
// small typed helpers
// ------------------------------------------------------------------------------------------
template <typename T> struct Vec;
template <> struct Vec<float>  { using type = float4;  static constexpr int V = 4; };
template <> struct Vec<double> { using type = double2; static constexpr int V = 2; };

// Vector `pl` (components pl*V .. pl*V+V-1) of env i sits at vector pl * stride + i * env_stride of the
// allocation (include/copter_b200.h, "Memory layout"): planes (stride >= n, env_stride 1) or one row per
// env (stride 1, env_stride 12/V).  Every kernel that reads or writes state addresses it this way.
template <typename T>
__device__ __forceinline__ void load_state(const T* __restrict__ state, int64_t stride, int64_t env_stride, int64_t i, T (&s)[12]) {
    using V4 = typename Vec<T>::type;
    constexpr int V = Vec<T>::V;
    const V4* env = reinterpret_cast<const V4*>(state) + i * env_stride;
#pragma unroll
    for (int pl = 0; pl < 12 / V; ++pl) {
        V4 v = env[(int64_t)pl * stride];
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int j = 0; j < V; ++j) s[pl * V + j] = e[j];
    }
}

template <typename T>
__device__ __forceinline__ void store_state(T* __restrict__ state, int64_t stride, int64_t env_stride, int64_t i, const T (&s)[12]) {
    using V4 = typename Vec<T>::type;
    constexpr int V = Vec<T>::V;
    V4* env = reinterpret_cast<V4*>(state) + i * env_stride;
#pragma unroll
    for (int pl = 0; pl < 12 / V; ++pl) {
        V4 v;
        T* e = reinterpret_cast<T*>(&v);
#pragma unroll
        for (int j = 0; j < V; ++j) e[j] = s[pl * V + j];
        env[(int64_t)pl * stride] = v;
    }
}

// meta word(s) <-> (status, steps, episode); `hi` is the wide-counter array or null (include/copter_b200.h)
__device__ __forceinline__ void decode_meta(uint32_t m, const uint32_t* hi, int64_t i, int& st, int& steps, uint32_t& episode) {
    st = (int)(m & 3u);
    if (hi) { steps = (int)(m >> 2); episode = hi[i]; }
    else    { steps = (int)((m >> 2) & 2047u); episode = m >> 13; }
}
__device__ __forceinline__ void store_meta(uint32_t* meta, uint32_t* hi, int64_t i, int st, int steps, uint32_t episode) {
    if (hi) { meta[i] = (uint32_t)st | ((uint32_t)steps << 2); hi[i] = episode; }
    else    meta[i] = (uint32_t)st | ((uint32_t)steps << 2) | (episode << 13);
}

// ------------------------------------------------------------------------------------------
// The common case of env_advance as straight-line code, for the K-fused loop: an AIRBORNE env that
// is not touching the ground, is past the first step of its episode (no reset perturbation left)
// and -- fp32 -- has all three angles inside the polynomial range of sincos_poly.  airborne_hot()
// is that precondition; under it airborne_arith() + airborne_flags() give exactly what env_advance gives.
// ------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ bool airborne_hot(const T (&s)[12], int st, int steps) {
    const T z = s[4], dz = s[5], phi = s[6], the = s[8], psi = s[10];
    // (bitwise on purpose: one straight run of compares, no short-circuit branches)
    int hot = (int)(st == ST_AIRBORNE) & (int)(steps != 1) & (int)!(z > (T)0 && dz > (T)0);
    if constexpr (sizeof(T) == 4) hot &= (int)(fmaxf(fmaxf(fabsf(phi), fabsf(the)), fabsf(psi)) <= 0.78539816f);
    return hot != 0;
}
// Returns the step's ending flags: bit 0 out of bounds, bit 1 over-angle (exclusive: the reference
// tests them with if / elif, task.py:111-118), bit 2 the env's own step limit; 0 = the episode goes
// on.  airborne_cause() turns them into the CAUSE_* bits env_advance reports.
enum { END_OOB = 1, END_ANGLE = 2, END_TIMEOUT = 4 };
// the arithmetic of one such step (no flags, no step counter)
template <typename T>
__device__ __forceinline__ void airborne_arith(const KParams<T>& kp, T (&s)[12], const Forces<T>& f, T& na, T& nc) {
    T sph, cph, sth, cth, sps, cps;
    if constexpr (sizeof(T) == 4) { sincos_poly<T>(s[6], sph, cph); sincos_poly<T>(s[8], sth, cth); sincos_poly<T>(s[10], sps, cps); }
    else sincos3_t(s[6], s[8], s[10], sph, cph, sth, cth, sps, cps);
    const T none[3] = {(T)0, (T)0, (T)0};
    airborne_integrate<T, T, 3, false>(kp, s, f, none, sph, cph, sth, cth, sps, cps, na, nc);
}
// task.py:111-130 with the stale status AIRBORNE, on the state after the step
template <typename T, int VARIANT>
__device__ __forceinline__ int airborne_flags(const KParams<T>& kp, T x, T y, T phi, T the, bool timeout) {
    if constexpr (Variant<VARIANT>::reward == REWARD_TAKEOFF) return timeout ? END_TIMEOUT : 0;
    const bool oob = abs_t(x) >= kp.bounds || abs_t(y) >= kp.bounds;
    const bool ang = !oob && (abs_t(phi) >= kp.max_angle || abs_t(the) >= kp.max_angle);
    return (oob ? END_OOB : 0) | (ang ? END_ANGLE : 0) | (timeout ? END_TIMEOUT : 0);
}
// "Calm" after a straight-line step: the step ended nothing (in bounds, under the angle limit, not
// the step limit) AND the env is still in airborne_hot()'s common case, so the next substep can be
// straight-line too.  Deliberately a little stricter than the two conditions it implies (psi is held
// to the angle limit as well, `<` instead of `<=` at the polynomial range): a lane that is not calm
// just goes back to the exact tests.  Five compares instead of the flags + hot + two warp votes.
template <typename T>
__device__ __forceinline__ bool airborne_calm(const KParams<T>& kp, T x, T y, T z, T dz, T phi, T the, T psi, bool timeout) {
    const T m_xy = max_t(abs_t(x), abs_t(y));
    const T m_ang = max_t(max_t(abs_t(phi), abs_t(the)), abs_t(psi));
    return (int)!timeout & (int)(m_xy < kp.bounds) & (int)(m_ang < kp.calm_angle) & (int)!(z > (T)0 && dz > (T)0);
}
__device__ __forceinline__ int airborne_cause(int end) {
    return ((end & END_OOB) ? CAUSE_OOB : 0) | ((end & END_ANGLE) ? CAUSE_ANGLE : 0) | ((end & END_TIMEOUT) ? CAUSE_TIMEOUT : 0);
}

// Row-major float32 observation of a warp's 32 envs, staged through shared memory so the
// global stores are contiguous 8-byte-per-lane warp stores.  `tile` is this warp's
// 32*O-float region; `row0` the first env of the warp; `rows` how many of its envs exist.
template <int VARIANT, typename T>
__device__ __forceinline__ void write_obs_rows(float* __restrict__ obs, float* tile, int lane,
                                               int64_t row0, int rows, const T (&s)[12]) {
    constexpr int O = Variant<VARIANT>::O, first = Variant<VARIANT>::first, H = O / 2;
    float2* t2 = reinterpret_cast<float2*>(tile);
#pragma unroll
    for (int j = 0; j < H; ++j)
        t2[lane * H + j] = make_float2((float)s[first + 2 * j], (float)s[first + 2 * j + 1]);
    __syncwarp();
    float2* out = reinterpret_cast<float2*>(obs + row0 * O);
#pragma unroll
    for (int j = 0; j < H; ++j) {
        const int e = j * 32 + lane;
        if (e < rows * H) out[e] = t2[e];
    }
    __syncwarp();
}

}  // namespace copter
