// copter_kernels.cu -- hand-written sm_100a kernels for the batched copter step, plus the
// C ABI declared in include/copter_b200.h.
//
// One thread per env.  State lives in HBM as 12/V "vector planes" of 128-bit vectors
// (float4 / double2) so that every state access of a warp is one fully coalesced 128-bit
// load or store; the packed meta word, the action row and the reward are coalesced too, and
// the row-major float32 observation is staged through a per-warp shared-memory tile so that
// it leaves the SM as contiguous 256-byte warp stores instead of a 40-byte-strided scatter.
// K reference steps are fused per launch with the whole env state held in registers.
//
// The device-side arithmetic (what each function restates, precision) is in copter_physics.cuh.

#include <stdlib.h>

#include "copter_physics.cuh"
#include "copter_policy.cuh"
#include "copter_policy_tc.cuh"

namespace {

using namespace copter;

template <typename T>
struct StepArgs {
    T* state; uint32_t* meta; uint32_t* meta_hi; const T* action; float* obs; T* reward; uint8_t* done;
    const T* init_force; T* ep_return; double* stats; float* final_obs; uint8_t* cause;
    int64_t n, stride, env_stride, env_offset; uint64_t seed; int k; int auto_reset;
    int64_t prefetch_ahead;     // > 0: tile t asks L2 for the inputs of tile t + prefetch_ahead (prefetch_tile)
};

// One env's inputs exactly as they sit in HBM (128-bit vectors): load_raw issues every load, and
// ties the fp64 action row to the loaded words, before decode_raw unpacks anything.
template <typename T, int A> struct RawEnv {
    typename Vec<T>::type plane[12 / Vec<T>::V];
    T act[A];
    uint32_t meta, meta_hi;
};

__device__ __forceinline__ uint32_t low_word(float v)  { return __float_as_uint(v); }
__device__ __forceinline__ uint32_t low_word(double v) { return (uint32_t)__double2loint(v); }
__device__ __forceinline__ float  or_words(float v, uint32_t m)  { return __uint_as_float(__float_as_uint(v) | m); }
__device__ __forceinline__ double or_words(double v, uint32_t m) { return __hiloint2double(__double2hiint(v) | (int)m, __double2loint(v) | (int)m); }

template <typename T, int A>
__device__ __forceinline__ void load_raw(const StepArgs<T>& a, int64_t i, RawEnv<T, A>& r) {
    using V4 = typename Vec<T>::type;
    constexpr int V = Vec<T>::V;
    const V4* env = reinterpret_cast<const V4*>(a.state) + i * a.env_stride;       // as load_state
#pragma unroll
    for (int pl = 0; pl < 12 / V; ++pl)
        r.plane[pl] = env[(int64_t)pl * a.stride];
    r.meta = a.meta[i];
    r.meta_hi = a.meta_hi ? a.meta_hi[i] : 0u;
    if constexpr (A == 4 && sizeof(T) == 4) {
        const float4 v = reinterpret_cast<const float4*>(a.action)[i];
        r.act[0] = v.x; r.act[1] = v.y; r.act[2] = v.z; r.act[3] = v.w;
    } else if constexpr (A == 4) {
        const double2 v0 = reinterpret_cast<const double2*>(a.action)[2 * i];
        const double2 v1 = reinterpret_cast<const double2*>(a.action)[2 * i + 1];
        r.act[0] = v0.x; r.act[1] = v0.y; r.act[2] = v1.x; r.act[3] = v1.y;
    } else if constexpr (A == 2 && sizeof(T) == 4) {
        const float2 v = reinterpret_cast<const float2*>(a.action)[i];
        r.act[0] = v.x; r.act[1] = v.y;
    } else if constexpr (A == 2) {
        const double2 v = reinterpret_cast<const double2*>(a.action)[i];
        r.act[0] = v.x; r.act[1] = v.y;
    } else {
        r.act[0] = a.action[i];
    }
    // ptxas is free to place the first use of the action row (its clip) anywhere after the action
    // loads -- and has placed it BEFORE the state loads (fp64 Hover3D: 58 instructions and one full
    // memory round trip between the two groups, 0.221 instead of 0.190 ms per launch; which
    // instantiation is hit changes with unrelated edits).  The tie below makes every word of the
    // action row depend on the meta word and one word of every state plane through a value the compiler cannot know
    // is zero (the sign bit of n), so that no use of the action can be scheduled
    // before all of this env's loads have been issued.  Measured (B200): the tie costs 1 % where ptxas
    // had the good order anyway (0.1908 vs 0.1887 ms fp64; fp32 K = 1 0.4191 vs 0.4176, K = 4 0.593 vs
    // 0.585) and saves 14 % where it had not, so it is applied to the fp64 kernels, where the bad
    // order has been seen; the fp32 kernels keep ptxas' own schedule, pinned by tests/test_sass_guards.py.
    if (sizeof(T) == 8) {
        uint32_t mix = r.meta;
#pragma unroll
        for (int pl = 0; pl < 12 / V; ++pl) mix |= low_word(r.plane[pl].x);
        mix &= (uint32_t)((uint64_t)a.n >> 63);
#pragma unroll
        for (int j = 0; j < A; ++j) r.act[j] = or_words(r.act[j], mix);
    }
}

template <typename T, int VARIANT>
__device__ __forceinline__ void decode_raw(const RawEnv<T, Variant<VARIANT>::A>& r, bool wide, T (&s)[12], T (&m)[4], int& st, int& steps, uint32_t& episode) {
    constexpr int V = Vec<T>::V;
#pragma unroll
    for (int pl = 0; pl < 12 / V; ++pl) {
        const T* e = reinterpret_cast<const T*>(&r.plane[pl]);
#pragma unroll
        for (int j = 0; j < V; ++j) s[pl * V + j] = e[j];
    }
    st = (int)(r.meta & 3u);
    if (wide) { steps = (int)(r.meta >> 2); episode = r.meta_hi; }
    else      { steps = (int)((r.meta >> 2) & 2047u); episode = r.meta >> 13; }
    // action row, clipped to [0,1] (task.py:91; not for the Takeoff variant) and fanned out (_get_motors)
    motors_from_action<T, VARIANT>(r.act, m);
}

// Folds the episodes that ended in this warp (flag `ended_lane`) into the statistics: ballot /
// popc per cause bit, REDUX for the length sum, a shuffle tree for the fp64 return sum; lane 0
// then issues a handful of global atomics into this warp's slot (COPTER_STATS_SLOTS rows, 128
// bytes apart, so concurrent warps rarely hit the same line).  Nothing is issued when no
// episode ended -- the common case.  Warp-uniform call.
template <typename T>
__device__ __forceinline__ void flush_episode_stats(double* stats, int lane, bool ended_lane, int ep_cause,
                                                    int ep_len, T ep_ret, bool has_returns) {
    const unsigned full = 0xffffffffu;
    const unsigned ended = __ballot_sync(full, ended_lane);
    if (!ended) return;
    // The lengths are summed as 16-bit halves: with wide counters an episode lasts up to 2^30 - 2 steps, and
    // 32 of those overflow a 32-bit sum (which the REDUX would return wrapped).
    const unsigned len = ended_lane ? (unsigned)ep_len : 0u;
    const unsigned len_lo = __reduce_add_sync(full, len & 0xFFFFu), len_hi = __reduce_add_sync(full, len >> 16);
    const double len_sum = (double)len_hi * 65536.0 + (double)len_lo;
    double ret_sum = ended_lane ? (double)ep_ret : 0.0;
    if (has_returns) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ret_sum += __shfl_xor_sync(full, ret_sum, o);
    }
    unsigned by_cause[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) by_cause[c] = __ballot_sync(full, ended_lane && ((ep_cause >> c) & 1));
    if (lane == 0) {
        double* row = stats + (size_t)((blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5)) % COPTER_STATS_SLOTS) * COPTER_STATS_LEN;
        atomicAdd(&row[COPTER_STAT_EPISODES], (double)__popc(ended));
        atomicAdd(&row[COPTER_STAT_LENGTH_SUM], len_sum);
        if (has_returns) atomicAdd(&row[COPTER_STAT_RETURN_SUM], ret_sum);
        // cause bits: LANDED, BONUS, OOB, ANGLE, CRASHED, TIMEOUT
        const int slot[6] = {COPTER_STAT_LANDED, COPTER_STAT_BONUS, COPTER_STAT_OOB, COPTER_STAT_ANGLE, COPTER_STAT_CRASHED, COPTER_STAT_TIMEOUT};
#pragma unroll
        for (int c = 0; c < 6; ++c) if (by_cause[c]) atomicAdd(&row[slot[c]], (double)__popc(by_cause[c]));
    }
}

// Executed env-steps: thread 0 of CTA 0 credits the launch with n * K up front; a warp whose
// envs idled after finishing inside a K-fused launch takes the idle substeps back.
__device__ __forceinline__ void credit_env_steps(double* stats, int64_t n, int k) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&stats[COPTER_STAT_ENV_STEPS], (double)n * (double)k);
}
__device__ __forceinline__ void debit_idle_steps(double* stats, int lane, int idle) {
    idle = __reduce_add_sync(0xffffffffu, idle);
    if (idle && lane == 0)
        atomicAdd(&stats[(size_t)((blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5)) % COPTER_STATS_SLOTS) * COPTER_STATS_LEN + COPTER_STAT_ENV_STEPS], -(double)idle);
}

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------

// One tile (this thread's env `i`) in from HBM, through K substeps and out to HBM.
// SINGLE = the K == 1 specialisation: no substep loop, no idle bookkeeping (about 40 fewer
// instructions per env-step on the HBM-bound path).
template <typename T, int VARIANT, bool STATS, bool SINGLE>
__device__ __forceinline__ void step_tile(const KParams<T>& kp, const StepArgs<T>& a, float* tiles, int64_t tile_id) {
    constexpr int O = Variant<VARIANT>::O, A = Variant<VARIANT>::A;
    // (recomputed here rather than passed in: cheaper than keeping five values live across the body)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row0 = tile_id * kBlock + warp * 32;           // first env of this warp
    const int64_t i = row0 + lane;
    const bool valid = i < a.n;
    const int64_t left = a.n - row0;                             // envs from row0 on (may be <= 0 in the last tile)
    const int rows = left >= 32 ? 32 : (left > 0 ? (int)left : 0);
    float* tile = tiles + warp * (32 * O);
    T s[12];
    T m[4] = {(T)0, (T)0, (T)0, (T)0};
    int st = ST_LANDED, steps = 1; uint32_t episode = 0;
    T total = (T)0; bool done_any = false;
    T ret = (T)0, ep_ret = (T)0; int ep_cause = 0, ep_len = 0, n_steps = 0;     // STATS only

    if (valid) {
        RawEnv<T, A> cur;
        load_raw<T, A>(a, i, cur);
        decode_raw<T, VARIANT>(cur, a.meta_hi != nullptr, s, m, st, steps, episode);
        if (STATS && a.ep_return) ret = a.ep_return[i];
    } else {
#pragma unroll
        for (int j = 0; j < 12; ++j) s[j] = (T)0;
    }

    Shaping<T> pre_sh = lander_shaping<T>(kp, s);
    // the action is fixed for the K substeps of a launch, so Eq. 6 (the fp64 stage) runs once
    const Forces<T> forces = motor_forces<T>(kp, m[0], m[1], m[2], m[3]);

    // The reset perturbation is consumed by the first step of an episode (steps == 1).  Inside
    // a launch that can only be substep 0: an env that resets mid-launch idles afterwards.
    T pert[3] = {(T)0, (T)0, (T)0};
    if (valid && steps == 1) {
        T f[3];
        if (a.init_force) { f[0] = a.init_force[3 * i]; f[1] = a.init_force[3 * i + 1]; f[2] = a.init_force[3 * i + 2]; }
        else reset_force<T>(kp, a.seed, (uint64_t)(a.env_offset + i), episode, f);
#pragma unroll
        for (int j = 0; j < 3; ++j) pert[j] = f[j] * kp.invM;              // dynamics/__init__.py:229
    }

    if constexpr (SINGLE) {
        if (valid) {
            T r; bool dn; int cause;
            env_substep<T, VARIANT>(kp, s, st, steps, forces, pert, pre_sh, r, dn, cause);
            total = r;
            if (STATS) { n_steps = 1; ret += r; }
            if (dn) {
                done_any = true;
                ep_cause = cause;
                if (STATS) { ep_len = steps - 1; ep_ret = ret; ret = (T)0; }   // `steps` is 1 right after reset (task.py:191,197)
                if (a.final_obs) {   // terminal observation; rows of unfinished envs stay untouched
#pragma unroll
                    for (int j = 0; j < O; ++j) a.final_obs[i * O + j] = (float)s[Variant<VARIANT>::first + j];
                }
                if (a.auto_reset) {
                    reset_state<T>(kp, s, st, steps);
                    episode = (episode + 1) & kp.ep_mask;
                }
            }
        }
    } else {
        // K substeps under one action: the summed reward telescopes (RewardRun, copter_core.h)
        RewardRun<T> run;
        run_begin<T, VARIANT>(kp, run, s);
        T na = (T)0, nc = (T)0, dz_prev = s[5]; int cause = 0;
        bool live = valid;                                             // has an env that still takes substeps in this launch
        bool ended = false;                                            // its episode ended in this launch
#pragma unroll 1
        for (int k = 0; k < a.k; ++k) {
            if (__all_sync(0xffffffffu, !live)) break;                 // whole warp finished: idle
            // Straight-line substep when every live env of the warp is in the common case (airborne,
            // clear of the ground, past the first step of its episode, small angles): no status
            // machine, no perturbation, one predicated region.  Anything else takes the general step.
            const bool hot = airborne_hot<T>(s, st, steps);
            const bool fast = __all_sync(0xffffffffu, (int)!live | (int)hot);
            bool dn = false;
            if (fast) {                                                // warp-uniform
                // Streak of straight-line substeps: as long as every live lane stays calm (airborne_calm:
                // nothing ended, still in the common case) the next substep needs neither the ending flags
                // nor the hot test -- one compare chain and one vote per substep.  The loop is executed by
                // the whole warp (k stays uniform); lanes whose env already finished in this launch idle in it.
                bool calm = true, tmo = false;
                int streak = 0;
                do {
                    if (live) {
                        dz_prev = s[5];
                        tmo = steps == kp.max_steps;
                        airborne_arith<T>(kp, s, forces, na, nc);
                        ++steps;
                        calm = airborne_calm<T>(kp, s[0], s[2], s[4], s[5], s[6], s[8], s[10], tmo);
                        if (calm) { run.na += na; run.nc += nc; }
                    }
                    ++streak; ++k;
                } while (k < a.k && __all_sync(0xffffffffu, calm));
                --k;                                                   // the for statement counts the last one
                if (live) {
                    run.steps += streak;
                    steps = min(steps, kp.steps_cap);
                    int end = 0;
                    if (!calm) {                                       // back to the exact tests for this lane's last step
                        end = airborne_flags<T, VARIANT>(kp, s[0], s[2], s[6], s[8], tmo);
                        if (!(end & END_ANGLE)) { run.na += na; run.nc += nc; }
                    }
                    dn = end != 0;
                    if (dn) cause = airborne_cause(end);
                }
            } else if (live) {
                dz_prev = s[5];
                env_advance<T, VARIANT>(kp, s, st, steps, forces, pert, na, nc, dn, cause);
                pert[0] = (T)0; pert[1] = (T)0; pert[2] = (T)0;
                run_step<T>(run, na, nc, cause);
            }
            // An env that ends idles for the rest of the launch, so everything its ending needs -- the run's reward, the
            // terminal observation, the reset -- waits until after the loop, where the lanes that did not end take the
            // same run_reward call: one converged call instead of a divergent one at every ending.
            if (dn) { live = false; ended = true; ep_cause = cause; }
        }
        done_any = ended;
        if (valid) {
            total = run_reward<T, VARIANT>(kp, run, s, done_any ? ep_cause : 0, na, nc, dz_prev);
            if (STATS) { n_steps = run.steps; ret += total; }
            if (done_any) {
                if (STATS) { ep_len = steps - 1; ep_ret = ret; ret = (T)0; }   // `steps` is 1 right after reset (task.py:191,197)
                if (a.final_obs) {   // terminal observation; rows of unfinished envs stay untouched
#pragma unroll
                    for (int j = 0; j < O; ++j) a.final_obs[i * O + j] = (float)s[Variant<VARIANT>::first + j];
                }
                if (a.auto_reset) {
                    reset_state<T>(kp, s, st, steps);
                    episode = (episode + 1) & kp.ep_mask;
                }
            }
        }
    }

    if (valid) {
        store_state<T>(a.state, a.stride, a.env_stride, i, s);
        store_meta(a.meta, a.meta_hi, i, st, steps, episode);
        a.reward[i] = total;
        a.done[i] = done_any ? 1 : 0;
        if (a.cause) a.cause[i] = (uint8_t)ep_cause;
        if (STATS && a.ep_return) a.ep_return[i] = ret;
    }
    if (a.obs) write_obs_rows<VARIANT, T>(a.obs, tile, lane, row0, rows, s);
    if (STATS) {
        flush_episode_stats<T>(a.stats, lane, done_any, ep_cause, ep_len, ep_ret, a.ep_return != nullptr);
        if (!SINGLE) debit_idle_steps(a.stats, lane, valid ? a.k - n_steps : 0);
    }
}

// A fp32 K = 1 step moves 68 B per env into the SM, but a CTA issues its loads only when it starts and then holds
// its slot through ~500 warp-instructions of arithmetic per 32 envs, so the bytes in flight from HBM sag whenever
// the resident CTAs compute at once: the step ran 11-17 % above the same byte pattern without the arithmetic
// (profiles/k1_ceiling_and_bulk_prefetch.txt).  So thread 0 of each CTA asks L2 for the inputs of the tile
// `prefetch_ahead` tiles later -- about one wave of resident CTAs ahead, so the lines arrive before that CTA
// starts and are still in L2 when it does -- with bulk prefetches (cp.async.bulk.prefetch.L2: no registers,
// no shared memory, nothing to wait for), and that CTA's own loads then hit L2.  The same bytes come from HBM,
// earlier rather than twice: one wave of tiles is ~13 MB of the 126 MB L2.  Used on device memory in 16-byte
// aligned rows or planes only (launch_step); a tile past the last full one is not prefetched.  Results are
// unchanged: the prefetch only moves lines into L2.
__device__ __forceinline__ void prefetch_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
}
template <typename T, int A>
__device__ __forceinline__ void prefetch_tile(const StepArgs<T>& a, int64_t tile) {
    if (threadIdx.x != 0 || (tile + 1) * kBlock > a.n) return;
    const int64_t row0 = tile * kBlock;
    if (a.env_stride == 1) {                                          // planes: one block per plane
        for (int pl = 0; pl < 3; ++pl) prefetch_l2(reinterpret_cast<const float4*>(a.state) + pl * a.stride + row0, kBlock * 16);
    } else {                                                          // rows: the tile's rows are one block
        prefetch_l2(a.state + row0 * 12, kBlock * 48);
    }
    prefetch_l2(a.action + row0 * A, kBlock * A * sizeof(T));
    prefetch_l2(a.meta + row0, kBlock * 4);
}

template <typename T, int VARIANT, bool STATS>
__global__ void __launch_bounds__(kBlock, sizeof(T) == 4 ? COPTER_STEP_CTAS_PER_SM : 2)
copter_step_kernel(const __grid_constant__ KParams<T> kp, const __grid_constant__ StepArgs<T> a) {
    constexpr int O = Variant<VARIANT>::O;
    __shared__ __align__(16) float tiles[kWarpsPerBlock][32 * O];

    if (STATS) credit_env_steps(a.stats, a.n, a.k);

    // the grid holds exactly one CTA per tile (launch_step_v), so there is no tile loop and no tile
    // count to derive
    if constexpr (sizeof(T) == 4) if (a.prefetch_ahead) prefetch_tile<T, Variant<VARIANT>::A>(a, (int64_t)blockIdx.x + a.prefetch_ahead);
    if (a.k == 1) step_tile<T, VARIANT, STATS, true>(kp, a, &tiles[0][0], (int64_t)blockIdx.x);
    else          step_tile<T, VARIANT, STATS, false>(kp, a, &tiles[0][0], (int64_t)blockIdx.x);
}

// ------------------------------------------------------------------------------------------
// Multi-step rollout with on-device action sources: n_steps reference steps per launch, the
// env state in registers throughout, the motor commands drawn on the device (no action tensor
// in HBM).  Equivalent, step for step, to n_steps launches of copter_step_kernel with k = 1
// fed the same commands (a finished env resets and keeps going -- no idling here).
// ------------------------------------------------------------------------------------------
template <typename T>
struct RolloutArgs {
    T* state; uint32_t* meta; uint32_t* meta_hi; float* obs; T* reward_sum; uint8_t* done_any;
    const T* init_force; T* ep_return; double* stats;
    T* reward_tn; uint8_t* done_tn; T* action_tn;
    int64_t n, stride, env_stride, env_offset, first_step; uint64_t seed;
    int n_steps, auto_reset, src_kind; T src_scale, src_offset;
    T* controller;              // [n][16] PID memories (COPTER_SRC_PID), [n][24] (COPTER_SRC_PID_HOVER)
    T rate_kp, rate_ki, rate_kd, rate_windup, rate_big, pos_kp, pos_ki, pos_kd, pos_windup, pos_target, descent_kp, descent_kd;
    T alt_kp, alt_ki, alt_kd, alt_windup, alt_target;
    uint8_t* cause_tn; float* final_obs_tn;   // ending records (RECORD instantiations only)
};

__device__ __forceinline__ double log_t(double a) { return log(a); }

// Four variates xi_j = N(0,1) | U(-1,1) of (env, step, stream tag) from Philox4x32-10 with counter
// (env_lo, env_hi, step, tag), key = seed (low word XOR the step's high word).
//   U(-1,1): RN(c 2^-31 - 1), one rounding of the exact value.
//   N(0,1):  Box-Muller on u1 = RN((c + 1) 2^-32) in (0, 1], u2 = RN(c' 2^-32), pairs (c0,c1), (c2,c3).
template <typename T>
__device__ __forceinline__ void draw_variates(uint64_t seed, uint64_t env, uint64_t step, uint32_t tag, bool uniform, T (&xi)[4]) {
    uint32_t c[4] = {(uint32_t)env, (uint32_t)(env >> 32), (uint32_t)step, tag};
    philox4x32_10(c, (uint32_t)seed ^ (uint32_t)(step >> 32), (uint32_t)(seed >> 32));
    if constexpr (sizeof(T) == 4) {
        // fp32: the same roundings without the FP64 pipe -- an integer converted with round-to-nearest
        // and scaled by a power of two is the single rounding of the exact value (c 2^-31 - 1 =
        // (c - 2^31) 2^-31 with c - 2^31 an int32).  The Gaussian transform uses the MUFU forms of sqrt
        // and sin/cos (on an angle folded into [-pi, pi)): absolute error 5e-7 on the direction, i.e.
        // <= 4e-6 on a variate at the 6.7-sigma end of the range; the fp64 path below keeps the library
        // functions throughout.
        if (uniform) {
#pragma unroll
            for (int j = 0; j < 4; ++j) xi[j] = __int2float_rn((int)(c[j] ^ 0x80000000u)) * 0x1p-31f;
        } else {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float u1 = __ull2float_rn((unsigned long long)c[2 * h] + 1ull) * 0x1p-32f;      // (0, 1]
                const float u2 = __uint2float_rn(c[2 * h + 1]) * 0x1p-32f;                            // [0, 1]
                float r;
                asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(-2.0f * logf(u1)));    // library logf: lg2.approx loses the small radii (u1 -> 1)
                // cos / sin(2 pi u2) = -cos / -sin(2 pi (u2 - 1/2)): the folded angle stays where sin.approx is accurate
                const float ang = 6.283185307179586f * (u2 - 0.5f);
                xi[2 * h] = -r * __cosf(ang); xi[2 * h + 1] = -r * __sinf(ang);
            }
        }
    } else {
        if (uniform) {
#pragma unroll
            for (int j = 0; j < 4; ++j) xi[j] = (T)fma((double)c[j], 0x1p-31, -1.0);     // exact, one rounding
        } else {                                                                         // Box-Muller, two pairs
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const T u1 = (T)(((double)c[2 * h] + 1.0) * 0x1p-32);                   // (0, 1]
                const T u2 = (T)((double)c[2 * h + 1] * 0x1p-32);
                const T r = sqrt_t((T)-2 * log_t(u1));
                T sn, cs;
                sincos_t((T)6.283185307179586 * u2, sn, cs);
                xi[2 * h] = r * cs; xi[2 * h + 1] = r * sn;
            }
        }
    }
}

// Command vector of (env, step): offset + scale * xi, xi_j = 1 | N(0,1) | U(-1,1); stream tag 1
// (the reset forces use 0, the policy rollout's exploration noise 2).
template <typename T, int A>
__device__ __forceinline__ void draw_action(const RolloutArgs<T>& a, uint64_t env, uint64_t step, T (&act)[A]) {
    T xi[4] = {(T)1, (T)1, (T)1, (T)1};
    if (a.src_kind != COPTER_SRC_CONST) draw_variates<T>(a.seed, env, step, 1u, a.src_kind == COPTER_SRC_UNIFORM, xi);
#pragma unroll
    for (int j = 0; j < A; ++j) act[j] = a.src_offset + a.src_scale * xi[j];
}


// ------------------------------------------------------------------------------------------
// The reference's PID heuristic as an on-device action source (COPTER_SRC_PID).  Restates
// attic/mars/pidcontrollers/__init__.py:12-146 (controllers) and attic/mars/lander3d.py:64-87
// (the Lander3D heuristic and its quad-X mixer).  Each controller's memory is
// (errorI, lastError, deltaError1, deltaError2).
// ------------------------------------------------------------------------------------------
template <typename T> struct PidMem { T errI, last, d1, d2; };

// _PidController.compute (pidcontrollers/__init__.py:32-59)
template <typename T>
__device__ __forceinline__ T pid_compute(T kp, T ki, T kd, T windup, T target, T actual, PidMem<T>& m) {
    const T error = target - actual;
    T out = error * kp;
    if (ki > (T)0) {
        m.errI = fmin(fmax(m.errI + error, -windup), windup);       // constrainAbs (:61-67)
        out += m.errI * ki;
    }
    if (kd > (T)0) {
        const T de = error - m.last;
        out += (m.d1 + m.d2 + de) * kd;
        m.d2 = m.d1; m.d1 = de; m.last = error;
    }
    return out;
}

// AngularVelocityPidController.getDemand (:131-146): integral reset on a fast rotation
template <typename T>
__device__ __forceinline__ T rate_demand(const RolloutArgs<T>& a, T rate, PidMem<T>& m) {
    if (abs_t(rate) > a.rate_big) { m.errI = (T)0; m.last = (T)0; }                      // reset() (:61-65)
    return pid_compute<T>(a.rate_kp, a.rate_ki, a.rate_kd, a.rate_windup, (T)0, rate, m);
}

// _SetPointPidController.getDemand (:70-88): position error -> velocity set-point -> demand
template <typename T>
__device__ __forceinline__ T poshold_demand(const RolloutArgs<T>& a, T x, T dx, PidMem<T>& m) {
    const T target_velocity = (a.pos_target - x) * (T)1;                                   // posPid(1, 0, 0)
    return pid_compute<T>(a.pos_kp, a.pos_ki, a.pos_kd, a.pos_windup, target_velocity, dx, m);
}

// Lander3D.heuristic (attic/mars/lander3d.py:64-87) on the float32 observation the caller of
// the reference would hold; `mem` = (phi_rate, theta_rate, x_poshold [fed y], y_poshold [fed x]).
template <typename T>
__device__ __forceinline__ void pid_heuristic(const RolloutArgs<T>& a, const T (&s)[12], PidMem<T> (&mem)[4], T (&act)[4]) {
    T o[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) o[j] = (T)(float)s[j];
    const T phi_todo = rate_demand<T>(a, o[7], mem[0]) + poshold_demand<T>(a, o[2], o[3], mem[2]);
    const T theta_todo = rate_demand<T>(a, -o[9], mem[1]) + poshold_demand<T>(a, o[0], o[1], mem[3]);
    const T descent_todo = o[4] * a.descent_kp + o[5] * a.descent_kd;                      // DescentPidController (:110-121)
    const T t = (descent_todo + (T)1) / (T)2, r = phi_todo, p = theta_todo;
    const T mix[4] = {t - r - p, t + r + p, t + r - p, t - r + p};                         // lander3d.py:87
#pragma unroll
    for (int j = 0; j < 4; ++j) act[j] = a.src_offset + a.src_scale * mix[j];
}

// Hover3D.heuristic (attic/mars/hover3d.py:65-92, controllers :33-38 and hover.py:23): the same
// roll/pitch loops plus a yaw-rate PID and the altitude-hold set-point controller
// (pidcontrollers/__init__.py:91-99: demand on (-z, -dz), position error -> climb-rate set-point ->
// PI on the climb rate), mixed with the yaw term.  `mem` = (roll_rate, pitch_rate, x_poshold [fed y],
// y_poshold [fed x], yaw_rate, altitude).
template <typename T>
__device__ __forceinline__ void pid_hover_heuristic(const RolloutArgs<T>& a, const T (&s)[12], PidMem<T> (&mem)[6], T (&act)[4]) {
    T o[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) o[j] = (T)(float)s[j];
    const T roll_todo = rate_demand<T>(a, o[7], mem[0]) + poshold_demand<T>(a, o[2], o[3], mem[2]);
    const T pitch_todo = rate_demand<T>(a, -o[9], mem[1]) + poshold_demand<T>(a, o[0], o[1], mem[3]);
    const T yaw_todo = rate_demand<T>(a, -o[11], mem[4]);
    const T climb_target = (a.alt_target - (-o[4])) * (T)1;                                // posPid(1, 0, 0) on -z
    const T hover_todo = pid_compute<T>(a.alt_kp, a.alt_ki, a.alt_kd, a.alt_windup, climb_target, -o[5], mem[5]);
    const T t = (hover_todo + (T)1) / (T)2, r = roll_todo, p = pitch_todo, y = yaw_todo;
    const T mix[4] = {t - r - p - y, t + r + p - y, t + r - p + y, t - r + p + y};         // hover3d.py:92
#pragma unroll
    for (int j = 0; j < 4; ++j) act[j] = a.src_offset + a.src_scale * mix[j];
}

// The 2-D / 1-D demos (attic/heuristic/lander2d.py:14-24, lander1d.py:14-20, hover2d.py:17-31,
// hover1d.py:14-20): the demand is the command itself (no (t+1)/2), 2-D adds -/+ the roll
// correction for the two motor pairs.  Controller memories keep their 3-D slots (0 = roll rate,
// 2 = position hold fed y, 5 = altitude hold), so one layout serves every variant.
template <typename T, int A, int NMEM, bool HOVER>
__device__ __forceinline__ void pid_planar_heuristic(const RolloutArgs<T>& a, const T (&s)[12], PidMem<T> (&mem)[NMEM], T (&act)[A]) {
    const T y = (T)(float)s[2], dy = (T)(float)s[3], z = (T)(float)s[4], dz = (T)(float)s[5], dphi = (T)(float)s[7];
    T demand;
    if constexpr (HOVER) demand = pid_compute<T>(a.alt_kp, a.alt_ki, a.alt_kd, a.alt_windup, (a.alt_target - (-z)) * (T)1, -dz, mem[NMEM - 1]);
    else                 demand = z * a.descent_kp + dz * a.descent_kd;
    if constexpr (A == 1) {
        act[0] = a.src_offset + a.src_scale * demand;
    } else {
        T todo = poshold_demand<T>(a, y, dy, mem[2]);
        if constexpr (HOVER) todo = rate_demand<T>(a, dphi, mem[0]) + todo;            // hover2d.py:23-26
        act[0] = a.src_offset + a.src_scale * (demand - todo);
        act[1] = a.src_offset + a.src_scale * (demand + todo);
    }
}

// Row t of a rollout's ending records: the COPTER_CAUSE_* bits env i's episode ended with on this step (0 while
// it runs) and, where it ended, the observation of the terminal state -- the bytes copter_step_* (k = 1) writes
// into cause / final_obs.  Called before the reset replaces the state.  The rollout kernels take it in separate
// RECORD instantiations, so the ones without records compile exactly as before.
template <int VARIANT, typename T>
__device__ __forceinline__ void record_ending(uint8_t* cause_tn, float* final_obs_tn, int t, int64_t n, int64_t i,
                                              bool dn, int cause, const T (&s)[12]) {
    constexpr int O = Variant<VARIANT>::O;
    const int64_t row = (int64_t)t * n + i;
    if (cause_tn) cause_tn[row] = (uint8_t)cause;
    if (dn && final_obs_tn) {
#pragma unroll
        for (int j = 0; j < O; ++j) final_obs_tn[row * O + j] = (float)s[Variant<VARIANT>::first + j];
    }
}

// PID: 0 = drawn commands, 1 = landing heuristics (4 controller memories), 2 = hover heuristics (6)
template <typename T, int VARIANT, bool STATS, int PID, bool RECORD>
__global__ void __launch_bounds__(kBlock, sizeof(T) == 4 ? (PID ? 5 : COPTER_F32_CTAS_PER_SM) : 2)
copter_rollout_kernel(const __grid_constant__ KParams<T> kp, const __grid_constant__ RolloutArgs<T> a) {
    constexpr int O = Variant<VARIANT>::O, A = Variant<VARIANT>::A;
    __shared__ __align__(16) float tiles[kWarpsPerBlock][32 * O];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (STATS) credit_env_steps(a.stats, a.n, a.n_steps);
    const int64_t n_tiles = (a.n + kBlock - 1) / kBlock;
    for (int64_t tile_id = blockIdx.x; tile_id < n_tiles; tile_id += gridDim.x) {
        const int64_t row0 = tile_id * kBlock + warp * 32, i = row0 + lane;
        const bool valid = i < a.n;
        const int rows = (int)max((int64_t)0, min((int64_t)32, a.n - row0));
        T s[12];
        int st = ST_LANDED, steps = 1; uint32_t episode = 0;
        T total = (T)0, ret = (T)0; bool done_any = false;
        if (valid) {
            load_state<T>(a.state, a.stride, a.env_stride, i, s);
            decode_meta(a.meta[i], a.meta_hi, i, st, steps, episode);
            if (STATS && a.ep_return) ret = a.ep_return[i];
        } else {
#pragma unroll
            for (int j = 0; j < 12; ++j) s[j] = (T)0;
        }
        Shaping<T> pre_sh = lander_shaping<T>(kp, s);
        // Without per-step reward output the launch's reward sum telescopes per episode (RewardRun).
        // Closing a run costs more than a step's own reward, so the reset-dominated U(-1,1) stream
        // (episodes of ~6 steps: some lane of every warp finishes on every step) keeps the per-step
        // evaluation: measured 5.2e10 vs 4.5e10 env-steps/s there, 1.25e11 vs 1.15e11 on the
        // constant-thrust stream the other way round.
        const bool per_step = a.reward_tn != nullptr || a.src_kind == COPTER_SRC_UNIFORM;
        RewardRun<T> run;
        run_begin<T, VARIANT>(kp, run, s);
        T na = (T)0, nc = (T)0, dz_prev = s[5];
        constexpr int NMEM = PID == 2 ? 6 : 4;
        PidMem<T> mem[NMEM];
        if constexpr (PID != 0) {
            if (valid) {
#pragma unroll
                for (int c = 0; c < NMEM; ++c) { const T* q = a.controller + i * (4 * NMEM) + 4 * c; mem[c].errI = q[0]; mem[c].last = q[1]; mem[c].d1 = q[2]; mem[c].d2 = q[3]; }
            }
        }
        for (int t = 0; t < a.n_steps; ++t) {
            bool dn = false; int cause = 0, ep_len = 0; T ep_ret = (T)0;
            if (valid) {
                T act[A], m[4];
                if constexpr (PID == 1 && A == 4) pid_heuristic<T>(a, s, mem, act);
                else if constexpr (PID == 2 && A == 4) pid_hover_heuristic<T>(a, s, mem, act);
                else if constexpr (PID != 0) pid_planar_heuristic<T, A, NMEM, PID == 2>(a, s, mem, act);
                else draw_action<T, A>(a, (uint64_t)(a.env_offset + i), (uint64_t)(a.first_step + t), act);
                if (a.action_tn) {
#pragma unroll
                    for (int j = 0; j < A; ++j) a.action_tn[((int64_t)t * a.n + i) * A + j] = act[j];
                }
                motors_from_action<T, VARIANT>(act, m);                                     // task.py:91 + _get_motors
                const Forces<T> forces = motor_forces<T>(kp, m[0], m[1], m[2], m[3]);
                T pert[3] = {(T)0, (T)0, (T)0};
                if (steps == 1) {
                    T f[3];
                    if (a.init_force) { f[0] = a.init_force[3 * i]; f[1] = a.init_force[3 * i + 1]; f[2] = a.init_force[3 * i + 2]; }
                    else reset_force<T>(kp, a.seed, (uint64_t)(a.env_offset + i), episode, f);
#pragma unroll
                    for (int j = 0; j < 3; ++j) pert[j] = f[j] * kp.invM;
                }
                if (per_step) {
                    T r;
                    env_substep<T, VARIANT>(kp, s, st, steps, forces, pert, pre_sh, r, dn, cause);
                    total += r;
                    if (STATS) ret += r;
                    if (a.reward_tn) a.reward_tn[(int64_t)t * a.n + i] = r;
                } else {
                    dz_prev = s[5];
                    env_advance<T, VARIANT>(kp, s, st, steps, forces, pert, na, nc, dn, cause);
                    run_step<T>(run, na, nc, cause);
                    if (dn) {
                        const T seg = run_reward<T, VARIANT>(kp, run, s, cause, na, nc, dz_prev);
                        total += seg;
                        if (STATS) ret += seg;
                    }
                }
                if (a.done_tn) a.done_tn[(int64_t)t * a.n + i] = dn ? 1 : 0;
                if (RECORD) record_ending<VARIANT, T>(a.cause_tn, a.final_obs_tn, t, a.n, i, dn, cause, s);
                if (dn) {
                    done_any = true;
                    if (STATS) { ep_len = steps - 1; ep_ret = ret; ret = (T)0; }
                    if (a.auto_reset) {
                        reset_state<T>(kp, s, st, steps);
                        episode = (episode + 1) & kp.ep_mask;
                        pre_sh = lander_shaping<T>(kp, s);
                    }
                    run_begin<T, VARIANT>(kp, run, s);
                }
            }
            if (STATS) flush_episode_stats<T>(a.stats, lane, dn, cause, ep_len, ep_ret, a.ep_return != nullptr);
        }
        if (valid && !per_step) {
            const T seg = run_reward<T, VARIANT>(kp, run, s, 0, na, nc, dz_prev);      // the episode still open at launch end
            total += seg;
            if (STATS) ret += seg;
        }
        if (valid) {
            store_state<T>(a.state, a.stride, a.env_stride, i, s);
            store_meta(a.meta, a.meta_hi, i, st, steps, episode);
            if (a.reward_sum) a.reward_sum[i] = total;
            if (a.done_any) a.done_any[i] = done_any ? 1 : 0;
            if (STATS && a.ep_return) a.ep_return[i] = ret;
            if constexpr (PID != 0) {
#pragma unroll
                for (int c = 0; c < NMEM; ++c) { T* q = a.controller + i * (4 * NMEM) + 4 * c; q[0] = mem[c].errI; q[1] = mem[c].last; q[2] = mem[c].d1; q[3] = mem[c].d2; }
            }
        }
        if (a.obs) write_obs_rows<VARIANT, T>(a.obs, tiles[warp], lane, row0, rows, s);
    }
}

// ------------------------------------------------------------------------------------------
// Policy-in-the-loop rollout in ONE launch (BASELINE.json configs[4]; SURVEY.md 8f rank 1): for
// n_steps steps, each warp evaluates the tanh MLP policy for its 32 envs (policy_forward_warp,
// copter_policy.cuh) from the state its lanes hold in registers, and every lane then advances
// its own env by one reference step with the resulting command.  State, flight status and the
// running shaping never touch HBM between steps; what leaves the SM per env-step is the row t
// of the [T, N] rollout buffers the learner asks for.  Step for step identical to
// copter_policy_mlp_f32 followed by copter_step_f32 (k = 1), n_steps times.
// ------------------------------------------------------------------------------------------
struct PolicyRolloutArgs {
    float* state; uint32_t* meta; uint32_t* meta_hi; float* obs; float* reward_sum; uint8_t* done_any;
    const float* init_force; float* ep_return; double* stats;
    float* reward_tn; uint8_t* done_tn; float* action_tn; float* obs_tn;
    int64_t n, stride, env_stride, env_offset, first_step; uint64_t seed; int n_steps, auto_reset;
    PolicyWeights w;
    const float* action_std;    // [A] or null: Gaussian exploration noise around the network's output
    uint8_t* cause_tn; float* final_obs_tn;   // ending records (RECORD instantiations only)
};

constexpr int kPolicyRolloutCtasPerSm = 5;   // measured (profiles/r1_sweep_policy_occupancy.txt): 3: 0.413, 4: 0.420, 5: 0.400, 6: 0.425 ms per env-step

template <int VARIANT, bool STATS, bool RECORD>
__global__ void __launch_bounds__(128, kPolicyRolloutCtasPerSm)
copter_policy_rollout_kernel(const __grid_constant__ KParams<float> kp, const __grid_constant__ PolicyRolloutArgs a) {
    using T = float;
    static_assert(kBlock == 128, "policy kernels are written for 4 warps per CTA");
    constexpr int O = Variant<VARIANT>::O, A = Variant<VARIANT>::A, FIRST = Variant<VARIANT>::first;
    __shared__ __align__(16) PolicySmem sm;
    __shared__ __align__(16) PolicyWarpTile wtile[4];
    __shared__ __align__(16) float tiles[4][32 * O];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    policy_load_weights<O, A>(sm, a.w);
    __syncthreads();
    if (STATS) credit_env_steps(a.stats, a.n, a.n_steps);

    const int64_t n_tiles = (a.n + kBlock - 1) / kBlock;
    for (int64_t tile_id = blockIdx.x; tile_id < n_tiles; tile_id += gridDim.x) {
        const int64_t row0 = tile_id * kBlock + warp * 32, i = row0 + lane;
        if (row0 >= a.n) continue;                                   // warp-uniform
        const bool valid = i < a.n;
        const int rows = (int)min((int64_t)32, a.n - row0);
        T s[12];
        int st = ST_LANDED, steps = 1; uint32_t episode = 0;
        T total = (T)0, ret = (T)0; bool done_any = false;
        if (valid) {
            load_state<T>(a.state, a.stride, a.env_stride, i, s);
            decode_meta(a.meta[i], a.meta_hi, i, st, steps, episode);
            if (STATS && a.ep_return) ret = a.ep_return[i];
        } else {
#pragma unroll
            for (int j = 0; j < 12; ++j) s[j] = (T)0;
        }
        Shaping<T> pre_sh = lander_shaping<T>(kp, s);
        for (int t = 0; t < a.n_steps; ++t) {
            // the observation the policy acts on at step t
            if (a.obs_tn) write_obs_rows<VARIANT, T>(a.obs_tn + (int64_t)t * a.n * O, tiles[warp], lane, row0, rows, s);
            T act[A];
            policy_forward_warp<FIRST, O, A>(sm, wtile[warp], lane, s, a.w.out_scale, a.w.out_offset, act);
            bool dn = false; int cause = 0, ep_len = 0; T ep_ret = (T)0;
            if (valid) {
                T m[4];
                if (a.action_std) {                                   // exploration: action ~ N(policy(obs), std^2)
                    T xi[4];
                    draw_variates<T>(a.seed, (uint64_t)(a.env_offset + i), (uint64_t)(a.first_step + t), 2u, false, xi);
#pragma unroll
                    for (int j = 0; j < A; ++j) act[j] = fmaf(a.action_std[j], xi[j], act[j]);
                }
                if (a.action_tn) {
                    T* row = a.action_tn + ((int64_t)t * a.n + i) * A;
                    if constexpr (A == 4) *reinterpret_cast<float4*>(row) = make_float4(act[0], act[1], act[2], act[3]);
                    else if constexpr (A == 2) *reinterpret_cast<float2*>(row) = make_float2(act[0], act[1]);
                    else row[0] = act[0];
                }
                motors_from_action<T, VARIANT>(act, m);                                     // task.py:91 + _get_motors
                const Forces<T> forces = motor_forces<T>(kp, m[0], m[1], m[2], m[3]);
                T pert[3] = {(T)0, (T)0, (T)0};
                if (steps == 1) {
                    T f[3];
                    if (a.init_force) { f[0] = a.init_force[3 * i]; f[1] = a.init_force[3 * i + 1]; f[2] = a.init_force[3 * i + 2]; }
                    else reset_force<T>(kp, a.seed, (uint64_t)(a.env_offset + i), episode, f);
#pragma unroll
                    for (int j = 0; j < 3; ++j) pert[j] = f[j] * kp.invM;
                }
                T r;
                env_substep<T, VARIANT>(kp, s, st, steps, forces, pert, pre_sh, r, dn, cause);
                total += r;
                if (STATS) ret += r;
                if (a.reward_tn) a.reward_tn[(int64_t)t * a.n + i] = r;
                if (a.done_tn) a.done_tn[(int64_t)t * a.n + i] = dn ? 1 : 0;
                if (RECORD) record_ending<VARIANT, T>(a.cause_tn, a.final_obs_tn, t, a.n, i, dn, cause, s);
                if (dn) {
                    done_any = true;
                    if (STATS) { ep_len = steps - 1; ep_ret = ret; ret = (T)0; }
                    if (a.auto_reset) {
                        reset_state<T>(kp, s, st, steps);
                        episode = (episode + 1) & kp.ep_mask;
                        pre_sh = lander_shaping<T>(kp, s);
                    }
                }
            }
            if (STATS) flush_episode_stats<T>(a.stats, lane, dn, cause, ep_len, ep_ret, a.ep_return != nullptr);
        }
        if (valid) {
            store_state<T>(a.state, a.stride, a.env_stride, i, s);
            store_meta(a.meta, a.meta_hi, i, st, steps, episode);
            if (a.reward_sum) a.reward_sum[i] = total;
            if (a.done_any) a.done_any[i] = done_any ? 1 : 0;
            if (STATS && a.ep_return) a.ep_return[i] = ret;
        }
        if (a.obs) write_obs_rows<VARIANT, T>(a.obs, tiles[warp], lane, row0, rows, s);
    }
}

// ------------------------------------------------------------------------------------------
// The same rollout on the 5th-generation tensor cores (round 2): the structure of
// copter_mlp_policy_tc_kernel (copter_policy_tc.cuh) with the env step INSIDE its epilogue.
// There a tile is 128 envs and epilogue thread t owns row t of the tile and lane t of tensor
// memory -- which is exactly one thread per env, so the thread that pulls env t's action out of
// TMEM also holds env t's state in registers and steps it.  Per env-step and CTA:
//   epilogue thread   observation row (bf16) -> shared memory (layer-1 A operand)      arrive ready
//   MMA warp          wait ready; tcgen05.mma layer 1 -> TMEM; tcgen05.commit -> done
//   epilogue thread   wait done; tcgen05.ld its row; tanh; bf16 -> shared memory       arrive ready
//   MMA warp          layer 2 ...                       epilogue: the same             arrive ready
//   MMA warp          layer 3 (N = 16) ...              epilogue: tcgen05.ld 4 columns, action = offset +
//                     scale tanh(.), exploration noise, Eq. 6, one reference step, reward / done row t
// State, flight status and the running shaping never leave the registers between the steps of the
// horizon; the grid holds one CTA per tile and the resident CTAs take the pending tiles over (cluster launch
// control, tc::next_tile), 6 CTAs (24 epilogue warps) share an SM and fill one another's MMA round trips.
// The per-env arithmetic is that of the tcgen05 policy kernel followed by
// copter_step_f32 (k = 1): bit-identical to that two-kernel path
// (tests/test_gpu_rollout.py::test_fused_policy_rollout_equals_policy_kernel_plus_step[*-1]).
// ------------------------------------------------------------------------------------------
// Measured, 2^23 envs, horizon 16, ms per env-step.  First version (static grid stride over the tiles, MMAs issued from
// inside an `if (lane == 0)` branch; profiles/r2_sweep_policy_tc_ctas.txt, r2_sweep_policy_tc_rollout.txt):
//   3 CTAs/SM 0.501, 4 CTAs/SM (94 registers) 0.444 / 0.441 (TMEM read-back double- / single-buffered in registers),
//   5 CTAs/SM (72 registers) 0.424, 6 CTAs/SM (64 registers) 0.524 -- behind the warp-MMA kernel above (0.404).
// The clock64 timeline of the standalone kernel (tools/microbench/policy_tc_trace.cu) showed why: the warp scheduler
// favours the oldest CTA of an SM, so a static split leaves the youngest CTA 30 % behind and the SM idling at the end;
// and a layer took 250-600 cycles to ISSUE.  With stolen tiles, warp-uniform issue from prebuilt descriptors and the
// observation staging folded into the A tile (profiles/r2_sweep_policy_tc_rollout2.txt):
//   4 CTAs/SM 0.376, 5 CTAs/SM 0.373, 6 CTAs/SM (64 registers, no spills) 0.342, 7 CTAs/SM (56 registers) 0.348
// -- 2.45e10 env-steps/s, 15 % faster than the warp-MMA kernel, so this kernel is the default of the fused rollout
// (COPTER_B200_POLICY_ROLLOUT_TC=0 selects the warp-MMA kernel).  The TMEM read-back stays single-buffered in registers
// (hidden_epilogue<false>): double-buffered it costs 16 more registers for no gain (the knob is removed; the last tree
// that has it is commit d11af01).
constexpr int kPolicyRolloutTcCtasPerSm = 6;      // x 64 TMEM columns <= the SM's 512; 64 registers, 31.7 KB of shared memory (4: 0.376, 5: 0.373, 6: 0.342, 7: 0.348 ms per env-step)

struct RolloutTcSmem {
    tc::Smem mlp;                                   // weights, the A tile, the mbarriers
    // The per-warp observation staging of write_obs_rows (4 x 1.5 KB) lives INSIDE the hidden A tile, past the
    // 4 KB its layer-1 alias occupies: observations are recorded at the start of an env-step and after the last one,
    // when no MMA reads that tile and no thread writes it before layer 1 has completed (6 KB less per CTA).
    __device__ __forceinline__ float* stage(int warp) { return reinterpret_cast<float*>(reinterpret_cast<char*>(mlp.slot.a) + 4096) + warp * (32 * 12); }
};
static_assert(4096 + 4 * 32 * 12 * sizeof(float) <= sizeof(tc::SlotSmem), "observation staging fits behind the layer-1 alias");

template <int VARIANT, bool STATS, bool RECORD>
__global__ void __launch_bounds__(tc::kThreads, kPolicyRolloutTcCtasPerSm)
copter_policy_rollout_tc_kernel(const __grid_constant__ KParams<float> kp, const __grid_constant__ PolicyRolloutArgs a) {
    using T = float;
    constexpr int O = Variant<VARIANT>::O, A = Variant<VARIANT>::A, FIRST = Variant<VARIANT>::first;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    RolloutTcSmem& rs = *reinterpret_cast<RolloutTcSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
    tc::Smem& sm = rs.mlp;
    const int t_id = threadIdx.x, warp = t_id >> 5, lane = t_id & 31;
    constexpr int kMmaWarp = tc::kTile / 32;
    if (t_id == 0) {
        tc::bar_init(&sm.done, 1);
        tc::bar_init(&sm.ready, tc::kTile);
        tc::bar_init(&sm.clc_bar[0], 1); tc::bar_init(&sm.clc_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) tc::tmem_alloc(sm);
    tc::load_weights<O, A>(sm, a.w.w1, a.w.b1, a.w.w2, a.w.b2, a.w.w3, a.w.b3);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = sm.tmem_base;
    if (STATS) credit_env_steps(a.stats, a.n, a.n_steps);

    if (warp == kMmaWarp) {
        // ===== MMA issuer: 3 layers per env-step, n_steps env-steps per tile.  Warp-uniform, the issuing lane elected per
        // layer (tc::issue_layer_uniform); tiles by cluster launch control, one request in flight (tc::next_tile) =====
        const tc::LayerDescs d = tc::make_layer_descs(sm, tmem_base);
        uint32_t phase = 0, clc_phase = 0, tile_id = blockIdx.x;
        tc::request_tile(sm, 0);
        for (int k = 0; tile_id != tc::kNoTile; ++k) {
            for (int t = 0; t < a.n_steps; ++t)
#pragma unroll
                for (int layer = 1; layer <= 3; ++layer) {
                    tc::bar_wait(&sm.ready, phase); phase ^= 1u;
                    tc::issue_layer_uniform(d, layer, &sm.done);
                }
            tile_id = tc::next_tile(sm, k, clc_phase);
            if (tile_id != tc::kNoTile) tc::request_tile(sm, k + 1);      // clc_resp[(k + 1) & 1] was last read at the end of tile k - 1
        }
    } else {
        // ===== epilogue warps: thread <-> env row <-> TMEM lane =====
        const int row = t_id;                                                        // 0..127
        const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);        // this warp's quarter of the TMEM lanes
        tc::SlotSmem& ss = sm.slot;
        uint32_t phase = 0, clc_phase = 0, tile_id = blockIdx.x;
        for (int k = 0; tile_id != tc::kNoTile; tile_id = tc::next_tile(sm, k, clc_phase), ++k) {
            const int64_t row0 = (int64_t)tile_id * tc::kTile + warp * 32, i = row0 + lane;
            const bool valid = i < a.n;
            const int64_t left = a.n - row0;
            const int rows = left >= 32 ? 32 : (left > 0 ? (int)left : 0);
            T s[12];
            int st = ST_LANDED, steps = 1; uint32_t episode = 0;
            T total = (T)0, ret = (T)0; bool done_any = false;
            if (valid) {
                load_state<T>(a.state, a.stride, a.env_stride, i, s);
                decode_meta(a.meta[i], a.meta_hi, i, st, steps, episode);
                if (STATS && a.ep_return) ret = a.ep_return[i];
            } else {
#pragma unroll
                for (int j = 0; j < 12; ++j) s[j] = (T)0;
            }
            Shaping<T> pre_sh = lander_shaping<T>(kp, s);
            for (int t = 0; t < a.n_steps; ++t) {
                // the observation the policy acts on at step t
                if (a.obs_tn && rows > 0) write_obs_rows<VARIANT, T>(a.obs_tn + (int64_t)t * a.n * O, rs.stage(warp), lane, row0, rows, s);
                tc::write_obs_row<FIRST, O>(ss, row, s);
                tc::fence_before_sync();
                tc::bar_arrive(&sm.ready);
#pragma unroll
                for (int layer = 1; layer <= 2; ++layer) {
                    tc::bar_wait(&sm.done, phase); phase ^= 1u;
                    tc::fence_after_sync();
                    tc::hidden_epilogue<false>(lane_base + tc::kColHidden, ss.a, row);
                    tc::fence_async_smem();
                    tc::fence_before_sync();
                    tc::bar_arrive(&sm.ready);
                }
                tc::bar_wait(&sm.done, phase); phase ^= 1u;
                tc::fence_after_sync();
                float pre[4];
                tc::tmem_ld4(lane_base + tc::kColOut, pre);
                T act[A];
#pragma unroll
                for (int j = 0; j < A; ++j) act[j] = fmaf(a.w.out_scale, tc::tanh_mufu(pre[j]), a.w.out_offset);
                bool dn = false; int cause = 0, ep_len = 0; T ep_ret = (T)0;
                if (valid) {
                    T m[4];
                    if (a.action_std) {                                   // exploration: action ~ N(policy(obs), std^2)
                        T xi[4];
                        draw_variates<T>(a.seed, (uint64_t)(a.env_offset + i), (uint64_t)(a.first_step + t), 2u, false, xi);
#pragma unroll
                        for (int j = 0; j < A; ++j) act[j] = fmaf(a.action_std[j], xi[j], act[j]);
                    }
                    if (a.action_tn) {
                        T* arow = a.action_tn + ((int64_t)t * a.n + i) * A;
                        if constexpr (A == 4) *reinterpret_cast<float4*>(arow) = make_float4(act[0], act[1], act[2], act[3]);
                        else if constexpr (A == 2) *reinterpret_cast<float2*>(arow) = make_float2(act[0], act[1]);
                        else arow[0] = act[0];
                    }
                    motors_from_action<T, VARIANT>(act, m);                                     // task.py:91 + _get_motors
                    const Forces<T> forces = motor_forces<T>(kp, m[0], m[1], m[2], m[3]);
                    T pert[3] = {(T)0, (T)0, (T)0};
                    if (steps == 1) {
                        T f[3];
                        if (a.init_force) { f[0] = a.init_force[3 * i]; f[1] = a.init_force[3 * i + 1]; f[2] = a.init_force[3 * i + 2]; }
                        else reset_force<T>(kp, a.seed, (uint64_t)(a.env_offset + i), episode, f);
#pragma unroll
                        for (int j = 0; j < 3; ++j) pert[j] = f[j] * kp.invM;
                    }
                    T r;
                    env_substep<T, VARIANT>(kp, s, st, steps, forces, pert, pre_sh, r, dn, cause);
                    total += r;
                    if (STATS) ret += r;
                    if (a.reward_tn) a.reward_tn[(int64_t)t * a.n + i] = r;
                    if (a.done_tn) a.done_tn[(int64_t)t * a.n + i] = dn ? 1 : 0;
                    if (RECORD) record_ending<VARIANT, T>(a.cause_tn, a.final_obs_tn, t, a.n, i, dn, cause, s);
                    if (dn) {
                        done_any = true;
                        if (STATS) { ep_len = steps - 1; ep_ret = ret; ret = (T)0; }
                        if (a.auto_reset) {
                            reset_state<T>(kp, s, st, steps);
                            episode = (episode + 1) & kp.ep_mask;
                            pre_sh = lander_shaping<T>(kp, s);
                        }
                    }
                }
                if (STATS) flush_episode_stats<T>(a.stats, lane, dn, cause, ep_len, ep_ret, a.ep_return != nullptr);
            }
            if (valid) {
                store_state<T>(a.state, a.stride, a.env_stride, i, s);
                store_meta(a.meta, a.meta_hi, i, st, steps, episode);
                if (a.reward_sum) a.reward_sum[i] = total;
                if (a.done_any) a.done_any[i] = done_any ? 1 : 0;
                if (STATS && a.ep_return) a.ep_return[i] = ret;
            }
            if (a.obs && rows > 0) write_obs_rows<VARIANT, T>(a.obs, rs.stage(warp), lane, row0, rows, s);
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == kMmaWarp) tc::tmem_free(tmem_base);
}

// ------------------------------------------------------------------------------------------
// Generalised advantage estimation over the [T][n] rows of a rollout (copter_gae_f32; the
// recursion is written out in include/copter_b200.h).  One thread per env walks its column from
// row T-1 back to row 0; every row is one coalesced access of the warp.  Bound by HBM: 17 bytes
// per element (reward, value, cause in; advantage, return out), plus final_value where a
// truncation is read.  The loads do not depend on the recursion, so a block of kGaeRows rows is
// loaded before its arithmetic runs -- kGaeRows rows of loads in flight per thread instead of
// one dependent round trip per row.  Every byte is touched once: streaming (evict-first) loads
// and stores.
// ------------------------------------------------------------------------------------------
struct GaeArgs {
    const float* reward; const float* value; const float* last_value; const uint8_t* cause; const float* final_value;
    float* adv; float* ret;
    int64_t n; int n_steps; float gamma, lam;
};
constexpr int kGaeRows = 8, kGaeBlock = 256;

__global__ void __launch_bounds__(kGaeBlock) copter_gae_kernel(const __grid_constant__ GaeArgs a) {
    const int64_t i = (int64_t)blockIdx.x * kGaeBlock + threadIdx.x;
    if (i >= a.n) return;
    const float gamma = a.gamma, gamma_lam = a.gamma * a.lam;
    float next = a.last_value[i], adv = 0.0f;            // value of row t + 1 and A_next
    for (int t0 = a.n_steps - 1; t0 >= 0; t0 -= kGaeRows) {
        float r[kGaeRows], v[kGaeRows], fv[kGaeRows];
        int c[kGaeRows];
#pragma unroll
        for (int k = 0; k < kGaeRows; ++k) {
            r[k] = 0.0f; v[k] = 0.0f; c[k] = 0;
            if (t0 - k >= 0) {
                const int64_t o = (int64_t)(t0 - k) * a.n + i;
                r[k] = __ldcs(a.reward + o); v[k] = __ldcs(a.value + o); c[k] = __ldcs(a.cause + o);
            }
        }
#pragma unroll
        for (int k = 0; k < kGaeRows; ++k) {                 // the terminal state's value: truncations only
            fv[k] = 0.0f;
            if (t0 - k >= 0 && a.final_value && (c[k] & CAUSE_TIMEOUT)) fv[k] = __ldcs(a.final_value + (int64_t)(t0 - k) * a.n + i);
        }
#pragma unroll
        for (int k = 0; k < kGaeRows; ++k) {
            if (t0 - k >= 0) {
                const int64_t o = (int64_t)(t0 - k) * a.n + i;
                const float boot = c[k] == 0 ? next : fv[k];
                const float delta = r[k] + gamma * boot - v[k];
                adv = delta + gamma_lam * (c[k] == 0 ? adv : 0.0f);
                __stcs(a.adv + o, adv);
                if (a.ret) __stcs(a.ret + o, adv + v[k]);
                next = v[k];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Log-probability of the policy rollout's sampled actions (copter_policy_logp_f32).  The rollout
// draws action = mu + std * xi with xi = draw_variates(seed, env, step, tag 2), so the density of
// what it sampled needs no network: log N(a; mu, std^2) = -1/2 sum xi_j^2 - sum log std_j - A/2 log 2 pi,
// from the same xi bits the rollout drew (the same device function).  One thread per env walks
// its T steps; every row t is one coalesced store of the warp.  Philox and the Box-Muller
// transform are the cost (HBM sees 4 bytes per env-step).
// ------------------------------------------------------------------------------------------
struct LogpArgs {
    uint64_t seed; int64_t env_offset, n, first_step; int n_steps;
    const float* action_std; float* logp;
};
constexpr int kLogpBlock = 256;

template <int A>
__global__ void __launch_bounds__(kLogpBlock) copter_policy_logp_kernel(const __grid_constant__ LogpArgs a) {
    const int64_t i = (int64_t)blockIdx.x * kLogpBlock + threadIdx.x;
    if (i >= a.n) return;
    float c = -0.5f * (float)A * 1.8378770664093453f;              // log 2 pi
#pragma unroll
    for (int j = 0; j < A; ++j) c -= logf(a.action_std[j]);
    for (int t = 0; t < a.n_steps; ++t) {
        float xi[4];
        draw_variates<float>(a.seed, (uint64_t)(a.env_offset + i), (uint64_t)(a.first_step + t), 2u, false, xi);
        float q = 0.0f;
#pragma unroll
        for (int j = 0; j < A; ++j) q = fmaf(xi[j], xi[j], q);
        __stcs(a.logp + (int64_t)t * a.n + i, fmaf(-0.5f, q, c));
    }
}

template <typename T, int VARIANT>
__global__ void __launch_bounds__(kBlock)
copter_reset_kernel(const __grid_constant__ KParams<T> kp, T* state, uint32_t* meta, uint32_t* meta_hi, float* obs, T* ep_return,
                    int64_t n, int64_t stride, int64_t env_stride, int keep_episode) {
    constexpr int O = Variant<VARIANT>::O;
    __shared__ __align__(16) float tiles[kWarpsPerBlock][32 * O];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_tiles = (n + kBlock - 1) / kBlock;
    for (int64_t tile_id = blockIdx.x; tile_id < n_tiles; tile_id += gridDim.x) {
        const int64_t row0 = tile_id * kBlock + warp * 32, i = row0 + lane;
        const int rows = (int)max((int64_t)0, min((int64_t)32, n - row0));
        T s[12]; int st, steps;
        reset_state<T>(kp, s, st, steps);
        if (i < n) {
            store_state<T>(state, stride, env_stride, i, s);
            // COPTER_F_KEEP_EPISODE: the env's next episode index, so that a reset() per episode draws a new
            // reset force every time (the reference draws fresh np.random.uniform forces, task.py:175-184)
            uint32_t episode = 0;
            if (keep_episode) {
                int st_old, steps_old;
                decode_meta(meta[i], meta_hi, i, st_old, steps_old, episode);
                episode = (episode + 1) & kp.ep_mask;
            }
            store_meta(meta, meta_hi, i, st, steps, episode);
            if (ep_return) ep_return[i] = (T)0;
        }
        if (obs) write_obs_rows<VARIANT, T>(obs, tiles[warp], lane, row0, rows, s);
    }
}

// Batched Dynamics.setMotors (dynamics/__init__.py:114-197), all four statuses reachable.
template <typename T>
__global__ void __launch_bounds__(kBlock)
copter_dynamics_kernel(const __grid_constant__ KParams<T> kp, T* state, uint8_t* status, int32_t* ticks,
                       T* perturb, const T* motors, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock) {
        T s[12], p[6], m[4];
        load_state<T>(state, n, 1, i, s);
        int st = status[i];
#pragma unroll
        for (int j = 0; j < 6; ++j) p[j] = perturb[6 * i + j];
#pragma unroll
        for (int j = 0; j < 4; ++j) m[j] = motors[4 * i + j];
        const Forces<T> f = motor_forces<T>(kp, m[0], m[1], m[2], m[3]);
        T na, nc;
        const bool finished = dynamics_update<T, 6, true>(kp, s, st, f, p, na, nc);
        store_state<T>(state, n, 1, i, s);
        status[i] = (uint8_t)st;
        if (finished) {                                            // :194-197
#pragma unroll
            for (int j = 0; j < 6; ++j) perturb[6 * i + j] = (T)0;
            ticks[i] += 1;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(kBlock)
copter_reset_force_kernel(const __grid_constant__ KParams<T> kp, T* out, const uint32_t* episode,
                          int64_t n, int64_t env_offset, uint64_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock) {
        T f[3];
        reset_force<T>(kp, seed, (uint64_t)(env_offset + i), episode ? episode[i] : 0u, f);
        out[3 * i] = f[0]; out[3 * i + 1] = f[1]; out[3 * i + 2] = f[2];
    }
}

// ------------------------------------------------------------------------------------------
// host-side launch helpers
// ------------------------------------------------------------------------------------------
// Per-device caches (the library is re-entrant and the caller selects the device: nothing here may be
// remembered across devices).  Benign races: every thread that fills a slot writes the same value.
constexpr int kMaxDevices = 64;
int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return dev;
}
int sm_count() {
    static int sms[kMaxDevices] = {0};
    const int dev = current_device();
    if (sms[dev] == 0) {
        int q = 0;
        if (cudaDeviceGetAttribute(&q, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || q <= 0) q = 148;
        sms[dev] = q;
    }
    return sms[dev];
}
template <auto Kernel>
int ctas_per_sm(int block) {
    static int per_sm[kMaxDevices] = {0};
    const int dev = current_device();
    if (per_sm[dev] == 0) {
        int q = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, Kernel, block, 0) != cudaSuccess || q <= 0) q = 4;
        per_sm[dev] = q;
    }
    return per_sm[dev];
}

// Grid: one CTA per tile of kBlock envs, scheduled by the hardware as CTAs retire.  Measured on
// B200 (Lander3D fp32, 2^24 envs, K = 1): 6.7 TB/s, against 5.6 TB/s for a persistent grid of
// SMs x resident CTAs walking the tiles with a grid stride.  The loss is the static split (the SMs
// do not all see the same memory bandwidth; a persistent grid fed by cluster launch control is
// level with this shape -- DESIGN.md, "Grid shape"), so the hardware scheduler does the balancing.
// (profiles/README.md has the sweep.)  The other kernels keep their tile loop, so a grid capped at
// 2^31-1 CTAs still covers any n.
int grid_for(int64_t n) {
    const int64_t tiles = (n + kBlock - 1) / kBlock;
    const int64_t cap = (int64_t)0x7fffffff;
    return (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
}
// the step kernel has no tile loop: every tile needs its own CTA
constexpr int64_t kMaxEnvsPerLaunch = (int64_t)0x7fffffff * kBlock;

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// The state addressing of a call (include/copter_b200.h, "Memory layout"): vectors between planes (0: n) and between
// envs (0: 1).  False when the 12/V planes of the n envs would overlap.
template <typename T>
bool state_layout(int64_t n, int64_t state_stride, int64_t state_env_stride, int64_t& stride, int64_t& env_stride) {
    constexpr int64_t planes = 12 / Vec<T>::V;
    stride = state_stride > 0 ? state_stride : n;
    env_stride = state_env_stride > 0 ? state_env_stride : 1;
    return env_stride <= stride ? stride / env_stride >= n : env_stride / planes >= stride;
}

int check_params(const CopterParams* p, bool wide = false) {
    if (!p) return COPTER_E_ARG;
    if (p->max_steps < 1 || p->max_steps > (wide ? COPTER_MAX_STEPS_LIMIT_WIDE : COPTER_MAX_STEPS_LIMIT)) return COPTER_E_RANGE;
    if (!(p->M > 0) || !(p->Ix > 0) || !(p->Iy > 0) || !(p->Iz > 0) || !(p->fps > 0)) return COPTER_E_RANGE;
    return 0;
}

template <typename T, int VARIANT>
int launch_step_v(const KParams<T>& kp, const StepArgs<T>& a, cudaStream_t s) {
    if (a.stats) copter_step_kernel<T, VARIANT, true><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
    else         copter_step_kernel<T, VARIANT, false><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
    return (int)cudaGetLastError();
}

// `device_arrays`: every buffer is device memory (not step_host's mapped host arrays), the condition for the
// L2 prefetches of copter_step_kernel besides the ones launch_step checks itself.
template <typename T>
int launch_step(const CopterParams* p, const CopterBuffers* b, int64_t n, int64_t env_offset, uint64_t seed,
                int k, int variant, int flags, void* stream, bool device_arrays = true) {
    if (!b) return COPTER_E_ARG;
    int e = check_params(p, b->meta_hi != nullptr);
    if (e) return e;
    if (!b->state || !b->meta || !b->action || !b->reward || !b->done) return COPTER_E_ARG;
    StepArgs<T> a;
    if (n < 0 || n > kMaxEnvsPerLaunch || env_offset < 0 || k < 1 || !state_layout<T>(n, b->state_stride, b->state_env_stride, a.stride, a.env_stride)) return COPTER_E_RANGE;
    if (variant < 0 || variant >= COPTER_NUM_VARIANTS) return COPTER_E_VARIANT;
    if (!aligned16(b->state) || !aligned16(b->action) || (b->obs && !aligned16(b->obs))) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    const KParams<T> kp = make_kparams<T>(*p, b->meta_hi != nullptr);
    a.state = (T*)b->state; a.meta = b->meta; a.meta_hi = b->meta_hi; a.action = (const T*)b->action; a.obs = b->obs;
    a.reward = (T*)b->reward; a.done = b->done; a.init_force = (const T*)b->init_force;
    a.ep_return = (T*)b->ep_return; a.stats = b->stats; a.final_obs = b->final_obs; a.cause = b->cause;
    a.n = n; a.env_offset = env_offset; a.seed = seed; a.k = k; a.auto_reset = (flags & COPTER_F_AUTO_RESET) ? 1 : 0;
    // fp32 K = 1 on device memory, rows or planes, 16-byte aligned: one wave of resident CTAs ahead (measured on B200:
    // half a wave is level with it, two waves lose 3 % -- profiles/k1_l2_prefetch_ab.txt)
    a.prefetch_ahead = 0;
    if (sizeof(T) == 4 && k == 1 && device_arrays && aligned16(b->meta) && ((a.stride == 1 && a.env_stride == 3) || a.env_stride == 1))
        a.prefetch_ahead = (int64_t)sm_count() * COPTER_STEP_CTAS_PER_SM;
    cudaStream_t s = (cudaStream_t)stream;
    switch (variant) {
        case COPTER_LANDER3D: return launch_step_v<T, COPTER_LANDER3D>(kp, a, s);
        case COPTER_LANDER2D: return launch_step_v<T, COPTER_LANDER2D>(kp, a, s);
        case COPTER_LANDER1D: return launch_step_v<T, COPTER_LANDER1D>(kp, a, s);
        case COPTER_HOVER3D:  return launch_step_v<T, COPTER_HOVER3D>(kp, a, s);
        case COPTER_HOVER2D:  return launch_step_v<T, COPTER_HOVER2D>(kp, a, s);
        case COPTER_HOVER1D:  return launch_step_v<T, COPTER_HOVER1D>(kp, a, s);
        default:              return launch_step_v<T, COPTER_TAKEOFF>(kp, a, s);
    }
}

template <typename T, int VARIANT, bool R>
int launch_rollout_vr(const KParams<T>& kp, const RolloutArgs<T>& a, cudaStream_t s) {
    if (a.src_kind == COPTER_SRC_PID) {
        if (a.stats) copter_rollout_kernel<T, VARIANT, true, 1, R><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
        else         copter_rollout_kernel<T, VARIANT, false, 1, R><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
    } else if (a.src_kind == COPTER_SRC_PID_HOVER) {
        if constexpr (Variant<VARIANT>::A == 4 && Variant<VARIANT>::O != 12) {
            return COPTER_E_VARIANT;          // the 3-D hover heuristic reads the yaw rate: full-state observation only
        } else {
            if (a.stats) copter_rollout_kernel<T, VARIANT, true, 2, R><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
            else         copter_rollout_kernel<T, VARIANT, false, 2, R><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
        }
    } else {
        if (a.stats) copter_rollout_kernel<T, VARIANT, true, 0, R><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
        else         copter_rollout_kernel<T, VARIANT, false, 0, R><<<grid_for(a.n), kBlock, 0, s>>>(kp, a);
    }
    return (int)cudaGetLastError();
}

// the RECORD instantiations only when an ending record is asked for
template <typename T, int VARIANT>
int launch_rollout_v(const KParams<T>& kp, const RolloutArgs<T>& a, cudaStream_t s) {
    return (a.cause_tn || a.final_obs_tn) ? launch_rollout_vr<T, VARIANT, true>(kp, a, s) : launch_rollout_vr<T, VARIANT, false>(kp, a, s);
}

template <typename T>
int launch_rollout(const CopterParams* p, const CopterBuffers* b, const CopterActionSource* src, int64_t n,
                   int64_t env_offset, uint64_t seed, int64_t first_step, int n_steps, int variant, int flags,
                   void* reward_tn, uint8_t* done_tn, void* action_tn, const CopterPidGains* gains, void* controller,
                   uint8_t* cause_tn, float* final_obs_tn, void* stream) {
    if (!b) return COPTER_E_ARG;
    int e = check_params(p, b->meta_hi != nullptr);
    if (e) return e;
    if (!b->state || !b->meta || !src) return COPTER_E_ARG;
    if ((src->kind == COPTER_SRC_PID || src->kind == COPTER_SRC_PID_HOVER) && (!controller || !aligned16(controller))) return COPTER_E_ARG;
    RolloutArgs<T> a;
    if (n < 0 || env_offset < 0 || n_steps < 1 || first_step < 0 || !state_layout<T>(n, b->state_stride, b->state_env_stride, a.stride, a.env_stride)) return COPTER_E_RANGE;
    if (src->kind < COPTER_SRC_CONST || src->kind > COPTER_SRC_PID_HOVER) return COPTER_E_RANGE;
    if (variant < 0 || variant >= COPTER_NUM_VARIANTS) return COPTER_E_VARIANT;
    if (!aligned16(b->state) || (b->obs && !aligned16(b->obs))) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    const KParams<T> kp = make_kparams<T>(*p, b->meta_hi != nullptr);
    a.state = (T*)b->state; a.meta = b->meta; a.meta_hi = b->meta_hi; a.obs = b->obs; a.reward_sum = (T*)b->reward; a.done_any = b->done;
    a.init_force = (const T*)b->init_force; a.ep_return = (T*)b->ep_return; a.stats = b->stats;
    a.reward_tn = (T*)reward_tn; a.done_tn = done_tn; a.action_tn = (T*)action_tn; a.cause_tn = cause_tn; a.final_obs_tn = final_obs_tn;
    a.n = n; a.env_offset = env_offset; a.first_step = first_step;
    a.seed = seed; a.n_steps = n_steps; a.auto_reset = (flags & COPTER_F_AUTO_RESET) ? 1 : 0;
    a.src_kind = src->kind; a.src_scale = (T)src->scale; a.src_offset = (T)src->offset;
    CopterPidGains g;
    if (gains) g = *gains; else copter_default_pid_gains(&g);
    a.controller = (T*)controller;
    a.rate_kp = (T)g.rate_kp; a.rate_ki = (T)g.rate_ki; a.rate_kd = (T)g.rate_kd; a.rate_windup = (T)g.rate_windup; a.rate_big = (T)g.rate_big;
    a.pos_kp = (T)g.pos_kp; a.pos_ki = (T)g.pos_ki; a.pos_kd = (T)g.pos_kd; a.pos_windup = (T)g.pos_windup; a.pos_target = (T)g.pos_target;
    a.descent_kp = (T)g.descent_kp; a.descent_kd = (T)g.descent_kd;
    a.alt_kp = (T)g.alt_kp; a.alt_ki = (T)g.alt_ki; a.alt_kd = (T)g.alt_kd; a.alt_windup = (T)g.alt_windup; a.alt_target = (T)g.alt_target;
    cudaStream_t s = (cudaStream_t)stream;
    switch (variant) {
        case COPTER_LANDER3D: return launch_rollout_v<T, COPTER_LANDER3D>(kp, a, s);
        case COPTER_LANDER2D: return launch_rollout_v<T, COPTER_LANDER2D>(kp, a, s);
        case COPTER_LANDER1D: return launch_rollout_v<T, COPTER_LANDER1D>(kp, a, s);
        case COPTER_HOVER3D:  return launch_rollout_v<T, COPTER_HOVER3D>(kp, a, s);
        case COPTER_HOVER2D:  return launch_rollout_v<T, COPTER_HOVER2D>(kp, a, s);
        case COPTER_HOVER1D:  return launch_rollout_v<T, COPTER_HOVER1D>(kp, a, s);
        default:              return launch_rollout_v<T, COPTER_TAKEOFF>(kp, a, s);
    }
}

template <typename T, int VARIANT>
int launch_reset_v(const KParams<T>& kp, const CopterBuffers* b, int64_t n, int64_t stride, int64_t env_stride, int keep_episode, cudaStream_t s) {
    copter_reset_kernel<T, VARIANT><<<grid_for(n), kBlock, 0, s>>>(kp, (T*)b->state, b->meta, b->meta_hi, b->obs, (T*)b->ep_return, n, stride, env_stride, keep_episode);
    return (int)cudaGetLastError();
}

template <typename T>
int launch_reset(const CopterParams* p, const CopterBuffers* b, int64_t n, int variant, int flags, void* stream) {
    if (!b) return COPTER_E_ARG;
    int e = check_params(p, b->meta_hi != nullptr);
    if (e) return e;
    if (!b->state || !b->meta) return COPTER_E_ARG;
    int64_t stride, env_stride;
    if (n < 0 || !state_layout<T>(n, b->state_stride, b->state_env_stride, stride, env_stride)) return COPTER_E_RANGE;
    if (variant < 0 || variant >= COPTER_NUM_VARIANTS) return COPTER_E_VARIANT;
    if (!aligned16(b->state) || (b->obs && !aligned16(b->obs))) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    const KParams<T> kp = make_kparams<T>(*p, b->meta_hi != nullptr);
    const int keep = (flags & COPTER_F_KEEP_EPISODE) ? 1 : 0;
    cudaStream_t s = (cudaStream_t)stream;
    switch (variant) {
        case COPTER_LANDER3D: return launch_reset_v<T, COPTER_LANDER3D>(kp, b, n, stride, env_stride, keep, s);
        case COPTER_LANDER2D: return launch_reset_v<T, COPTER_LANDER2D>(kp, b, n, stride, env_stride, keep, s);
        case COPTER_LANDER1D: return launch_reset_v<T, COPTER_LANDER1D>(kp, b, n, stride, env_stride, keep, s);
        case COPTER_HOVER3D:  return launch_reset_v<T, COPTER_HOVER3D>(kp, b, n, stride, env_stride, keep, s);
        case COPTER_HOVER2D:  return launch_reset_v<T, COPTER_HOVER2D>(kp, b, n, stride, env_stride, keep, s);
        case COPTER_HOVER1D:  return launch_reset_v<T, COPTER_HOVER1D>(kp, b, n, stride, env_stride, keep, s);
        default:              return launch_reset_v<T, COPTER_TAKEOFF>(kp, b, n, stride, env_stride, keep, s);
    }
}

template <typename T>
int launch_dynamics(const CopterParams* p, void* state, uint8_t* status, int32_t* ticks, void* perturb,
                    const void* motors, int64_t n, void* stream) {
    int e = check_params(p);
    if (e) return e;
    if (!state || !status || !ticks || !perturb || !motors) return COPTER_E_ARG;
    if (n < 0) return COPTER_E_RANGE;
    if (!aligned16(state)) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    const KParams<T> kp = make_kparams<T>(*p);
    copter_dynamics_kernel<T><<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(kp, (T*)state, status, ticks, (T*)perturb, (const T*)motors, n);
    return (int)cudaGetLastError();
}

template <typename T>
int launch_reset_force(const CopterParams* p, T* out, const uint32_t* episode, int64_t n, int64_t env_offset,
                       uint64_t seed, void* stream) {
    int e = check_params(p);
    if (e) return e;
    if (!out) return COPTER_E_ARG;
    if (n < 0 || env_offset < 0) return COPTER_E_RANGE;
    if (n == 0) return 0;
    const KParams<T> kp = make_kparams<T>(*p);
    copter_reset_force_kernel<T><<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(kp, out, episode, n, env_offset, seed);
    return (int)cudaGetLastError();
}

// persistent grids for the policy kernels: the weights are converted to bf16 fragments once per CTA
template <auto Kernel>
int persistent_grid_for(int64_t n) {
    const int64_t tiles = (n + 127) / 128, cap = (int64_t)sm_count() * ctas_per_sm<Kernel>(128);
    return (int)(tiles < cap ? tiles : cap);
}

// Which policy kernel: 1 = tcgen05 / TMEM (copter_policy_tc.cuh, the default), 0 = warp-level mma.sync (copter_policy.cuh),
// from COPTER_B200_POLICY_TC in the environment (A/B runs, tests of both).
int policy_tc_setting() {
    const char* e = getenv("COPTER_B200_POLICY_TC");        // read on every call: tests and A/B runs flip it inside one process
    return e ? (atoi(e) != 0) : 1;
}
// The same choice for the fused policy + step rollout (copter_policy_rollout_f32).  Until the tcgen05 kernel took its
// tiles by cluster launch control and issued its MMAs warp-uniformly the warp-MMA kernel won (0.404 vs 0.424 ms per
// env-step at 2^23 envs); since then the tcgen05 kernel does (0.342 ms, 6 CTAs per SM), so it is the default.
int policy_rollout_tc_setting() {
    const char* e = getenv("COPTER_B200_POLICY_ROLLOUT_TC");
    return e ? (atoi(e) != 0) : 1;
}

template <int VARIANT>
int launch_policy_v(const PolicyArgs& a, cudaStream_t s) {
    using V = Variant<VARIANT>;
    if (policy_tc_setting()) {
        tc::Args t;
        t.state = a.state; t.stride = a.stride; t.env_stride = a.env_stride; t.n = a.n;
        t.w1 = a.w.w1; t.b1 = a.w.b1; t.w2 = a.w.w2; t.b2 = a.w.b2; t.w3 = a.w.w3; t.b3 = a.w.b3;
        t.out_scale = a.w.out_scale; t.out_offset = a.w.out_offset; t.action = a.action;
        constexpr auto kernel = tc::copter_mlp_policy_tc_kernel<V::first, V::O, V::A>;
        constexpr int smem = (int)sizeof(tc::Smem) + 128;                     // dynamic: past the 48 KB static limit
        static bool configured[kMaxDevices] = {false};
        const int dev = current_device();
        if (!configured[dev]) {
            if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return (int)cudaGetLastError();
            configured[dev] = true;
        }
        const int64_t tiles = (a.n + tc::kTile - 1) / tc::kTile;
        // cluster launch control: one CTA per tile in the grid, the resident CTAs take the pending ones over
        kernel<<<(int)tiles, tc::kThreads, smem, s>>>(t);
        return (int)cudaGetLastError();
    }
    copter_mlp_policy_kernel<V::first, V::O, V::A><<<persistent_grid_for<copter_mlp_policy_kernel<V::first, V::O, V::A>>(a.n), 128, 0, s>>>(a);
    return (int)cudaGetLastError();
}

// the critic: one instantiation per observation size (Variant<>: 2, 6, 10, 12)
template <int OBS>
int launch_value_o(const tc::ValueArgs& a, cudaStream_t s) {
    constexpr auto kernel = tc::copter_value_tc_kernel<OBS>;
    constexpr int smem = (int)sizeof(tc::Smem) + 128;
    static bool configured[kMaxDevices] = {false};
    const int dev = current_device();
    if (!configured[dev]) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return (int)cudaGetLastError();
        configured[dev] = true;
    }
    const int64_t tiles = (a.n + tc::kTile - 1) / tc::kTile;
    kernel<<<(int)tiles, tc::kThreads, smem, s>>>(a);                // cluster launch control, as above
    return (int)cudaGetLastError();
}

template <int VARIANT, bool STATS, bool RECORD>
int launch_policy_rollout_tc(const KParams<float>& kp, const PolicyRolloutArgs& a, cudaStream_t s) {
    constexpr auto kernel = copter_policy_rollout_tc_kernel<VARIANT, STATS, RECORD>;
    constexpr int smem = (int)sizeof(RolloutTcSmem) + 128;                     // dynamic: past the 48 KB static limit
    static bool configured[kMaxDevices] = {false};
    const int dev = current_device();
    if (!configured[dev]) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return (int)cudaGetLastError();
        configured[dev] = true;
    }
    const int64_t tiles = (a.n + tc::kTile - 1) / tc::kTile;
    kernel<<<(int)tiles, tc::kThreads, smem, s>>>(kp, a);           // cluster launch control, as above
    return (int)cudaGetLastError();
}

template <int VARIANT, bool R>
int launch_policy_rollout_vr(const KParams<float>& kp, const PolicyRolloutArgs& a, cudaStream_t s) {
    if (policy_rollout_tc_setting())    // the tcgen05 / TMEM kernel (the default); otherwise the warp-MMA kernel
        return a.stats ? launch_policy_rollout_tc<VARIANT, true, R>(kp, a, s) : launch_policy_rollout_tc<VARIANT, false, R>(kp, a, s);
    if (a.stats) copter_policy_rollout_kernel<VARIANT, true, R><<<persistent_grid_for<copter_policy_rollout_kernel<VARIANT, true, R>>(a.n), 128, 0, s>>>(kp, a);
    else         copter_policy_rollout_kernel<VARIANT, false, R><<<persistent_grid_for<copter_policy_rollout_kernel<VARIANT, false, R>>(a.n), 128, 0, s>>>(kp, a);
    return (int)cudaGetLastError();
}

// the RECORD instantiations only when an ending record is asked for
template <int VARIANT>
int launch_policy_rollout_v(const KParams<float>& kp, const PolicyRolloutArgs& a, cudaStream_t s) {
    return (a.cause_tn || a.final_obs_tn) ? launch_policy_rollout_vr<VARIANT, true>(kp, a, s) : launch_policy_rollout_vr<VARIANT, false>(kp, a, s);
}

bool policy_ok(const CopterMlpPolicy* m) {
    return m && m->w1 && m->b1 && m->w2 && m->b2 && m->w3 && m->b3;
}
PolicyWeights policy_weights(const CopterMlpPolicy* m) {
    PolicyWeights w;
    w.w1 = m->w1; w.b1 = m->b1; w.w2 = m->w2; w.b2 = m->b2; w.w3 = m->w3; w.b3 = m->b3;
    w.out_scale = m->out_scale; w.out_offset = m->out_offset;
    return w;
}

// ------------------------------------------------------------------------------------------
// host-buffer pipeline: the step for callers that hold numpy-style HOST arrays
// ------------------------------------------------------------------------------------------
struct Pipeline {
    int n_streams, device;
    cudaStream_t streams[8];
    cudaEvent_t start, done[8];
};

// A small shard is a latency problem, not a bandwidth one (the single-env facade: BASELINE.json configs[0]).  When
// every host array is page-locked and mapped into the device's address space (cudaHostAlloc / cudaHostRegister under
// unified addressing -- what torch's pin_memory() gives), the step kernel reads the commands from and writes its
// results to the HOST arrays directly: one launch and one stream synchronisation instead of an event, a copy in, a
// launch, three to five copies out and their events.  The device-side action / obs / reward / done buffers of `dev`
// are not touched on this path (state and counters are, of course).  Measured (profiles/r2_direct_path_sweep.txt, us per
// step_host call, copy pipeline -> direct): 1 env 37 -> 21, 4096 envs 50 -> 27, 65 536 envs 168 -> 128, 2^20 envs 2201 ->
// 1999, 2^22 level, 2^24 33.2 -> 33.9 ms (the chunked pipeline wins once the transfers dominate).  The limit is
// COPTER_DIRECT_MAX_ENVS, or COPTER_B200_DIRECT_MAX_ENVS in the environment (read once; 0 switches the path off).
#ifndef COPTER_DIRECT_MAX_ENVS
#define COPTER_DIRECT_MAX_ENVS 65536
#endif
// device address of a page-locked, mapped host array, or nullptr (asked on every call: an address seen before may
// belong to a different, pageable allocation by now)
static void* mapped_device_pointer(const void* host) {
    if (!host) return nullptr;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return attr.type == cudaMemoryTypeHost ? attr.devicePointer : nullptr;
}

template <typename T>
int step_host(Pipeline* pl, const CopterParams* p, const CopterBuffers* dev, const void* h_action, float* h_obs,
              void* h_reward, uint8_t* h_done, uint8_t* h_cause, float* h_final_obs, int64_t n, int64_t env_offset, uint64_t seed, int k, int variant,
              int flags, int64_t chunk, void* caller_stream) {
    if (!pl || !dev || !h_action || !h_reward || !h_done || !dev->action) return COPTER_E_ARG;
    if (variant < 0 || variant >= COPTER_NUM_VARIANTS) return COPTER_E_VARIANT;
    if (n < 0 || chunk <= 0) return COPTER_E_RANGE;
    const int O = copter_obs_size(variant), A = copter_action_size(variant);
    constexpr int V = Vec<T>::V;
    chunk = (chunk + 255) / 256 * 256;                    // keeps every sub-shard 16-byte aligned
    int64_t stride, env_stride;
    if (!state_layout<T>(n, dev->state_stride, dev->state_env_stride, stride, env_stride)) return COPTER_E_RANGE;
    cudaError_t ce;
    static const int64_t direct_max = [] { const char* e = getenv("COPTER_B200_DIRECT_MAX_ENVS"); return e ? (int64_t)atoll(e) : (int64_t)COPTER_DIRECT_MAX_ENVS; }();
    if (n > 0 && n <= direct_max) {                       // the direct path: see mapped_device_pointer
        const bool want_obs = h_obs && dev->obs, want_cause = h_cause && dev->cause, want_final = h_final_obs && dev->final_obs;
        void* d_action = mapped_device_pointer(h_action);
        void* d_reward = mapped_device_pointer(h_reward);
        void* d_done = mapped_device_pointer(h_done);
        void* d_obs = want_obs ? mapped_device_pointer(h_obs) : nullptr;
        void* d_cause = want_cause ? mapped_device_pointer(h_cause) : nullptr;
        void* d_final = want_final ? mapped_device_pointer(h_final_obs) : nullptr;
        if (d_action && d_reward && d_done && (!want_obs || d_obs) && (!want_cause || d_cause) && (!want_final || d_final) &&
            aligned16(d_action) && (!d_obs || aligned16(d_obs))) {
            CopterBuffers b = *dev;
            b.state_stride = stride;
            b.action = d_action; b.reward = d_reward; b.done = (uint8_t*)d_done;
            b.obs = want_obs ? (float*)d_obs : (dev->obs ? dev->obs : nullptr);
            b.cause = want_cause ? (uint8_t*)d_cause : dev->cause;
            b.final_obs = want_final ? (float*)d_final : dev->final_obs;
            const int e = launch_step<T>(p, &b, n, env_offset, seed, k, variant, flags, (cudaStream_t)caller_stream, false);
            if (e) return e;
            return (int)cudaStreamSynchronize((cudaStream_t)caller_stream);
        }
    }
    if ((ce = cudaEventRecord(pl->start, (cudaStream_t)caller_stream)) != cudaSuccess) return (int)ce;
    for (int s = 0; s < pl->n_streams; ++s)
        if ((ce = cudaStreamWaitEvent(pl->streams[s], pl->start, 0)) != cudaSuccess) return (int)ce;
    int c = 0;
    for (int64_t lo = 0; lo < n; lo += chunk, ++c) {
        const int64_t m = (n - lo < chunk) ? (n - lo) : chunk;
        cudaStream_t st = pl->streams[c % pl->n_streams];
        CopterBuffers b = *dev;
        b.state = (T*)dev->state + lo * env_stride * V;  // same layout, shifted by `lo` envs
        b.state_stride = stride;
        b.meta = dev->meta + lo;
        b.meta_hi = dev->meta_hi ? dev->meta_hi + lo : nullptr;
        b.action = (const T*)dev->action + lo * A;
        b.obs = dev->obs ? dev->obs + lo * O : nullptr;
        b.reward = (T*)dev->reward + lo;
        b.done = dev->done + lo;
        b.init_force = dev->init_force ? (const T*)dev->init_force + lo * 3 : nullptr;
        b.ep_return = dev->ep_return ? (T*)dev->ep_return + lo : nullptr;
        b.final_obs = dev->final_obs ? dev->final_obs + lo * O : nullptr;
        b.cause = dev->cause ? dev->cause + lo : nullptr;
        if ((ce = cudaMemcpyAsync((void*)b.action, (const T*)h_action + lo * A, sizeof(T) * m * A, cudaMemcpyHostToDevice, st)) != cudaSuccess) return (int)ce;
        const int e = launch_step<T>(p, &b, m, env_offset + lo, seed, k, variant, flags, st, false);
        if (e) return e;
        if (h_obs && b.obs && (ce = cudaMemcpyAsync(h_obs + lo * O, b.obs, sizeof(float) * m * O, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)ce;
        if ((ce = cudaMemcpyAsync((T*)h_reward + lo, b.reward, sizeof(T) * m, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)ce;
        if ((ce = cudaMemcpyAsync(h_done + lo, b.done, m, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)ce;
        if (h_cause && b.cause && (ce = cudaMemcpyAsync(h_cause + lo, b.cause, m, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)ce;
        if (h_final_obs && b.final_obs && (ce = cudaMemcpyAsync(h_final_obs + lo * O, b.final_obs, sizeof(float) * m * O, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return (int)ce;
    }
    for (int s = 0; s < pl->n_streams; ++s) {
        if ((ce = cudaEventRecord(pl->done[s], pl->streams[s])) != cudaSuccess) return (int)ce;
        if ((ce = cudaStreamWaitEvent((cudaStream_t)caller_stream, pl->done[s], 0)) != cudaSuccess) return (int)ce;
    }
    for (int s = 0; s < pl->n_streams; ++s)
        if ((ce = cudaStreamSynchronize(pl->streams[s])) != cudaSuccess) return (int)ce;
    return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int copter_abi_version(void) { return COPTER_ABI_VERSION; }

void copter_default_params(CopterParams* p) {
    if (!p) return;
    p->B = 5.E-03; p->D = 2.E-06; p->M = 1.380; p->L = 0.350;           // dji_phantom.py:12-17
    p->Ix = 2; p->Iy = 2; p->Iz = 3; p->Jr = 38E-04; p->maxrpm = 15000;  // dji_phantom.py:20-25
    p->landing_vel_x = 2.0; p->landing_vel_y = 1.0; p->landing_angle = M_PI / 4; p->G = 9.80665;   // dynamics:71-76
    p->fps = 100; p->initial_random_force = 30; p->out_of_bounds_penalty = 100;                    // task.py:25,32-38
    p->max_angle_deg = 45; p->bounds = 10; p->initial_altitude = 10; p->max_steps = 1000;
    p->target_radius = 2; p->yaw_penalty_factor = 50; p->xyz_penalty_factor = 25;                  // lander.py:17-23
    p->dz_max = 10; p->dz_penalty = 100; p->inside_radius_bonus = 100;
    p->rho = 1.225; p->lift_coefficient = 0.4;      // attic/mars/dynamics/__init__.py:83-84, ingenuity.py:55
    p->takeoff_target_altitude = 5;                 // attic/gym_copter/envs/takeoff.py:20
    p->dynamics_model = 0;
}

int copter_obs_size(int variant) {
    static const int o[COPTER_NUM_VARIANTS] = {10, 6, 2, 12, 6, 2, 10};
    return (variant < 0 || variant >= COPTER_NUM_VARIANTS) ? COPTER_E_VARIANT : o[variant];
}

int copter_action_size(int variant) {
    static const int a[COPTER_NUM_VARIANTS] = {4, 2, 1, 4, 2, 1, 4};
    return (variant < 0 || variant >= COPTER_NUM_VARIANTS) ? COPTER_E_VARIANT : a[variant];
}

int copter_reset_f32(const CopterParams* p, const CopterBuffers* b, int64_t n, int variant, int flags, void* stream) { return launch_reset<float>(p, b, n, variant, flags, stream); }
int copter_reset_f64(const CopterParams* p, const CopterBuffers* b, int64_t n, int variant, int flags, void* stream) { return launch_reset<double>(p, b, n, variant, flags, stream); }

int copter_step_f32(const CopterParams* p, const CopterBuffers* b, int64_t n, int64_t env_offset, uint64_t seed, int k, int variant, int flags, void* stream) {
    return launch_step<float>(p, b, n, env_offset, seed, k, variant, flags, stream);
}
int copter_step_f64(const CopterParams* p, const CopterBuffers* b, int64_t n, int64_t env_offset, uint64_t seed, int k, int variant, int flags, void* stream) {
    return launch_step<double>(p, b, n, env_offset, seed, k, variant, flags, stream);
}

int copter_rollout_f32(const CopterParams* p, const CopterBuffers* b, const CopterActionSource* src, int64_t n, int64_t env_offset, uint64_t seed,
                       int64_t first_step, int n_steps, int variant, int flags, float* reward_tn, uint8_t* done_tn, float* action_tn,
                       const CopterPidGains* gains, float* controller, uint8_t* cause_tn, float* final_obs_tn, void* stream) {
    return launch_rollout<float>(p, b, src, n, env_offset, seed, first_step, n_steps, variant, flags, reward_tn, done_tn, action_tn, gains, controller,
                              cause_tn, final_obs_tn, stream);
}
int copter_rollout_f64(const CopterParams* p, const CopterBuffers* b, const CopterActionSource* src, int64_t n, int64_t env_offset, uint64_t seed,
                       int64_t first_step, int n_steps, int variant, int flags, double* reward_tn, uint8_t* done_tn, double* action_tn,
                       const CopterPidGains* gains, double* controller, uint8_t* cause_tn, float* final_obs_tn, void* stream) {
    return launch_rollout<double>(p, b, src, n, env_offset, seed, first_step, n_steps, variant, flags, reward_tn, done_tn, action_tn, gains, controller,
                              cause_tn, final_obs_tn, stream);
}

void copter_default_pid_gains(CopterPidGains* g) {
    if (!g) return;
    g->rate_kp = 1.0; g->rate_ki = 0.0; g->rate_kd = 1.0; g->rate_windup = 6.0;          // AngularVelocityPidController (:126-135)
    g->rate_big = 40.0 * M_PI / 180.0;                                                    // BIG_DEGREES_PER_SECOND
    g->pos_kp = 0.00001; g->pos_ki = 0.1; g->pos_kd = 4.0; g->pos_windup = 0.2; g->pos_target = 0.0;   // PositionHoldPidController (:102-107)
    g->descent_kp = 1.15; g->descent_kd = 1.33;                                           // DescentPidController (:110-121)
    g->alt_kp = 0.2; g->alt_ki = 3.0; g->alt_kd = 0.0; g->alt_windup = 0.2; g->alt_target = 5.0;       // AltitudeHoldPidController (:93), windup :14
}

int copter_dynamics_f32(const CopterParams* p, void* state, uint8_t* status, int32_t* ticks, void* perturb, const void* motors, int64_t n, void* stream) {
    return launch_dynamics<float>(p, state, status, ticks, perturb, motors, n, stream);
}
int copter_dynamics_f64(const CopterParams* p, void* state, uint8_t* status, int32_t* ticks, void* perturb, const void* motors, int64_t n, void* stream) {
    return launch_dynamics<double>(p, state, status, ticks, perturb, motors, n, stream);
}

int copter_reset_force_f32(const CopterParams* p, float* out, const uint32_t* ep, int64_t n, int64_t env_offset, uint64_t seed, void* stream) {
    return launch_reset_force<float>(p, out, ep, n, env_offset, seed, stream);
}
int copter_reset_force_f64(const CopterParams* p, double* out, const uint32_t* ep, int64_t n, int64_t env_offset, uint64_t seed, void* stream) {
    return launch_reset_force<double>(p, out, ep, n, env_offset, seed, stream);
}

int copter_policy_mlp_f32(const void* state, int64_t state_stride, int64_t n, int variant, int hidden,
                          const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                          float out_scale, float out_offset, float* action, void* stream) {
    return copter_policy_mlp_strided_f32(state, state_stride, 0, n, variant, hidden, w1, b1, w2, b2, w3, b3, out_scale, out_offset, action, stream);
}

int copter_policy_mlp_strided_f32(const void* state, int64_t state_stride, int64_t state_env_stride, int64_t n, int variant, int hidden,
                                  const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                                  float out_scale, float out_offset, float* action, void* stream) {
    if (!state || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !action) return COPTER_E_ARG;
    if (variant < 0 || variant >= COPTER_NUM_VARIANTS) return COPTER_E_VARIANT;
    PolicyArgs a;
    if (n < 0 || hidden != kPolH || !state_layout<float>(n, state_stride, state_env_stride, a.stride, a.env_stride)) return COPTER_E_RANGE;
    if (!aligned16(state) || !aligned16(action)) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    a.state = (const float*)state; a.n = n;
    a.w.w1 = w1; a.w.b1 = b1; a.w.w2 = w2; a.w.b2 = b2; a.w.w3 = w3; a.w.b3 = b3;
    a.w.out_scale = out_scale; a.w.out_offset = out_offset; a.action = action;
    cudaStream_t s = (cudaStream_t)stream;
    switch (variant) {
        case COPTER_LANDER3D: return launch_policy_v<COPTER_LANDER3D>(a, s);
        case COPTER_LANDER2D: return launch_policy_v<COPTER_LANDER2D>(a, s);
        case COPTER_LANDER1D: return launch_policy_v<COPTER_LANDER1D>(a, s);
        case COPTER_HOVER3D:  return launch_policy_v<COPTER_HOVER3D>(a, s);
        case COPTER_HOVER2D:  return launch_policy_v<COPTER_HOVER2D>(a, s);
        case COPTER_HOVER1D:  return launch_policy_v<COPTER_HOVER1D>(a, s);
        default:              return launch_policy_v<COPTER_TAKEOFF>(a, s);
    }
}

int copter_policy_rollout_f32(const CopterParams* p, const CopterBuffers* b, const CopterMlpPolicy* policy, int64_t n,
                              int64_t env_offset, uint64_t seed, int64_t first_step, int n_steps, int variant, int flags,
                              float* reward_tn, uint8_t* done_tn, float* action_tn, float* obs_tn, uint8_t* cause_tn,
                              float* final_obs_tn, void* stream) {
    if (!b) return COPTER_E_ARG;
    int e = check_params(p, b->meta_hi != nullptr);
    if (e) return e;
    if (!b->state || !b->meta || !policy_ok(policy)) return COPTER_E_ARG;
    PolicyRolloutArgs a;
    if (n < 0 || env_offset < 0 || first_step < 0 || n_steps < 1 || policy->hidden != kPolH ||
        !state_layout<float>(n, b->state_stride, b->state_env_stride, a.stride, a.env_stride)) return COPTER_E_RANGE;
    if (variant < 0 || variant >= COPTER_NUM_VARIANTS) return COPTER_E_VARIANT;
    if (!aligned16(b->state) || (b->obs && !aligned16(b->obs)) || (action_tn && !aligned16(action_tn)) || (obs_tn && !aligned16(obs_tn))) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    const KParams<float> kp = make_kparams<float>(*p, b->meta_hi != nullptr);
    a.state = (float*)b->state; a.meta = b->meta; a.meta_hi = b->meta_hi; a.obs = b->obs; a.reward_sum = (float*)b->reward; a.done_any = b->done;
    a.init_force = (const float*)b->init_force; a.ep_return = (float*)b->ep_return; a.stats = b->stats;
    a.reward_tn = reward_tn; a.done_tn = done_tn; a.action_tn = action_tn; a.obs_tn = obs_tn;
    a.cause_tn = cause_tn; a.final_obs_tn = final_obs_tn;
    a.n = n; a.env_offset = env_offset; a.seed = seed;
    a.first_step = first_step; a.n_steps = n_steps; a.auto_reset = (flags & COPTER_F_AUTO_RESET) ? 1 : 0;
    a.w = policy_weights(policy); a.action_std = policy->action_std;
    cudaStream_t s = (cudaStream_t)stream;
    switch (variant) {
        case COPTER_LANDER3D: return launch_policy_rollout_v<COPTER_LANDER3D>(kp, a, s);
        case COPTER_LANDER2D: return launch_policy_rollout_v<COPTER_LANDER2D>(kp, a, s);
        case COPTER_LANDER1D: return launch_policy_rollout_v<COPTER_LANDER1D>(kp, a, s);
        case COPTER_HOVER3D:  return launch_policy_rollout_v<COPTER_HOVER3D>(kp, a, s);
        case COPTER_HOVER2D:  return launch_policy_rollout_v<COPTER_HOVER2D>(kp, a, s);
        case COPTER_HOVER1D:  return launch_policy_rollout_v<COPTER_HOVER1D>(kp, a, s);
        default:              return launch_policy_rollout_v<COPTER_TAKEOFF>(kp, a, s);
    }
}

int copter_gae_f32(const float* reward_tn, const float* value_tn, const float* last_value, const uint8_t* cause_tn,
                   const float* final_value_tn, int64_t n, int n_steps, float gamma, float lam, float* adv_tn, float* ret_tn,
                   void* stream) {
    if (!reward_tn || !value_tn || !last_value || !cause_tn || !adv_tn || n < 0 || n_steps < 1) return COPTER_E_ARG;
    if (n == 0) return 0;
    const int64_t blocks = (n + kGaeBlock - 1) / kGaeBlock;
    if (blocks > 0x7fffffff) return COPTER_E_RANGE;
    GaeArgs a;
    a.reward = reward_tn; a.value = value_tn; a.last_value = last_value; a.cause = cause_tn; a.final_value = final_value_tn;
    a.adv = adv_tn; a.ret = ret_tn; a.n = n; a.n_steps = n_steps; a.gamma = gamma; a.lam = lam;
    copter_gae_kernel<<<(int)blocks, kGaeBlock, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

int copter_value_mlp_f32(const float* rows, int64_t row_stride, int64_t m, int variant, int hidden,
                         const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3,
                         const uint8_t* select, uint32_t select_mask, float* value, void* stream) {
    if (!rows || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !value || m < 0) return COPTER_E_ARG;
    const int obs = copter_obs_size(variant);
    if (obs < 0) return COPTER_E_VARIANT;
    if (row_stride < obs || hidden != kPolH || (m + tc::kTile - 1) / tc::kTile > 0x7fffffff) return COPTER_E_RANGE;
    for (const void* ptr : {(const void*)rows, (const void*)w1, (const void*)b1, (const void*)w2, (const void*)b2, (const void*)w3,
                            (const void*)b3, (const void*)value})
        if (reinterpret_cast<uintptr_t>(ptr) & 3u) return COPTER_E_ALIGN;
    if (m == 0) return 0;
    tc::ValueArgs a;
    a.rows = rows; a.row_stride = row_stride; a.n = m; a.select = select; a.select_mask = select_mask;
    a.w1 = w1; a.b1 = b1; a.w2 = w2; a.b2 = b2; a.w3 = w3; a.b3 = b3; a.value = value;
    cudaStream_t s = (cudaStream_t)stream;
    switch (obs) {
        case 2:  return launch_value_o<2>(a, s);
        case 6:  return launch_value_o<6>(a, s);
        case 10: return launch_value_o<10>(a, s);
        default: return launch_value_o<12>(a, s);
    }
}

int copter_policy_logp_f32(uint64_t seed, int64_t env_offset, int64_t n, int64_t first_step, int n_steps, int variant,
                           const float* action_std, float* logp_tn, void* stream) {
    if (!action_std || !logp_tn || n < 0 || n_steps < 1) return COPTER_E_ARG;
    const int act = copter_action_size(variant);
    if (act < 0) return COPTER_E_VARIANT;
    if (env_offset < 0 || first_step < 0 || (n + kLogpBlock - 1) / kLogpBlock > 0x7fffffff) return COPTER_E_RANGE;
    if ((reinterpret_cast<uintptr_t>(action_std) & 3u) || (reinterpret_cast<uintptr_t>(logp_tn) & 3u)) return COPTER_E_ALIGN;
    if (n == 0) return 0;
    LogpArgs a;
    a.seed = seed; a.env_offset = env_offset; a.n = n; a.first_step = first_step; a.n_steps = n_steps;
    a.action_std = action_std; a.logp = logp_tn;
    const int blocks = (int)((n + kLogpBlock - 1) / kLogpBlock);
    cudaStream_t s = (cudaStream_t)stream;
    if (act == 4) copter_policy_logp_kernel<4><<<blocks, kLogpBlock, 0, s>>>(a);
    else if (act == 2) copter_policy_logp_kernel<2><<<blocks, kLogpBlock, 0, s>>>(a);
    else copter_policy_logp_kernel<1><<<blocks, kLogpBlock, 0, s>>>(a);
    return (int)cudaGetLastError();
}

int copter_pipeline_create(int n_streams, void** out) {
    if (!out || n_streams < 1 || n_streams > 8) return COPTER_E_ARG;
    Pipeline* pl = new Pipeline();
    pl->n_streams = 0;
    pl->device = 0;
    cudaError_t ce = cudaGetDevice(&pl->device);
    bool have_start = false;
    if (ce == cudaSuccess) { ce = cudaEventCreateWithFlags(&pl->start, cudaEventDisableTiming); have_start = ce == cudaSuccess; }
    for (int s = 0; s < n_streams && ce == cudaSuccess; ++s) {
        ce = cudaStreamCreateWithFlags(&pl->streams[s], cudaStreamNonBlocking);
        if (ce != cudaSuccess) break;
        ce = cudaEventCreateWithFlags(&pl->done[s], cudaEventDisableTiming);
        if (ce != cudaSuccess) { cudaStreamDestroy(pl->streams[s]); break; }
        pl->n_streams = s + 1;                       // stream s and its event both exist
    }
    if (ce != cudaSuccess) {                         // release what was created before the failure
        for (int s = 0; s < pl->n_streams; ++s) { cudaStreamDestroy(pl->streams[s]); cudaEventDestroy(pl->done[s]); }
        if (have_start) cudaEventDestroy(pl->start);
        delete pl;
        return (int)ce;
    }
    *out = pl;
    return 0;
}

int copter_pipeline_destroy(void* pipeline) {
    Pipeline* pl = (Pipeline*)pipeline;
    if (!pl) return COPTER_E_ARG;
    int prev = -1;                                   // the streams belong to the device that was current at creation
    if (cudaGetDevice(&prev) == cudaSuccess && prev != pl->device) cudaSetDevice(pl->device); else prev = -1;
    for (int s = 0; s < pl->n_streams; ++s) { cudaStreamDestroy(pl->streams[s]); cudaEventDestroy(pl->done[s]); }
    cudaEventDestroy(pl->start);
    if (prev >= 0) cudaSetDevice(prev);
    delete pl;
    return 0;
}

int copter_step_host_f32(void* pipeline, const CopterParams* p, const CopterBuffers* dev, const float* h_action, float* h_obs,
                         float* h_reward, uint8_t* h_done, uint8_t* h_cause, float* h_final_obs, int64_t n, int64_t env_offset,
                         uint64_t seed, int k, int variant, int flags, int64_t chunk_envs, void* stream) {
    return step_host<float>((Pipeline*)pipeline, p, dev, h_action, h_obs, h_reward, h_done, h_cause, h_final_obs, n, env_offset, seed, k, variant, flags, chunk_envs, stream);
}
int copter_step_host_f64(void* pipeline, const CopterParams* p, const CopterBuffers* dev, const double* h_action, float* h_obs,
                         double* h_reward, uint8_t* h_done, uint8_t* h_cause, float* h_final_obs, int64_t n, int64_t env_offset,
                         uint64_t seed, int k, int variant, int flags, int64_t chunk_envs, void* stream) {
    return step_host<double>((Pipeline*)pipeline, p, dev, h_action, h_obs, h_reward, h_done, h_cause, h_final_obs, n, env_offset, seed, k, variant, flags, chunk_envs, stream);
}

}  // extern "C"
