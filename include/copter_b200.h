/*
 * copter_b200.h -- C ABI of libcopter_b200.so: the batched, B200-native (sm_100a) replacement
 * for the reference's per-env physics + env step.
 *
 * The reference (simondlevy/gym-copter) is pure Python and has no FFI of its own; the
 * boundary this library sits behind is its Python class API.  Each entry point below names
 * the reference interface it replaces (paths relative to the reference root):
 *
 *   copter_default_params      gym_copter/dynamics/vehicles/dji_phantom.py:9-26,
 *                              gym_copter/dynamics/__init__.py:71-76,
 *                              gym_copter/envs/task.py:25,32-38, gym_copter/envs/lander.py:17-23
 *   copter_reset_{f32,f64}     _Task._reset / Lander.reset      envs/task.py:145-197, envs/lander.py:35-37
 *   copter_step_{f32,f64}      _Task.step + Lander._get_reward/_get_state/_get_motors
 *                              envs/task.py:77-137, envs/lander.py:39-74,95-97
 *                              (which call Dynamics.setMotors, dynamics/__init__.py:114-197)
 *   copter_rollout_{f32,f64}   the caller's loop `for t: env.step(heuristic action)` (lander.py:40-64)
 *                              with the constant / --random command streams generated on the device
 *   copter_dynamics_{f32,f64}  Dynamics.setMotors driven directly (take-off style use)
 *                              dynamics/__init__.py:114-197,210-229
 *   copter_policy_mlp_f32,     the consumer's loop obs -> net -> clip -> env.step (attic/drl/3dtest.py:36-61):
 *   copter_policy_rollout_f32  the network alone, and network + step fused over a whole horizon
 *   copter_step_host_{f32,f64} the same step for callers holding HOST buffers (numpy actions as in
 *                              lander.py:42-44), host<->device copies pipelined inside the call
 *
 * Ownership: every device buffer is allocated and owned by the caller (PyTorch CUDA tensors
 * in the shipped host code).  The library never allocates device memory for the caller,
 * never frees, and never synchronises the stream it is given (copter_step_host_* is the one
 * exception: it returns after its own internal streams have drained).
 * Errors: every function returns 0 on success, a positive cudaError_t from the launch, or a
 * negative COPTER_E_* argument error.  No exceptions cross the ABI.
 * Threading: stateless and re-entrant; the caller selects the device (cudaSetDevice /
 * torch.cuda.device) and passes the stream.  Launches are asynchronous.
 *
 * Memory layout (N envs, T = float or double, V = 16/sizeof(T) elements per 128-bit vector):
 *   state   12/V 128-bit vectors per env; vector p (components pV .. pV+V-1) of env i is vector
 *                           p * state_stride + i * state_env_stride of the allocation
 *                           (CopterBuffers), so a thread reads its env with 12/V 128-bit loads.  Two layouts:
 *                             planes  T[12/V][N][V]  state_stride N, state_env_stride 1 (the default);
 *                             rows    T[N][12]       state_stride 1, state_env_stride 12/V: one 48- / 96-byte
 *                                                    row per env, whose components first .. first+O-1 are the
 *                                                    observation when T = float -- what a float32
 *                                                    CopterVecEnv keeps, so its steps pass obs = NULL and
 *                                                    write 40 bytes less (a float64 one keeps planes).
 *                           A warp's 12/V accesses cover one contiguous span in either layout.
 *                           Component order = the reference's state vector
 *                           (dynamics/__init__.py:48-59): x dx y dy z dz phi dphi theta dtheta psi dpsi.
 *   meta    uint32[N]       bits 0-1 flight status (COPTER_STATUS_*), bits 2-12 the env's
 *                           `steps` counter (envs/task.py:128-130; saturates at 2047), bits 13-31
 *                           episode index (wraps at 2^19; keys the reset-force stream).
 *   meta_hi uint32[N]       optional WIDE counters (the reference takes any max_steps, envs/task.py:35):
 *                           when CopterBuffers.meta_hi is given, meta holds status (bits 0-1) and a
 *                           30-bit steps counter (bits 2-31), meta_hi the 32-bit episode index; max_steps
 *                           may then be anything up to COPTER_MAX_STEPS_LIMIT_WIDE.  4 more bytes read
 *                           and written per env and launch; the default layout is unchanged.
 *   action  T[N][A]         row-major, A = action size of the variant.
 *   obs     float[N][O]     row-major float32 (envs/task.py:133), O = observation size.
 *   reward  T[N]; done uint8[N] (0/1).
 */
#ifndef COPTER_B200_H
#define COPTER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COPTER_ABI_VERSION 6

/* dynamics/__init__.py:65-68 */
enum { COPTER_STATUS_CRASHED = 0, COPTER_STATUS_LANDED = 1, COPTER_STATUS_LEVELING = 2, COPTER_STATUS_AIRBORNE = 3 };

/* env variants: the live Lander (= Lander3D) and the attic-defined projections (SURVEY.md 2.2) */
/* COPTER_TAKEOFF is the attic take-off env (attic/gym_copter/envs/takeoff.py:18-91): the 10-component
   observation, four motor commands handed to Dynamics.setMotors UNCLIPPED whatever the flight status
   (so a LANDED vehicle takes off, dynamics/__init__.py:147-149), reward = change of -|altitude -
   takeoff_target_altitude|, no bounds / angle limit / landing logic: only the step limit ends an episode.
   Construct it with initial_altitude = 0 and initial_random_force = 0 to start LANDED and unperturbed
   as that env does (the Python shell does). */
enum { COPTER_LANDER3D = 0, COPTER_LANDER2D = 1, COPTER_LANDER1D = 2,
       COPTER_HOVER3D = 3, COPTER_HOVER2D = 4, COPTER_HOVER1D = 5, COPTER_TAKEOFF = 6, COPTER_NUM_VARIANTS = 7 };

enum { COPTER_E_ARG = -1, COPTER_E_VARIANT = -2, COPTER_E_ALIGN = -3, COPTER_E_RANGE = -4 };

/* bits of CopterBuffers.cause: what ended the episode (several can hold at once).  LANDED = the
   stale status was LANDED (envs/lander.py:64-66), BONUS = inside the target radius (:69-72), OOB /
   ANGLE = envs/task.py:111,116, CRASHED = :121, TIMEOUT = the env's own step limit (:128), which is
   what gymnasium's TimeLimit(max_episode_steps=1000) reports as `truncated`. */
enum { COPTER_CAUSE_LANDED = 1, COPTER_CAUSE_BONUS = 2, COPTER_CAUSE_OOB = 4, COPTER_CAUSE_ANGLE = 8,
       COPTER_CAUSE_CRASHED = 16, COPTER_CAUSE_TIMEOUT = 32 };

/* flags: COPTER_F_AUTO_RESET for copter_step_* / copter_rollout_* / copter_policy_rollout_f32 /
   copter_step_host_*; COPTER_F_KEEP_EPISODE for copter_reset_* */
enum { COPTER_F_AUTO_RESET = 1, COPTER_F_KEEP_EPISODE = 2 };

/* episode statistics: double[COPTER_STATS_SLOTS][COPTER_STATS_LEN], accumulated with atomics and never
   cleared by the library.  Each WARP adds to slot (global warp index % COPTER_STATS_SLOTS) so that the
   atomics of concurrent warps land on different 128-byte lines; the statistic is the sum over the slots. */
#define COPTER_STATS_SLOTS 64
enum { COPTER_STAT_EPISODES = 0, COPTER_STAT_RETURN_SUM = 1, COPTER_STAT_LENGTH_SUM = 2,
       COPTER_STAT_LANDED = 3, COPTER_STAT_BONUS = 4, COPTER_STAT_CRASHED = 5, COPTER_STAT_OOB = 6,
       COPTER_STAT_ANGLE = 7, COPTER_STAT_TIMEOUT = 8, COPTER_STAT_ENV_STEPS = 9, COPTER_STATS_LEN = 16 };

#define COPTER_META_STATUS(m)  ((m) & 3u)
#define COPTER_META_STEPS(m)   (((m) >> 2) & 2047u)
#define COPTER_META_EPISODE(m) ((m) >> 13)
#define COPTER_MAX_STEPS_LIMIT 2046                 /* compact meta word (11-bit steps counter) */
#define COPTER_MAX_STEPS_LIMIT_WIDE 0x3FFFFFFE      /* with CopterBuffers.meta_hi (30-bit steps counter) */

typedef struct CopterParams {
    /* vehicle (dji_phantom.py:9-26) */
    double B, D, M, L, Ix, Iy, Iz, Jr, maxrpm;
    /* dynamics/__init__.py:71-76 */
    double landing_vel_x, landing_vel_y, landing_angle, G;
    /* envs/task.py:25,32-38 */
    double fps, initial_random_force, out_of_bounds_penalty, max_angle_deg, bounds, initial_altitude;
    /* envs/lander.py:17-23 */
    double target_radius, yaw_penalty_factor, xyz_penalty_factor, dz_max, dz_penalty, inside_radius_bonus;
    /* alternate vehicle/world model of attic/mars/dynamics/__init__.py (see dynamics_model) */
    double rho, lift_coefficient;
    /* attic/gym_copter/envs/takeoff.py:20 (COPTER_TAKEOFF only) */
    double takeoff_target_altitude;
    int32_t max_steps;
    int32_t dynamics_model;     /* bit set of COPTER_MODEL_*; 0 = the live gym_copter/dynamics model */
} CopterParams;

/* dynamics_model bits.  The live model (0) is Dynamics.setMotors of gym_copter/dynamics/__init__.py:
   thrust U1 = B sum(w^2), U2/U3 = L B (...), gyroscopic term Omega = 0 (:135).  The older
   attic/mars/dynamics/__init__.py:135-164,249-290 differs in two ways that can be switched on
   separately:
     COPTER_MODEL_LIFT  rotor lift 0.5 rho S C_L (w L/2)^2 with S = 0.05 L 4 instead of B w^2, and
                        roll/pitch torques U2/U3 = lift differences WITHOUT the arm length (:146-158);
     COPTER_MODEL_GYRO  live rotor gyroscopic coupling: Omega = (w0+w1)-(w2+w3) (:143) entering
                        phi'' as -Jr/Ix theta' Omega and theta'' as -Jr/Iy phi' Omega (:269-283).
   With G = 3.721 and rho = 0.017 this is the Mars world of attic/mars/dynamics/ingenuity.py:69-71. */
enum { COPTER_MODEL_LIFT = 1, COPTER_MODEL_GYRO = 2 };

int copter_abi_version(void);
void copter_default_params(CopterParams* p);
int copter_obs_size(int variant);      /* O, or COPTER_E_VARIANT */
int copter_action_size(int variant);   /* A, or COPTER_E_VARIANT */

/* Buffers of one shard of envs; all device pointers. Nullable members are marked. */
typedef struct CopterBuffers {
    void*       state;       /* 12/V vectors per env, addressed as in "Memory layout" */
    uint32_t*   meta;        /* [n] */
    const void* action;      /* T[n][A]            (unused by reset) */
    float*      obs;         /* [n][O]             nullable: skip the observation write */
    void*       reward;      /* T[n]               (unused by reset) */
    uint8_t*    done;        /* [n]                (unused by reset) */
    const void* init_force;  /* T[n][3] nullable: injected reset force (N) used instead of the Philox draw */
    void*       ep_return;   /* T[n]   nullable: running episode return, feeds COPTER_STAT_RETURN_SUM */
    double*     stats;       /* [COPTER_STATS_SLOTS][COPTER_STATS_LEN] nullable */
    float*      final_obs;   /* [n][O] nullable: observation of the terminal state of envs that finished */
    uint8_t*    cause;       /* [n] nullable (step only): why the env finished in this launch, bit set of
                                COPTER_CAUSE_*; 0 when it did not finish */
    int64_t     state_stride;/* vectors between the state planes; 0 means n. Lets a call step a sub-range
                                [lo, lo+n) of a larger shard: pass state + lo vectors, stride = shard size */
    uint32_t*   meta_hi;     /* [n] nullable: wide counters (see "Memory layout"): 32-bit episode index */
    int64_t     state_env_stride; /* vectors between consecutive envs; 0 means 1 (planes).  12/V with
                                state_stride 1 is the row layout.  Layouts whose envs overlap are COPTER_E_RANGE */
} CopterBuffers;

/*
 * Reset every env of the shard: default pose, status, steps = 1, obs of the initial state.
 * The episode index becomes 0 -- or, with COPTER_F_KEEP_EPISODE, the env's previous index + 1, so that
 * a caller's reset() per episode (the reference's loop, lander.py:29) draws a NEW reset force each
 * time, as the reference's np.random.uniform does (envs/task.py:175-184,199-202).
 * The reset force is not stored: it is (re)generated on the first step of
 * an episode from Philox4x32-10 with counter (env_lo, env_hi, episode, 0), key = seed,
 * env = env_offset + i, unless init_force is given to copter_step_*.
 */
int copter_reset_f32(const CopterParams* p, const CopterBuffers* b, int64_t n, int variant, int flags, void* stream);
int copter_reset_f64(const CopterParams* p, const CopterBuffers* b, int64_t n, int variant, int flags, void* stream);

/*
 * One launch = k_substeps reference steps for each of the n envs under one action (rewards
 * summed; an env that finishes idles for the rest of the launch).  With COPTER_F_AUTO_RESET
 * a finished env is replaced in the same launch by a fresh reset state and `obs` holds that
 * state's observation; without it the env keeps stepping past `done` like the reference.
 */
int copter_step_f32(const CopterParams* p, const CopterBuffers* b, int64_t n, int64_t env_offset,
                    uint64_t seed, int k_substeps, int variant, int flags, void* stream);
int copter_step_f64(const CopterParams* p, const CopterBuffers* b, int64_t n, int64_t env_offset,
                    uint64_t seed, int k_substeps, int variant, int flags, void* stream);

/*
 * Multi-step rollout with an on-device action source: n_steps reference steps per env in ONE
 * launch with the state in registers, the motor commands generated on the device instead of
 * read from HBM.  Step t of the launch uses the command vector
 *     action_j = offset + scale * xi_j,   xi = 1 (CONST) | N(0,1) (RANDN) | U(-1,1) (UNIFORM),
 * xi drawn from Philox4x32-10 with counter (env_lo, env_hi, first_step + t, 1), key = seed,
 * so a rollout is reproducible and independent of how it is cut into launches.  CONST with
 * offset 1.625e-2 is the reference's heuristic, RANDN with scale 1.625e-2 its `--random`
 * stream (lander.py:21,42).  Equivalent step for step to n_steps calls of copter_step_* with
 * k_substeps = 1 on the same commands (finished envs reset and continue; nothing idles).
 * b->action is unused; b->reward / b->done (nullable here) receive the per-env reward SUM and
 * "any episode finished" flag of the launch, b->obs the observation after the last step.
 * Optional per-step outputs: reward_tn T[n_steps][n], done_tn uint8[n_steps][n] (GAE-ready
 * layout), action_tn T[n_steps][n][A] (the commands used, before clipping), and the episode
 * endings a learner needs to tell a termination from a truncation:
 *   cause_tn uint8[n_steps][n]       the COPTER_CAUSE_* bits of the episode env i ended on step t,
 *                                    else 0; written for every env on every step, so
 *                                    done_tn[t][i] == (cause_tn[t][i] != 0)
 *   final_obs_tn float[n_steps][n][O] the observation of that terminal state (with auto-reset,
 *                                    obs of step t + 1 already belongs to the next episode);
 *                                    written only where cause_tn[t][i] != 0, other rows untouched
 * Per step these are exactly the bytes copter_step_* (k_substeps = 1) writes into b->cause and
 * b->final_obs, which the rollout calls leave unused.
 */
enum { COPTER_SRC_CONST = 0, COPTER_SRC_RANDN = 1, COPTER_SRC_UNIFORM = 2, COPTER_SRC_PID = 3, COPTER_SRC_PID_HOVER = 4 };
typedef struct CopterActionSource { int32_t kind; int32_t reserved; double scale; double offset; } CopterActionSource;

/*
 * COPTER_SRC_PID: the reference's PID landing heuristic evaluated on the device -- attic/mars/
 * lander3d.py:64-87 (roll/pitch rate PIDs + position-hold PIDs + descent PD, quad-X mixer
 * [t-r-p, t+r+p, t+r-p, t-r+p]) over attic/mars/pidcontrollers/__init__.py:12-146 -- fed, like
 * the reference's caller loop (attic/mars/task.py:134-160), with the float32 observation of the
 * previous step; action_j = offset + scale * mixer_j.  On the 2-D / 1-D variants the same source
 * is the reference's planar demo (attic/heuristic/lander2d.py:14-24: [d - p, d + p] with d the
 * descent demand and p the position-hold demand on (y, dy); lander1d.py:14-20: d alone -- no
 * (t+1)/2 there), using the same memory slots.  `controller`
 * T[n][16] holds the four controllers' memories (errorI, lastError, deltaError1, deltaError2 for
 * phi-rate, theta-rate, x_poshold, y_poshold); it persists across episodes exactly as the
 * reference's controller objects do (they live in the env, not in an episode); zero it to start.
 * `gains` NULL selects the reference's constants (copter_default_pid_gains).
 *
 * COPTER_SRC_PID_HOVER: the hover demo's heuristic -- attic/mars/hover3d.py:65-92 (controller set
 * :33-38 plus the altitude-hold controller of attic/mars/hover.py:23, pidcontrollers/__init__.py:
 * 70-99): the same roll/pitch loops, a yaw-rate PID on -dpsi and the altitude-hold set-point
 * controller on (-z, -dz), mixer [t-r-p-y, t+r+p-y, t+r-p+y, t-r+p+y] with t = (hover+1)/2.  It
 * reads the yaw rate, so among the four-motor variants it needs the 12-component observation
 * (COPTER_HOVER3D); on the 2-D / 1-D variants it is attic/heuristic/hover2d.py:17-31
 * ([h - r, h + r], h = altitude-hold demand, r = roll-rate PID + position hold on (y, dy)) and
 * hover1d.py:14-20 (h alone).  `controller`
 * is T[n][24] here: the four memories above, then yaw-rate and altitude-hold.  With
 * scale = 2 x the hover command (0.03312, so that t = 1/2 hovers) the reference's own gains
 * hold the live vehicle at 5 m for whole 1000-step episodes.
 */
typedef struct CopterPidGains {
    double rate_kp, rate_ki, rate_kd, rate_windup, rate_big;      /* AngularVelocityPidController */
    double pos_kp, pos_ki, pos_kd, pos_windup, pos_target;        /* PositionHoldPidController */
    double descent_kp, descent_kd;                                /* DescentPidController */
    double alt_kp, alt_ki, alt_kd, alt_windup, alt_target;        /* AltitudeHoldPidController (COPTER_SRC_PID_HOVER) */
} CopterPidGains;
void copter_default_pid_gains(CopterPidGains* g);

int copter_rollout_f32(const CopterParams* p, const CopterBuffers* b, const CopterActionSource* src,
                       int64_t n, int64_t env_offset, uint64_t seed, int64_t first_step, int n_steps,
                       int variant, int flags, float* reward_tn, uint8_t* done_tn, float* action_tn,
                       const CopterPidGains* gains_or_null, float* controller_or_null,
                       uint8_t* cause_tn, float* final_obs_tn, void* stream);
int copter_rollout_f64(const CopterParams* p, const CopterBuffers* b, const CopterActionSource* src,
                       int64_t n, int64_t env_offset, uint64_t seed, int64_t first_step, int n_steps,
                       int variant, int flags, double* reward_tn, uint8_t* done_tn, double* action_tn,
                       const CopterPidGains* gains_or_null, double* controller_or_null,
                       uint8_t* cause_tn, float* final_obs_tn, void* stream);

/*
 * Batched Dynamics.setMotors: state T[12/V][n][V], status uint8[n], ticks int32[n],
 * perturb T[n][6] (ACCELERATIONS, i.e. force/M as stored by Dynamics.perturb; consumed and
 * zeroed exactly when the reference does), motors T[n][4].
 */
int copter_dynamics_f32(const CopterParams* p, void* state, uint8_t* status, int32_t* ticks,
                        void* perturb, const void* motors, int64_t n, void* stream);
int copter_dynamics_f64(const CopterParams* p, void* state, uint8_t* status, int32_t* ticks,
                        void* perturb, const void* motors, int64_t n, void* stream);

/* Reset-force stream exposed for tests and host-side mirrors: out T[n][3]. */
int copter_reset_force_f32(const CopterParams* p, float* out, const uint32_t* episode_or_null,
                           int64_t n, int64_t env_offset, uint64_t seed, void* stream);
int copter_reset_force_f64(const CopterParams* p, double* out, const uint32_t* episode_or_null,
                           int64_t n, int64_t env_offset, uint64_t seed, void* stream);

/*
 * The policy network of the rollout loop the reference's consumers run on the host -- obs -> net
 * -> clip -> env.step (attic/drl/3dtest.py:36-61) -- as one kernel: the tanh MLP
 * O -> 64 -> 64 -> A of BASELINE.json configs[4], reading the env's fp32 state in place
 * (observation = state components first..first+O-1 of the variant) and writing the action rows
 * copter_step_f32 consumes:  action = out_offset + out_scale * tanh(W3 tanh(W2 tanh(W1 obs + b1) + b2) + b3).
 * Weights use the torch.nn.Linear layouts W[out][in] (fp32, device memory); they and the
 * activations are rounded to 16 bits for the tensor-core MMAs (fp32 accumulation): bf16 everywhere in the
 * warp-MMA kernels; in the tcgen05 kernels bf16 for the observation and layer 1's weights, fp16 for the
 * hidden activations (values in [-1, 1]) and the weights of layers 2 and 3.  hidden must be 64.
 * Two implementations of the same network exist, selectable per call through the environment (tests and
 * A/B runs; the defaults are the measured-faster ones): COPTER_B200_POLICY_TC=1 (default) evaluates it with
 * tcgen05.mma and accumulators in tensor memory, =0 with warp-level mma.sync; they differ in rounding
 * (bias carried as bf16 hi + lo, a quarter of the hidden tanh as FMA-pipe polynomials in the former), both
 * within 2e-2 of the fp32 network.  COPTER_B200_POLICY_ROLLOUT_TC=1 (default) / 0 makes the same choice
 * for copter_policy_rollout_f32 below; each fused kernel is bit-identical to the standalone kernel of
 * its own kind followed by copter_step_f32.
 */
int copter_policy_mlp_f32(const void* state, int64_t state_stride, int64_t n, int variant, int hidden,
                          const float* w1, const float* b1, const float* w2, const float* b2,
                          const float* w3, const float* b3, float out_scale, float out_offset,
                          float* action, void* stream);
/* The same on any state layout: state_env_stride vectors between consecutive envs (0 means 1, which is
   copter_policy_mlp_f32); the row layout of "Memory layout" is state_stride 1, state_env_stride 3. */
int copter_policy_mlp_strided_f32(const void* state, int64_t state_stride, int64_t state_env_stride, int64_t n,
                                  int variant, int hidden, const float* w1, const float* b1, const float* w2,
                                  const float* b2, const float* w3, const float* b3, float out_scale,
                                  float out_offset, float* action, void* stream);

/*
 * Policy-in-the-loop rollout in ONE launch: for n_steps steps, action_t = policy(obs_t) with the
 * MLP of copter_policy_mlp_f32 evaluated from the env state held in registers, then one
 * reference step (k_substeps = 1) under that action -- the whole caller loop of
 * attic/drl/3dtest.py:36-61 (obs -> net -> clip -> env.step) for T steps without the state,
 * the observation or the action ever passing through HBM.  Step for step identical to
 * copter_policy_mlp_f32 followed by copter_step_f32.  b->action is unused; b->reward / b->done
 * (nullable) receive the per-env reward sum and "any episode finished" flag of the launch,
 * b->obs (nullable) the observation after the last step.  Optional per-step outputs (nullable):
 * reward_tn float[n_steps][n], done_tn uint8[n_steps][n], action_tn float[n_steps][n][A] (the
 * commands before the env's clip), obs_tn float[n_steps][n][O] (the observation the policy
 * acted on at step t), cause_tn uint8[n_steps][n] and final_obs_tn float[n_steps][n][O] (the
 * episode endings and terminal observations, as for copter_rollout_*).
 * Exploration (what an on-policy learner such as PPO rolls out): with policy->action_std set
 * (A floats, device memory) the command is drawn around the network's output,
 *     action_j = out_offset + out_scale * tanh(.)_j + action_std[j] * xi_j,   xi ~ N(0,1),
 * xi from Philox4x32-10 with counter (env_lo, env_hi, first_step + t, 2) (Box-Muller as in
 * COPTER_SRC_RANDN; stream tag 2), key = seed: reproducible, and independent of how the rollout
 * is cut into launches when the caller advances first_step by n_steps.  action_tn then holds the
 * sampled commands the learner needs for its log-probabilities.
 */
typedef struct CopterMlpPolicy {
    const float *w1, *b1, *w2, *b2, *w3, *b3;   /* torch.nn.Linear layouts W[out][in], b[out]; fp32 device memory */
    int32_t hidden;                             /* must be 64 */
    float out_scale, out_offset;                /* action = out_offset + out_scale * tanh(.) */
    const float* action_std;                    /* nullable: [A] standard deviations of the Gaussian exploration noise */
} CopterMlpPolicy;
int copter_policy_rollout_f32(const CopterParams* p, const CopterBuffers* b, const CopterMlpPolicy* policy,
                              int64_t n, int64_t env_offset, uint64_t seed, int64_t first_step, int n_steps,
                              int variant, int flags, float* reward_tn, uint8_t* done_tn, float* action_tn,
                              float* obs_tn, uint8_t* cause_tn, float* final_obs_tn, void* stream);

/*
 * Generalised advantage estimation over the [T][n] rows of a rollout, one pass on the device.
 * For each env i and t = n_steps-1 .. 0 (fp32, evaluated in this order):
 *     next  = t == T-1 ? last_value[i] : value[t+1][i]
 *     c     = cause[t][i];  trunc = (c & COPTER_CAUSE_TIMEOUT) != 0
 *     boot  = c == 0 ? next : (trunc && final_value ? final_value[t][i] : 0)
 *     delta = reward[t][i] + gamma * boot - value[t][i]
 *     A     = delta + gamma * lam * (c == 0 ? A_next : 0)            (A_next = 0 at t = T-1)
 *     adv[t][i] = A;  ret[t][i] = A + value[t][i]
 * cause_tn is the cause_tn row block of copter_rollout_* / copter_policy_rollout_f32.  A step
 * that ended by the env's own step limit (COPTER_CAUSE_TIMEOUT, gymnasium's `truncated`) is
 * bootstrapped from final_value, the caller's value of the terminal observation (final_obs_tn);
 * with final_value NULL every ending, truncations included, is treated as a termination (boot 0).
 * value_tn float[n_steps][n], last_value float[n] (value of the observation after the last
 * step), final_value float[n_steps][n] (read only where a truncation is), adv_tn float[n_steps][n],
 * ret_tn float[n_steps][n] (nullable).  COPTER_E_ARG for a NULL required pointer, n < 0 or
 * n_steps < 1 (checked before anything touches the device).
 */
int copter_gae_f32(const float* reward_tn, const float* value_tn, const float* last_value,
                   const uint8_t* cause_tn, const float* final_value_tn_or_null,
                   int64_t n, int n_steps, float gamma, float lam,
                   float* adv_tn, float* ret_tn_or_null, void* stream);

/*
 * The critic of an on-policy learner, Linear(O,64) -> tanh -> Linear(64,64) -> tanh -> Linear(64,1)
 * (linear output), on m fp32 observation rows: row r is rows[r * row_stride + 0 .. O-1]
 * (row_stride >= O floats, O = copter_obs_size(variant); 4-byte alignment is enough), so the
 * packed obs_tn / final_obs_tn rows of copter_policy_rollout_f32 (stride O) and the fp32 env's
 * observation inside its state rows (stride 12) are both read in place.  w1 [64][O], b1 [64],
 * w2 [64][64], b2 [64], w3 [1][64], b3 [1] (torch.nn.Linear layouts, fp32 device memory, read
 * on every call).  The tcgen05 kernel of copter_policy_mlp_f32 with a value head: bf16 rows and
 * layer-1 weights, fp16 hidden activations and layer-2 / -3 weights, biases as 16-bit hi + lo,
 * fp32 accumulation; value[r] = layer 3's accumulator.
 * select_or_null (uint8[m]): when given, only rows with select[r] & select_mask are evaluated and
 * every other value[r] is left untouched (e.g. final_obs_tn at cause_tn & COPTER_CAUSE_TIMEOUT,
 * the only rows copter_gae_f32 reads).
 * COPTER_E_ARG for a NULL required pointer or m < 0; COPTER_E_VARIANT; COPTER_E_RANGE for
 * row_stride < O or hidden != 64; COPTER_E_ALIGN for a float pointer that is not 4-byte aligned.
 * m == 0 is a no-op.
 */
int copter_value_mlp_f32(const float* rows, int64_t row_stride, int64_t m, int variant, int hidden,
                         const float* w1, const float* b1, const float* w2, const float* b2,
                         const float* w3, const float* b3,
                         const uint8_t* select_or_null, uint32_t select_mask,
                         float* value, void* stream);

/*
 * Log-probability of the actions copter_policy_rollout_f32 sampled with exploration noise
 * (policy->action_std), for the same seed, env_offset, n, first_step and variant:
 *     logp_tn[t][i] = -1/2 sum_j xi_j^2 - sum_j log action_std[j] - (A/2) log(2 pi),   j < A
 * with xi the rollout's own N(0,1) draws of (seed, env_offset + i, first_step + t): exactly the
 * density the action was drawn from, whichever rollout kernel ran and however the rollout was
 * sharded or cut into horizons.  action_std float[A] (device, read in place), logp_tn
 * float[n_steps][n].  COPTER_E_ARG for a NULL pointer, n < 0 or n_steps < 1; COPTER_E_VARIANT;
 * COPTER_E_RANGE for env_offset < 0 or first_step < 0; COPTER_E_ALIGN for a pointer that is not
 * 4-byte aligned.  n == 0 is a no-op.
 */
int copter_policy_logp_f32(uint64_t seed, int64_t env_offset, int64_t n, int64_t first_step, int n_steps,
                           int variant, const float* action_std, float* logp_tn, void* stream);

/*
 * The same step for callers that hold HOST arrays (the reference's callers pass numpy
 * arrays, lander.py:42-44).  The shard is cut into chunks of `chunk_envs`; for each chunk
 * the action rows are copied host->device, the step kernel runs on that sub-range, and
 * obs/reward/done are copied device->host, round-robin over the pipeline's streams so the
 * two PCIe directions and the kernel overlap.  `dev` are the device buffers of the whole
 * shard (dev->action is the device staging area for the actions).  Host arrays should be
 * page-locked for the copies to be asynchronous.  Work is ordered after `stream`; the call
 * returns when all chunks have landed in the host arrays.  h_cause / h_final_obs (nullable)
 * receive dev->cause / dev->final_obs when those device buffers are given.
 * Shards of at most 65 536 envs (COPTER_B200_DIRECT_MAX_ENVS in the environment overrides the limit, 0 switches
 * the path off) whose host arrays are all page-locked and mapped
 * (cudaHostAlloc / cudaHostRegister under unified addressing) take a direct path: ONE launch whose kernel
 * reads the commands from and writes obs / reward / done / cause / final_obs to the host arrays themselves,
 * then one stream synchronisation; the device-side action / obs / reward / done buffers of `dev` are not
 * touched on that path.
 */
int copter_pipeline_create(int n_streams, void** out_pipeline);      /* 1..8 streams */
int copter_pipeline_destroy(void* pipeline);
int copter_step_host_f32(void* pipeline, const CopterParams* p, const CopterBuffers* dev,
                         const float* h_action, float* h_obs_or_null, float* h_reward, uint8_t* h_done,
                         uint8_t* h_cause_or_null, float* h_final_obs_or_null, int64_t n, int64_t env_offset, uint64_t seed, int k_substeps, int variant,
                         int flags, int64_t chunk_envs, void* stream);
int copter_step_host_f64(void* pipeline, const CopterParams* p, const CopterBuffers* dev,
                         const double* h_action, float* h_obs_or_null, double* h_reward, uint8_t* h_done,
                         uint8_t* h_cause_or_null, float* h_final_obs_or_null, int64_t n, int64_t env_offset, uint64_t seed, int k_substeps, int variant,
                         int flags, int64_t chunk_envs, void* stream);

#ifdef __cplusplus
}
#endif
#endif
