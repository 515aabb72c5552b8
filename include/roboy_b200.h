/*
 * roboy_b200.h -- C-ABI of the B200-native batched MSJ environment step.
 *
 * This is the drop-in boundary for gym-roboy's environment hot path.  Every entry point names
 * the reference interface it replaces (paths relative to gym_roboy/ in Roboy/gym-roboy).
 * The reference is pure Python, so the binding a maintainer adds is a ctypes stub
 * (INTEGRATION.md shows it); gym_roboy_b200/_native.py is that stub for this repo's host side.
 *
 * Conventions
 *   - plain C types only; `stream` is a cudaStream_t passed as void* (NULL = legacy default).
 *   - pointers suffixed _dev are device pointers (e.g. torch tensor .data_ptr()); suffixed
 *     _host are host pointers.  Device entry points are asynchronous on `stream`.
 *   - every call returns 0 on success, a negative ROBOY_E_* code on failure;
 *     roboy_last_error() returns a thread-local message for the last failure.
 *   - the reference reports contract violations by raising AssertionError; a batched device
 *     path cannot raise per env, so violations are recorded in an error word + the first
 *     offending global env id (roboy_errors) and counted in the statistics.
 *   - there is no CPU fallback: without a CUDA device roboy_create fails with ROBOY_E_CUDA.
 *
 * Memory layout in HBM (structure of arrays, n = n_envs of this shard; J = dim_joint = 3 and A = dim_action = 8 for MSJ):
 *   goal        float32 [J][n]   desired joint angles            (RoboyEnv._goal_state)
 *   step_flags  uint32  [n]      bits 0..23 step_num, bit 24 HELD_ZERO64, bit 25 HELD_INFEASIBLE
 *   held        float32 [2J][n]  StubSimulationClient._state: q_0..q_{J-1}, qd_0..qd_{J-1} (cold; read only
 *                                on the hold branch when HELD_ZERO64 is clear)
 *   obs         float32 [n][3J]  row-major [q, qd, goal], what the policy consumes (roboy_env.py:75-80)
 *   actions     float32 [n][A]   caller's, in [-1, 1]
 *   reward      float32 [n]
 *   done        uint8   [n]
 *   stats       float64 [8]      ROBOY_STAT_*
 */
#ifndef ROBOY_B200_H_
#define ROBOY_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ROBOY_B200_ABI_VERSION 2

#define ROBOY_DIM_JOINT 3  /* msj_robot.py:8  (the MSJ robot; other robots: roboy_cfg.dim_joint) */
#define ROBOY_DIM_ACTION 8 /* msj_robot.py:12 */
#define ROBOY_DIM_OBS 9    /* roboy_env.py:32-36: 3 * dim_joint */

/* Robots other than MSJ (roboy_robot.py:21-33; README.md:6-7 "MSJ platform, Upper Body, etc."): up to 15 joints and
 * 64 tendons, one bound per component.  15, because numpy's norm changes its summation order from 16 float64
 * elements on (OpenBLAS kernels, CPU dependent): beyond that, bit-exact parity with the reference is not defined. */
#define ROBOY_MAX_JOINT 15
#define ROBOY_JOINT_PAD 16
#define ROBOY_MAX_ACTION 64

/* error codes */
#define ROBOY_OK 0
#define ROBOY_E_ARG (-1)   /* bad argument (NULL handle, n == 0, misaligned pointer ...) */
#define ROBOY_E_CUDA (-2)  /* CUDA runtime failure, or no CUDA device: there is no CPU path */
#define ROBOY_E_ALLOC (-3)

/* step_flags bits */
#define ROBOY_STEP_MASK 0x00ffffffu
#define ROBOY_F_HELD_ZERO64 (1u << 24)     /* held state is the float64 zero state of roboy_robot.py:41-45 */
#define ROBOY_F_HELD_INFEASIBLE (1u << 25) /* held state has is_feasible == False */

/* bits of the device error word (the reference's AssertionErrors) */
#define ROBOY_ERR_ACTION 1u       /* roboy_env.py:52   action outside [-1,1]^8 or NaN */
#define ROBOY_ERR_REWARD_RANGE 2u /* roboy_env.py:109  reward outside reward_range */
#define ROBOY_ERR_GOAL_BOUNDS 4u  /* roboy_robot.py:76 injected goal outside the angle space */
#define ROBOY_ERR_STATE_BOUNDS 8u /* roboy_robot.py:76 joint angles handed in by an external simulator outside the angle
                                   * space or NaN (roboy_step_external / roboy_reset_external): where the reference's client
                                   * builds the state with robot.new_state(), ros_simulation_client.py:40-46 */

/* indices into the statistics vector */
enum {
    ROBOY_STAT_STEPS = 0,       /* env-steps executed */
    ROBOY_STAT_EPISODES = 1,    /* done flags raised */
    ROBOY_STAT_SUCCESSES = 2,   /* ... because _did_reach_goal (roboy_env.py:125-134) */
    ROBOY_STAT_TIMEOUTS = 3,    /* ... because step_num > 400 only (roboy_env.py:72-73) */
    ROBOY_STAT_SUM_REWARD = 4,  /* sum of all step rewards */
    ROBOY_STAT_SUM_EPLEN = 5,   /* sum of step_num - 1 over the raised done flags (with auto_reset off, an env left done
                                 * counts again on each further step) */
    ROBOY_STAT_HOLDS = 6,       /* steps that took the Stub's hold branch (simulation_client.py:38-39) */
    ROBOY_STAT_VIOLATIONS = 7,  /* env-steps with a non-zero error word */
    ROBOY_STAT_COUNT = 8
};

/* buffers owned by a handle, for roboy_buffer / roboy_export_dlpack */
enum {
    ROBOY_BUF_GOAL = 0, ROBOY_BUF_STEP_FLAGS = 1, ROBOY_BUF_HELD = 2, ROBOY_BUF_OBS = 3,
    ROBOY_BUF_REWARD = 4, ROBOY_BUF_DONE = 5, ROBOY_BUF_STATS = 6, ROBOY_BUF_TERMINAL_OBS = 7,
    ROBOY_BUF_DONE_BITS = 8, /* uint32 [ceil(n/32)], after roboy_enable_done_index */
    ROBOY_BUF_COUNT = 9
};

/* Constructor arguments of RoboyEnv (roboy_env.py:12-14) + the robot's bounds
 * (MsjRobot, msj_robot.py:8-16) + sharding.  Field order is ABI. */
typedef struct roboy_cfg {
    uint64_t n_envs;       /* envs in this shard (one shard per GPU) */
    uint64_t env_id_base;  /* global id of local env 0; Philox counters use the global id */
    uint64_t seed;         /* Philox key (RoboyEnv(seed=...), roboy_env.py:12,15) */
    float angle_low, angle_high; /* msj_robot.py:9 */
    float vel_low, vel_high;     /* msj_robot.py:10 */
    float act_low, act_high;     /* msj_robot.py:16 */
    int32_t max_episode_len;     /* roboy_env.py:28 */
    int32_t joint_vel_penalty;   /* roboy_env.py:13 */
    int32_t bonus_for_goal;      /* roboy_env.py:14 is_agent_getting_bonus_for_reaching_goal */
    int32_t auto_reset;          /* 1: reset-on-done inside the step (vec-env worker semantics) */
    float penalty_boundary;      /* roboy_env.py:26 */
    float bonus_goal;            /* roboy_env.py:27 */
    double reward_lo, reward_hi; /* roboy_env.py:30,109; +-inf disables the check */
    /* Other robots.  dim_joint / dim_action: RoboyRobot.get_joint_angles_space().shape[0] / get_action_space().shape[0]
     * (0 = MSJ's 3 / 8).  per_component_bounds != 0: the arrays below hold one low / high per joint or tendon
     * (spaces.Box built from arrays) and the six scalars above are ignored; == 0: the scalars apply to every component.
     * A robot with MSJ's dims and uniform bounds runs the tuned MSJ kernels, any other the generic ones (same results). */
    int32_t dim_joint, dim_action;
    int32_t per_component_bounds;
    int32_t reserved;
    float angle_low_v[ROBOY_JOINT_PAD], angle_high_v[ROBOY_JOINT_PAD];
    float vel_low_v[ROBOY_JOINT_PAD], vel_high_v[ROBOY_JOINT_PAD];
    float act_low_v[ROBOY_MAX_ACTION], act_high_v[ROBOY_MAX_ACTION];
} roboy_cfg;

typedef struct roboy_env roboy_env; /* opaque */

int roboy_abi_version(void);
const char *roboy_last_error(void);

/* Fill `cfg` with the MSJ robot constants (msj_robot.py:8-16), RoboyEnv's defaults
 * (roboy_env.py:12-14,26-28), auto_reset = 1 and an unbounded reward range. */
int roboy_cfg_msj(roboy_cfg *cfg);

/* Host-only helper (no GPU needed): the closed float32 interval [lo, hi] of action components
 * for which the Stub holds its state -- the pre-image of numpy's allclose(rescaled, 0)
 * (simulation_client.py:38) under the float32 rescale of roboy_env.py:157-158.  For MSJ this is
 * [-2^-24, 2^-25].  lo > hi means the interval is empty.  The step kernel compares against it.  The interval is taken over
 * every finite float32, not only [-1, 1]: a one-sided tendon range [0, hi] holds at a = -1 and just below it, and an
 * action outside the action space (error word, roboy_env.py:52) still meets the Stub the way numpy would treat it.
 * roboy_hold_interval: tendon 0;  roboy_hold_intervals: all dim_action tendons (lo, hi: float[dim_action]). */
int roboy_hold_interval(const roboy_cfg *cfg, float *lo, float *hi);
int roboy_hold_intervals(const roboy_cfg *cfg, float *lo, float *hi);

/* RoboyEnv.__init__ over StubSimulationClient.__init__ (roboy_env.py:12-38,
 * simulation_client.py:29-31) for n_envs envs on CUDA device `device`: allocates the SoA state
 * in HBM and runs the init kernel (held state := random sample, goal := random, step_num := 1). */
int roboy_create(const roboy_cfg *cfg, int device, roboy_env **out);
int roboy_destroy(roboy_env *env);

/* roboy_env.py:30,109 -- (re)set the reward range checked inside the step kernel. */
int roboy_set_reward_range(roboy_env *env, double lo, double hi);

/* RoboyEnv.reset (roboy_env.py:82-87) over Stub.forward_reset_command / read_state
 * (simulation_client.py:42-44,33-34) for every env with mask_dev[i] != 0 (NULL: all envs).
 * Writes obs rows of the reset envs into obs_dev (NULL: the handle's obs buffer). */
int roboy_reset(roboy_env *env, const uint8_t *mask_dev, float *obs_dev, void *stream);

/* RoboyEnv.step (roboy_env.py:51-70) fused with StubSimulationClient.forward_step_command
 * (simulation_client.py:36-40), RoboyRobot.normalize_state (roboy_robot.py:80-95),
 * compute_reward (roboy_env.py:92-112), _did_reach_goal (:125-134), _set_new_goal (:117-123)
 * and, when cfg.auto_reset, the vec-env worker's reset-on-done.  One launch over all envs.
 *   actions_dev float32 [n][8] in [-1,1];  outputs: NULL selects the handle's own buffer. */
int roboy_step(roboy_env *env, const float *actions_dev, float *obs_dev, float *reward_dev,
               uint8_t *done_dev, void *stream);

/* Open-loop variant: T consecutive RoboyEnv.step calls (roboy_env.py:51-70) on PRE-RECORDED actions
 * float32 [T][n][8], writing obs [T][n][9], reward [T][n], done [T][n].  One launch: each env's goal and
 * step counter stay in registers across the T steps (73 algorithmic bytes per env-step instead of
 * 93).  Bit-identical to T roboy_step calls; the call counter advances by T.  Use it to replay
 * recorded action sequences; a closed-loop policy needs roboy_step (or a CUDA graph of them). */
int roboy_step_many(roboy_env *env, uint32_t T, const float *actions_dev, float *obs_dev, float *reward_dev,
                    uint8_t *done_dev, void *stream);

/* The same step through HOST buffers -- the hop train_parallel.py:29 makes through SubprocVecEnv's pipes, once per
 * step for the whole population: chunked H2D(actions) -> kernel -> D2H(obs, reward, done) pipelined over internal
 * streams; returns when the outputs are in host memory.  This is the call a host-side (CPU policy) trainer makes, and
 * what bench.py's e2e number times.  The call is DEVICE-SYNCHRONOUS: it first waits for all work queued on the device
 * (whatever stream a preceding roboy_reset / roboy_set_* / roboy_step was issued on), and on a CUDA error it drains its
 * internal streams before returning, so no copy into the caller's buffers is ever left in flight. */
int roboy_step_host(roboy_env *env, const float *actions_host, float *obs_host, float *reward_host,
                    uint8_t *done_host);

/* Tuning of roboy_step_host's pipeline: envs per stage (multiple of 32; default 524,288), streams (1..8, default 2)
 * and the pattern:
 *   ROBOY_HOST_PATTERN_RING (default)  stage i runs H2D(actions_i) -> kernel_i -> D2H(obs_i, reward_i, done_i) on
 *                                      stream i % n_streams
 *   ROBOY_HOST_PATTERN_SPLIT           one "up" stream carries every H2D and kernel, n_streams - 1 "down" streams the
 *                                      D2H copies behind per-stage events
 * (measured: the ring of two streams is 7 % faster -- roboy_capi.cu).  roboy_set_host_ramp: run the first three stages
 * at 1/8, 1/4 and 1/2 of the stage size so the D2H engine starts sooner (default on). */
int roboy_set_host_pipeline(roboy_env *env, uint64_t stage_envs, int n_streams);
int roboy_set_host_ramp(roboy_env *env, int enable);
/* Unless the caller fixed the pipeline with roboy_set_host_pipeline, the stream count of the ring is tuned by measurement:
 * the second and third roboy_step_host calls of a handle time a ring of two streams and a single stream and the faster
 * one is kept (one GPU on its own PCIe link wants two; eight GPUs saturating the host's memory path want one).
 * roboy_set_host_autotune(env, 1) restores the defaults and re-arms the tuning; roboy_get_host_pipeline reads the
 * configuration in force (any pointer may be NULL). */
int roboy_set_host_autotune(roboy_env *env, int enable);
int roboy_get_host_pipeline(roboy_env *env, uint64_t *stage_envs, int *n_streams, int *pattern);
#define ROBOY_HOST_PATTERN_SPLIT 0
#define ROBOY_HOST_PATTERN_RING 1
int roboy_set_host_pattern(roboy_env *env, int pattern);

/* How roboy_step_host moves the outputs (and inputs):
 *   ROBOY_HOST_STAGED      copy engines both ways (default; any host memory, pinned for full speed)
 *   ROBOY_HOST_MAPPED_OUT  H2D by copy engine; the step kernel stores obs / reward / done straight into the caller's
 *                          page-locked buffers over PCIe (no HBM round trip, no D2H stage)
 *   ROBOY_HOST_MAPPED_ALL  one launch over the shard that also READS the actions from page-locked host memory
 * The mapped modes need buffers from cudaHostAlloc / cudaHostRegister / roboy_host_alloc. */
#define ROBOY_HOST_STAGED 0
#define ROBOY_HOST_MAPPED_OUT 1
#define ROBOY_HOST_MAPPED_ALL 2
int roboy_set_host_mode(roboy_env *env, int mode);

/* Page-locked, device-mapped host memory for the calls above (cudaHostAlloc portable | mapped, optionally
 * write-combined: faster for the GPU to read, slow for the CPU to read -- action buffers only). */
int roboy_host_alloc(uint64_t bytes, int write_combined, void **out_host);
int roboy_host_free(void *host);

/* Measurement only (bench.py's e2e.copy_ceiling): the copies of roboy_step_host WITHOUT the kernel, same buffers, same
 * 32 / 41 byte split per env.  directions: 1 = H2D, 2 = D2H, 3 = both concurrently.  monolithic = 0: the staged
 * pipeline's copy pattern; 1: one copy per array, the two directions on two independent streams.  Env state is not
 * touched.  Returns the wall-clock milliseconds per pass over all n envs, averaged over `iters` passes. */
int roboy_host_copy_probe(roboy_env *env, const float *actions_host, float *obs_host, float *reward_host,
                          uint8_t *done_host, int directions, int monolithic, int iters, double *ms_per_pass);

/* Optional side buffer float32 [n][9] receiving the pre-reset observation of envs that
 * finish an episode (the vec-env `terminal_observation`).  NULL disables. */
int roboy_set_terminal_obs(roboy_env *env, float *terminal_obs_dev);

/* The done list of the LAST roboy_step / roboy_step_host as indices (roboy_env.py:65-68 `if done:` -- which envs
 * finished; north_star: "bit-exact for done/reset masks and indices").  Once enabled, the step kernel also publishes its
 * done mask as bits (one warp ballot per 32 envs; ROBOY_BUF_DONE_BITS), and roboy_done_indices turns them into the
 * ASCENDING list of local env ids on the device: idx_dev int32 [capacity], *count_dev = number of done envs (entries
 * beyond capacity are dropped, the count is not clipped).  terminal_rows_dev (optional, float32 [capacity][9]) receives
 * the pre-reset observation of each listed env, gathered from the terminal-obs side buffer -- the rows a vec-env
 * returns as infos[i]["terminal_observation"].  Asynchronous on `stream`; deterministic. */
int roboy_enable_done_index(roboy_env *env, int enable);
int roboy_done_indices(roboy_env *env, int32_t *idx_dev, uint64_t capacity, uint32_t *count_dev, float *terminal_rows_dev,
                       void *stream);

/* Stand-alone GoalEnv.compute_reward(current_state, goal_state) (roboy_env.py:92-112) and
 * _did_reach_goal (:125-134) over float32 device arrays [k][3]; feasible_dev uint8 [k] or NULL
 * (all feasible); goal_qd_dev NULL = the float64 zero velocities of roboy_env.py:23.
 * reward_dev float64 [k] (the reference returns a python float), reached_dev uint8 [k] or NULL.
 * check_range: 0 = no range check; 1 = apply the handle's reward range (violations go to the error word);
 * 2 (ROBOY_REWARD_RANGE_PROBE) = the two calls of _create_reward_range (roboy_env.py:40-49): no check, and the float32
 * exponentials correctly rounded, so that the bounds the other rewards are checked against (:109) do not fall an ulp of the
 * device's expf inside the range they are meant to enclose. */
#define ROBOY_REWARD_RANGE_PROBE 2
int roboy_compute_reward(roboy_env *env, uint64_t k, const float *q_dev, const float *qd_dev,
                         const uint8_t *feasible_dev, const float *goal_q_dev, const float *goal_qd_dev,
                         double *reward_dev, uint8_t *reached_dev, int check_range, void *stream);

/* State injection (parity tests, RoboyEnv._set_new_goal(goal_joint_angle=...) roboy_env.py:117-123,
 * and tests that poke StubSimulationClient._state / RoboyEnv.step_num).  idx_dev: int64 [k]
 * local env indices; values are [k][3] float32 / [k] uint8 / [k] int32 device arrays. */
int roboy_set_goal(roboy_env *env, uint64_t k, const int64_t *idx_dev, const float *goal_q_dev, void *stream);
int roboy_set_state(roboy_env *env, uint64_t k, const int64_t *idx_dev, const float *q_dev,
                    const float *qd_dev, const uint8_t *feasible_dev, void *stream);
int roboy_set_step_num(roboy_env *env, uint64_t k, const int64_t *idx_dev, const int32_t *step_dev, void *stream);

/* SimulationClient.read_state (simulation_client.py:33-34) for k envs: the held state as
 * float32 [k][3] q, [k][3] qd, uint8 [k] feasible.  feasible byte: bit 0 = is_feasible, bit 1 = the state is the
 * reference's FLOAT64 zero state (roboy_robot.py:41-45 after forward_reset_command) -- a caller that keeps the
 * reference's RoboyEnv on top hands it float64 arrays then, so numpy promotes exactly as it does over the Stub. */
int roboy_read_state(roboy_env *env, uint64_t k, const int64_t *idx_dev, float *q_dev, float *qd_dev,
                     uint8_t *feasible_dev, void *stream);

/* The un-fused plug-in calls of SimulationClient (simulation_client.py:11-23), batched over the
 * shard, for callers that keep the reference's own RoboyEnv on top (INTEGRATION.md):
 *   roboy_sim_step   forward_step_command(action) -- simulation_client.py:36-40.  actions_dev is
 *                    float32 [n][8] in ROBOT units (after roboy_env.py:54-57); advances the call
 *                    counter; writes the returned state (q, qd [n][3], feasible [n] or NULL; same two bits as
 *                    roboy_read_state).
 *   roboy_sim_reset  forward_reset_command()      -- simulation_client.py:42-44, envs with
 *                    mask_dev[i] != 0 (NULL: all); advances the call counter.
 *   roboy_new_goal   get_new_goal_joint_angles()  -- simulation_client.py:46-47; writes [n][3]
 *                    draws to goal_q_dev and does NOT change the env's goal (RoboyEnv._set_new_goal
 *                    does that, via roboy_set_goal).  Repeated calls give fresh draws; the first call after
 *                    roboy_create / roboy_reseed returns the goal the env was constructed with (roboy_env.py:37). */
int roboy_sim_step(roboy_env *env, const float *actions_dev, float *q_dev, float *qd_dev, uint8_t *feasible_dev,
                   void *stream);
int roboy_sim_reset(roboy_env *env, const uint8_t *mask_dev, void *stream);
int roboy_new_goal(roboy_env *env, float *goal_q_dev, void *stream);

/* RoboyEnv constructor flags (roboy_env.py:13-14) and reset-on-done, changeable after create. */
int roboy_set_flags(roboy_env *env, int joint_vel_penalty, int bonus_for_goal, int auto_reset);
/* RoboyEnv.seed (roboy_env.py:114-115): re-key the Philox generator; state is left as is. */
int roboy_set_seed(roboy_env *env, uint64_t seed);
/* RoboyEnv(client, seed=s) (roboy_env.py:12,15 then :37): re-key AND redo the construction draws (held state, first
 * goal, step_num = 1, call counter = 0), so the first episode is reproducible from the env seed.  Synchronises. */
int roboy_reseed(roboy_env *env, uint64_t seed);

/* Zero-copy access to the handle's buffers (ROBOY_BUF_*): raw device pointer + byte size, or
 * a DLPack DLManagedTensor* (consume with PyCapsule "dltensor" -> torch.from_dlpack). */
int roboy_buffer(roboy_env *env, int which, void **dev_ptr, uint64_t *nbytes);
void *roboy_export_dlpack(roboy_env *env, int which);

/* Philox call counter (0 after create, +1 per reset/step call) -- with the state buffers and
 * the seed this is the complete checkpoint of the env shard.  The counter is DEVICE state: every
 * counter-advancing kernel reads it and its last CTA stores the new value, so roboy_step /
 * roboy_reset / roboy_sim_* launches carry no host state and can be captured in a CUDA graph and
 * replayed (each replay advances the counter).  Both calls below synchronise the device. */
int roboy_get_counter(roboy_env *env, uint64_t *t);
int roboy_set_counter(roboy_env *env, uint64_t t);

/* Episode statistics (ROBOY_STAT_*) accumulated on the device by the step kernel.
 * roboy_stats copies them to the host (synchronises `stream`); the device vector itself is
 * ROBOY_BUF_STATS, which is what the multi-GPU NCCL all-reduce operates on. */
int roboy_stats(roboy_env *env, double out_host[ROBOY_STAT_COUNT], void *stream);
int roboy_clear_stats(roboy_env *env, void *stream);   /* statistics and error word */
int roboy_clear_errors(roboy_env *env, void *stream);  /* error word only */
/* Device error word and first offending global env id (UINT64_MAX if none); synchronises. */
int roboy_errors(roboy_env *env, uint32_t *err_flags, uint64_t *first_bad_env, void *stream);

/* External-simulator feed (SURVEY.md 8f row 4).  RoboyEnv.step / reset (roboy_env.py:51-70, :82-87)
 * when the robot states come from an external simulator -- the role RosSimulationClient plays
 * (ros_simulation_client.py:40-60: q, qdot, feasible arrive over the wire) -- instead of the
 * in-process Stub: the caller forwards the actions to its simulator itself and hands the resulting
 * batch [n][3] q, [n][3] qd, [n] feasible (NULL = all feasible) to the same reward / done / goal
 * kernel.  The reference holds wire values as float64 arrays, so its float64 arithmetic applies.
 * No auto-reset: on done the goal is re-drawn (:67-68); the caller resets its simulator and calls
 * roboy_reset_external (mask NULL = all) with the post-reset states. */
int roboy_step_external(roboy_env *env, const float *q_dev, const float *qd_dev, const uint8_t *feasible_dev,
                        float *obs_dev, float *reward_dev, uint8_t *done_dev, void *stream);
int roboy_reset_external(roboy_env *env, const uint8_t *mask_dev, const float *q_dev, const float *qd_dev,
                         float *obs_dev, void *stream);

/* Rollout consumer (SURVEY.md 8f row 1): GAE(lambda) advantages and returns over rollout buffers
 * [T][n] that roboy_step filled in place -- what the PPO2 runner behind train_parallel.py:31-34
 * computes on the host.  done[t] = the episode ended AT step t (no bootstrap across it);
 * last_value [n] = V(observation after the last step).  Runs on the current device, async. */
int roboy_gae(uint64_t T, uint64_t n, const float *reward_dev, const float *value_dev, const uint8_t *done_dev,
              const float *last_value_dev, float gamma, float lam, float *adv_dev, float *ret_dev, void *stream);

/* Closed-loop rollout with the policy INSIDE the kernel (SURVEY.md 8f row 1; BASELINE.json configs[4]):
 * T steps of [MlpPolicy forward -> Gaussian sample -> clip to the action space -> RoboyEnv.step] for every
 * env in ONE launch -- the loop stable-baselines' PPO2 runner drives over a SubprocVecEnv in
 * train_parallel.py:28-35.  The policy is stable-baselines' MlpPolicy shape: separate D-64-64 tanh networks
 * (D = 3J inputs) for the action mean (A outputs) and the value (1 output), state-independent log-std.
 * Runs on every robot: MSJ-shaped handles (3 joints, 8 tendons, uniform bounds) on the tuned MSJ kernel, every
 * other robot (and MSJ under ROBOY_B200_FORCE_GENERIC=1) on the generic one.  Each env's observation, goal and
 * step counter stay on chip for the T steps; per env-step the kernel writes action 4A + logp 4 + value 4 +
 * obs 12J + reward 4 + done 1 = 4A + 12J + 13 bytes (81 for MSJ) and reads nothing.
 * Env outputs are bit-identical to T roboy_step calls on clip(actions, -1, 1).
 *
 * image_dev: the policy packed as float32 [offsets[ROBOY_POLICY_LAYOUT_FLOATS]] of roboy_policy_layout(3J, A),
 * 16-byte aligned (for MSJ that is [ROBOY_POLICY_IMAGE_FLOATS] at the ROBOY_POLICY_OFF_* offsets below).
 * Noise: Philox4x32-10 keyed by noise_seed, counter (global env id, env call counter, stream 4, sub = k / 4),
 * Box-Muller on word pair (k % 4) / 2 of that block, its first or second value by k % 2, for normal k = 0..A-1;
 * independent of how envs are sharded.
 *   obs_dev     float32 [T+1][n][3J] slot 0 = the observation to start from (input), slots 1..T written
 *   actions_dev float32 [T][n][A]    the UN-clipped samples (what PPO2's runner stores; env.step saw the clip)
 *   logp_dev    float32 [T][n]       log-density of the sample;  values_dev float32 [T+1][n] (slot T: bootstrap)
 *   reward_dev  float32 [T][n];  done_dev uint8 [T][n];  noise_dev float32 [T][n][A] or NULL (tests)
 * envs_per_thread: 0 = automatic (MSJ: 1 while all envs fit on the chip at once, else 2; other robots: 1). */
#define ROBOY_POLICY_HIDDEN 64
#define ROBOY_POLICY_OFF_W1 0
#define ROBOY_POLICY_OFF_B1 576
#define ROBOY_POLICY_OFF_W2 640
#define ROBOY_POLICY_OFF_B2 4736
#define ROBOY_POLICY_OFF_W3 4800
#define ROBOY_POLICY_OFF_B3 5312
#define ROBOY_POLICY_NET_FLOATS 5320
#define ROBOY_POLICY_OFF_VF 0
#define ROBOY_POLICY_OFF_PI 5320
#define ROBOY_POLICY_OFF_STD 10640
#define ROBOY_POLICY_OFF_LOGNORM 10648
#define ROBOY_POLICY_IMAGE_FLOATS 10652
/* Layout of the policy image of roboy_policy_rollout for dim_obs = D = 3J (J = 1..15) and dim_action = A (1..64),
 * in floats; a pure function (no GPU needed).  One network with W output columns is
 *   W1^T [D][64] | b1 [64] | W2^T [64][64] | b2 [64] | W3^T [64][W] | b3 [W]
 * i.e. W1 at 0, b1 at 64D, W2 at 64D + 64, b2 at 64D + 4160, W3 at 64D + 4224, b3 at 64D + 4224 + 64W, and
 * 64D + 4224 + 65W floats in all.  The image is
 *   value net (W = 8: the output column zero-padded from 1 to 8) | policy net (W = A8 = 8 * ceil(A / 8), zero-padded
 *   from A) | std [A8] (= exp(log_std), zero-padded) | lognorm (= -0.5*A*log(2 pi) - sum(log_std)) | padding to a
 *   multiple of 4 floats,
 * so every section starts 16-byte aligned.  For D = 9, A = 8 this is the ROBOY_POLICY_OFF_* image above.
 * offsets[ROBOY_POLICY_LAYOUT_WORDS] receives: W1, B1, W2, B2, W3 (within either network), the b3 of the value net
 * and of the policy net (within its network), the start of the value net, the policy net, std, lognorm, and the total.
 * Returns ROBOY_E_ARG for dims outside those ranges. */
#define ROBOY_POLICY_LAYOUT_W1 0
#define ROBOY_POLICY_LAYOUT_B1 1
#define ROBOY_POLICY_LAYOUT_W2 2
#define ROBOY_POLICY_LAYOUT_B2 3
#define ROBOY_POLICY_LAYOUT_W3 4
#define ROBOY_POLICY_LAYOUT_VF_B3 5
#define ROBOY_POLICY_LAYOUT_PI_B3 6
#define ROBOY_POLICY_LAYOUT_VF 7
#define ROBOY_POLICY_LAYOUT_PI 8
#define ROBOY_POLICY_LAYOUT_STD 9
#define ROBOY_POLICY_LAYOUT_LOGNORM 10
#define ROBOY_POLICY_LAYOUT_FLOATS 11
#define ROBOY_POLICY_LAYOUT_WORDS 12
int roboy_policy_layout(int dim_obs, int dim_action, uint32_t *offsets);
int roboy_policy_rollout(roboy_env *env, uint32_t T, const float *image_dev, uint64_t noise_seed, float *obs_dev,
                         float *actions_dev, float *logp_dev, float *values_dev, float *reward_dev, uint8_t *done_dev,
                         float *noise_dev, int envs_per_thread, void *stream);
/* The same rollout with the two networks' matrix products on the tensor cores (tcgen05.mma kind::f16, M = 128
 * envs per tile, float32 accumulators in tensor memory); MSJ-shaped handles only (ROBOY_E_ARG otherwise: other
 * robots run roboy_policy_rollout).  Env outputs remain bit-identical to T roboy_step calls on
 * clip(actions, -1, 1).  Two precisions:
 *   exact = 0  float16 operands (10-bit mantissa, as TF32), float32 accumulation, tanh.approx: action means and values
 *              agree with the float32 policy to ~1e-3.  The fastest path.
 *   exact = 1  every operand split x = hi + lo into two float16 (22 mantissa bits), products accumulated as
 *              A_hi W_hi + A_hi W_lo + A_lo W_hi in float32, and the float32 kernel's tanh: agrees with the float32
 *              policy to ~1e-6, like roboy_policy_rollout, at more than twice its speed.
 * tc_image_dev: ROBOY_TC_IMAGE_BYTES bytes, 16-byte aligned.  One network is, in float16 elements,
 *   W1 [64][16] | W2 [64][80] | W3 [16][80]
 * with each W = the torch Linear weight [out][in] zero-padded (9 -> 16 inputs, 64 -> 80 inputs, 8 or 1 -> 16
 * outputs) and the BIAS stored as input column 9 (W1) / 64 (W2, W3) -- the kernel feeds a constant 1 there --
 * in the tensor core's K-major core-matrix layout without swizzle:
 *   element index of W[n][k] = (n / 8) * (K / 8) * 64 + (k / 8) * 64 + (n % 8) * 8 + (k % 8);
 * the image is  value net | policy net  (HIGH halves: float16(w)),  then the same two networks again with the LOW
 * halves float16(w - high) at byte ROBOY_TC_OFF_LO_BYTES (read only when exact = 1),  then, as float32 at byte
 * ROBOY_TC_OFF_STD_BYTES,  std [8] | lognorm | 3 floats of padding | b2 [64] | b3 [16] of the value net | the same of
 * the policy net (float32 biases of the 64-input layers: exact = 1 adds them in its epilogue instead of the product).
 * tiles_per_group selects the kernel variant (results are bit-identical across variants): 0 = choose; 1 = each group of
 * 128 threads owns one 128-env tile, four tiles per SM (large populations); 2 = two tiles per group, worked on
 * alternately (an experiment, exact = 0 only: measured 35 % slower than 1 on B200); 3 = "merged" (exact = 0 only): the
 * value and the policy network of a tile advance together, three tensor-core round trips per step instead of six --
 * chosen automatically while the population is at most two tiles per SM, where those round trips bound the step. */
#define ROBOY_TC_K_HIDDEN 80
#define ROBOY_TC_OFF_W1 0
#define ROBOY_TC_OFF_W2 1024
#define ROBOY_TC_OFF_W3 6144
#define ROBOY_TC_NET_HALVES 7424
#define ROBOY_TC_OFF_VF 0
#define ROBOY_TC_OFF_PI 7424
#define ROBOY_TC_OFF_LO_BYTES 29696
#define ROBOY_TC_OFF_STD_BYTES 59392
#define ROBOY_TC_BIAS32_NET_FLOATS 80
#define ROBOY_TC_IMAGE_BYTES 60080
int roboy_policy_rollout_tc(roboy_env *env, uint32_t T, const float *tc_image_dev, uint64_t noise_seed, float *obs_dev,
                            float *actions_dev, float *logp_dev, float *values_dev, float *reward_dev, uint8_t *done_dev,
                            float *noise_dev, int tiles_per_group, int exact, void *stream);
/* Deterministic evaluation of a policy (stable-baselines' evaluate_policy(model, env, n_eval_episodes,
 * deterministic=True)) in ONE launch, on every robot: each env plays T steps of the policy mean and records its episodes
 * as they finish; nothing grows with T.  The contract:
 *  1. Image: image_dev is the roboy_policy_layout(3J, A) image of roboy_policy_rollout.  Only the policy net is read;
 *     the value net, std and lognorm are ignored.
 *  2. Steps: every env takes exactly T steps, calls t0+1 .. t0+T of the handle's call counter, with the action
 *     clip(mean(obs), -1, 1); a NaN mean stays NaN (ROBOY_ERR_ACTION, as in the rollouts).  The mean is evaluated with
 *     the instructions roboy_policy_rollout uses, so the env outputs are those of roboy_policy_rollout with std 0.
 *  3. State after the call: call counter, goals, step words, error word, first offender and ROBOY_STAT_* advance exactly
 *     as for T roboy_step calls on those actions.
 *  4. Observations: obs_dev float32 [n][3J] is read as the observation to start from and overwritten with the
 *     observation after call T (env.step continues from it).
 *  5. Which episodes count: an episode counts only if it starts inside the call.  An env whose step counter is at its
 *     reset value (1) when the call starts begins one at call 1; after every auto-reset inside the call the next
 *     episode begins at the next call.  An episode already in progress at the call is not counted.
 *  6. Records: the first `episodes` (K) counted episodes of env e go to slot k * n + e (64-bit) of the [K][n] arrays:
 *       returns_dev float64  the sum, in step order, of the float32 rewards of the episode (what evaluate_policy sums)
 *       lengths_dev uint32   step_num - 1 at the done (the term ROBOY_STAT_SUM_EPLEN adds)
 *       reached_dev uint8    1 if the done came from _did_reach_goal (also on a step that times out as well)
 *     Slots not filled hold NaN, 0, 0.  completed_dev uint32 [n]: every counted episode of env e that finished,
 *     including those beyond K.
 *  7. Refusals (ROBOY_E_ARG with a message): auto_reset off (no new episode would ever start), a NULL pointer, an
 *     image_dev not 16-byte aligned, an obs_dev not 4-byte aligned.  T == 0 returns without a launch (outputs untouched).
 *  8. Robots: every handle runs the generic env step, MSJ-shaped ones included; their env outputs equal roboy_step's
 *     bit for bit, except rewards under joint_vel_penalty, which agree to ~2e-7 (relative).
 *  9. Sharding: results do not depend on it (draws are keyed by global env id).
 * Per env-step: 64 * (3J + 64 + A8) FMAs (A8 = 8 * ceil(A / 8)); HBM traffic is the records and the goals drawn on done. */
int roboy_policy_evaluate(roboy_env *env, uint32_t T, const float *image_dev, float *obs_dev, uint32_t episodes,
                          double *returns_dev, uint32_t *lengths_dev, uint8_t *reached_dev, uint32_t *completed_dev,
                          void *stream);
/* PPO2 update (stable-baselines 2's PPO2._train_step, as documented upstream): the clipped-surrogate loss of one minibatch
 * and its gradient with respect to every MlpPolicy parameter, in float32, on every robot (dim_obs = 3J, J = 1..15;
 * dim_action = A = 1..64).  Handle-free; runs on the current device, async on `stream`.
 *  1. Samples: s = index_dev[i], i < M (64-bit row offsets into the [n_rows] buffers obs [n_rows][D], actions
 *     [n_rows][A] (the UN-clipped samples), logp, values (the values at collection), ret).  An index outside
 *     [0, n_rows) is counted (ROBOY_PPO_STAT_BAD_INDICES) and skipped, not read; every mean below is over the
 *     M_valid = M - bad valid samples (zero when there are none).
 *  2. Advantages: adv_s = ret_s - values_s (float32), normalised over the minibatch as (adv - mean) / (std + 1e-8), with
 *     the population std; the sums are float64.
 *  3. Policy: mean, v = the float32 MlpPolicy at obs_s; std = the image's std (exp(log_std)); z = (a - mean) / std;
 *     logp_new = lognorm - 1/2 sum z^2; ratio = exp(logp_new - logp_old).
 *  4. Loss: pg_loss = mean(max(-adv ratio, -adv clip(ratio, 1 - clip_range, 1 + clip_range)));
 *     vf_loss = 1/2 mean(max((v - R)^2, (v_clip - R)^2)), v_clip = v_old + clip(v - v_old, -clip_range_vf, clip_range_vf),
 *     or 1/2 mean((v - R)^2) when clip_range_vf < 0;  entropy = sum_k (log_std_k + 1/2 log(2 pi e));
 *     loss = pg_loss - ent_coef entropy + vf_coef vf_loss.
 *  5. Gradients follow TF's rules: maximum(x, y) passes the gradient to x where x >= y, clip_by_value passes it inside
 *     the closed range; the advantages and the old values are constants.
 *  6. grad_dev: d loss / d parameter in the layout of image_dev (roboy_policy_layout(dim_obs, dim_action)); the std slots
 *     hold d loss / d log_std; padded columns, the padded std slots and the lognorm slot are 0.
 *  7. stats_dev double[ROBOY_PPO_STAT_COUNT]; approxkl = 1/2 mean((logp_new - logp_old)^2), clipfrac = mean(|ratio - 1| >
 *     clip_range).
 *  8. Determinism: the result depends only on the inputs (not on the device, the stream or a CUDA-graph replay), bit
 *     for bit: every partial sum has a fixed place and order.
 *  9. workspace_dev: at least roboy_ppo_workspace_bytes(dim_obs, dim_action, M) bytes, 8-byte aligned.  The caller
 *     must provide that size: the call sees no buffer size, only the device allocation that holds workspace_dev.
 * 10. Refusals (ROBOY_E_ARG): dims outside the layout's range, M == 0, a NULL pointer, an image not 16-byte aligned, a
 *     workspace not 8-byte aligned, not in device memory, or with fewer bytes than that between workspace_dev and the
 *     end of its device allocation (cuMemGetAddressRange).  A buffer carved from a larger allocation (a pool
 *     allocator's block) is checked against the end of that allocation, not against the buffer's own end.
 * Algorithmic FMAs per sample (hidden width 64): 256 D + 24,576 + 192 (A + 1). */
enum {
    ROBOY_PPO_STAT_LOSS = 0,
    ROBOY_PPO_STAT_PG_LOSS = 1,
    ROBOY_PPO_STAT_VF_LOSS = 2,
    ROBOY_PPO_STAT_ENTROPY = 3,
    ROBOY_PPO_STAT_APPROXKL = 4,
    ROBOY_PPO_STAT_CLIPFRAC = 5,
    ROBOY_PPO_STAT_ADV_MEAN = 6,     /* of the raw advantages ret - values over the valid samples */
    ROBOY_PPO_STAT_ADV_STD = 7,      /* population std of the same */
    ROBOY_PPO_STAT_BAD_INDICES = 8,  /* indices outside [0, n_rows) */
    ROBOY_PPO_STAT_COUNT = 9
};
int roboy_ppo_workspace_bytes(int dim_obs, int dim_action, uint64_t M, uint64_t *bytes);
int roboy_ppo_grad(int dim_obs, int dim_action, const float *image_dev, uint64_t M, const int64_t *index_dev,
                   uint64_t n_rows, const float *obs_dev, const float *actions_dev, const float *logp_dev,
                   const float *values_dev, const float *ret_dev, float clip_range, float clip_range_vf,
                   float ent_coef, float vf_coef, float *grad_dev, double *stats_dev, void *workspace_dev,
                   void *stream);

/* Launch geometry roboy_policy_rollout uses for this handle (bench.py / tests); ept = envs per thread.  Refuses the
 * envs_per_thread values roboy_policy_rollout refuses (robots other than MSJ: 0 or 1). */
int roboy_policy_geometry(roboy_env *env, int envs_per_thread, int *grid, int *block, int *smem_bytes, int *ept);
int roboy_policy_tc_geometry(roboy_env *env, int tiles_per_group, int exact, int *grid, int *block, int *smem_bytes, int *tpg);

/* Introspection for bench.py / tests: kernels launched by this handle so far, and the
 * launch geometry the step kernel uses for this n_envs. */
int roboy_launch_count(roboy_env *env, uint64_t *launches);
int roboy_step_geometry(roboy_env *env, int *grid, int *block, int *smem_bytes);
/* The robot this handle was built for: joints, tendons, floats per observation row (3 * joints), and whether the tuned
 * MSJ kernels (1) or the generic ones (0) run its fused step.  Any pointer may be NULL. */
int roboy_robot_dims(roboy_env *env, int *dim_joint, int *dim_action, int *dim_obs, int *msj_kernels);
/* How this handle's fused step divides by the spans of the robot's spaces (roboy_robot.py:95): 1 = the three-instruction
 * core, proved equal to IEEE division for these spans (offline for MSJ, oracle/verify_fastdiv.c; by exhaustion over all
 * float32 numerators on this device at roboy_create for any other robot); 0 = IEEE division.  Results are identical. */
int roboy_fast_division(roboy_env *env, int *proved);
/* How this handle's fused step evaluates the velocity penalty of roboy_env.py:98-100 for a freshly sampled state:
 * 1 = in float32, with the reference's float64 expression re-run wherever the float32 result lies within 1e-5
 * (relative) of a bound of reward_range or the env reached its goal -- the reward_range assert (:109) stays exact and
 * the reward stays within 1e-6 of the reference's; 0 = the float64 expression always (more than 8 joints, an asymmetric
 * velocity space, or ROBOY_B200_PENALTY_F64=1 in the environment). */
int roboy_penalty_float32(roboy_env *env, int *on);
/* Measurement only: an EMPTY kernel launched exactly like roboy_step launches the step kernel (grid, block,
 * programmatic dependent launch) -- the launch-latency floor bench.py reports next to the launch-bound sizes.
 * Not counted by roboy_launch_count. */
int roboy_null_step(roboy_env *env, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ROBOY_B200_H_ */
