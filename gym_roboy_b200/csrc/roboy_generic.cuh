// Robot-generic kernels: any RoboyRobot plug-in (envs/robots/roboy_robot.py:21-33 -- "MSJ platform, Upper Body, etc.",
// README.md:6-7) with up to 15 joints and 64 tendons and one bound per component.  One thread per env, runtime dims.
//
// The tuned kernels of roboy_kernels.cu / roboy_policy*.cu are the MSJ instantiation (3 joints, 8 tendons, uniform
// bounds) of the hot step; everything else -- construction / reset, the un-fused SimulationClient calls, state
// injection, stand-alone compute_reward, the external-simulator feed, and the fused step of every other robot -- runs
// through the kernels declared here, for MSJ too.
//
// Why 15 joints: numpy's norm (OpenBLAS dot) sums sequentially below 16 float64 / 32 float32 elements and in
// SIMD-blocked partial sums, whose order depends on the host CPU's kernel, above -- beyond the cap bit-exact parity
// with the reference is not defined (pinned in oracle/roboy_oracle.c's header).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "philox.cuh"
#include "roboy_kernels.cuh"

namespace roboy {

constexpr int kMaxJoint = 15, kJointPad = 16, kMaxAction = 64;
// X(J) for every joint count with its own instantiation of the generic kernels: 1..kMaxJoint
#define ROBOY_GENERIC_JOINT_COUNTS(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15)

struct RobotSpec {
    int32_t J, A;                             // joints, tendons; observation rows hold 3 * J floats
    float a_lo[kJointPad], a_hi[kJointPad];   // joint angle space   (RoboyRobot.get_joint_angles_space)
    float v_lo[kJointPad], v_hi[kJointPad];   // joint velocity space (get_joint_vels_space)
    float hold_lo[kMaxAction], hold_hi[kMaxAction];  // per tendon: the float32 interval of [-1, 1] actions whose rescale
                                                     // (roboy_env.py:157-158) passes numpy's allclose(., 0)
                                                     // (simulation_client.py:38); lo > hi = empty
    float thr_angle, thr_vel;                 // roboy_env.py:24-25,127,130
    // ---- derived on the host (fill_robot_spec), read by the fused step only ----
    float a_span[kJointPad], v_span[kJointPad];      // fl32(max_k - min_k), the divisor of roboy_robot.py:95
    float a_span21[kJointPad];                       // a_span * 2^-21 (exact): the grid step of a state draw
    double v_gz[kJointPad];                          // roboy_robot.py:93-95 on the float64 zero velocity of the goal
    float v_gz_f[kJointPad];                         // (float)v_gz[k]; exact whenever pen.on
    PenaltyF32 pen;                                  // float32 evaluation of the velocity penalty (msj_math.cuh), J <= 8
    float thr_angle_sq_hi;                           // thr_angle^2 * (1 + 1e-5), rounded up: pre-filter of _did_reach_goal
    float hold_c, hold_h;                            // no action with |x - hold_c| > hold_h lies in any hold interval
    float hold_pad;                                  // a value in [-1, 1] outside that hull (hold_h < 0: nobody can hold)
    // ---- derived on the DEVICE and proved there by exhaustion (prove_generic_fastdiv) ----
    float a_rcp[kJointPad], v_rcp[kJointPad];        // the refined reciprocal the compiler's own division starts from
    int32_t fastdiv;                                 // 1: t / span == fma(rcp, fma(-span, t * rcp, t), t * rcp) for every t in
                                                     // [2^-60, 2^60] and each span of this robot, checked over all 2^32 floats
    float penalty_boundary, bonus_goal;       // roboy_env.py:26-27
    double reward_lo, reward_hi;              // roboy_env.py:30,109
};

struct GStepParams {
    uint64_t n, e_begin, e_end, gid_base;     // e_begin % 32 == 0
    CallCounter cc;
    PhiloxKeys keys;
    RobotSpec r;
    int32_t max_len;
    int32_t penalty, bonus, auto_reset;
    const float *actions;   // [n][A] in [-1, 1]
    float *goal;            // [J][n]
    uint32_t *step_flags;   // [n]
    const float *held;      // [2J][n]
    float *obs;             // [n][3J]
    float *reward;          // [n]
    uint8_t *done;          // [n]
    float *terminal_obs;    // [n][3J] or nullptr
    uint32_t *done_bits;    // [ceil(n/32)] or nullptr
    double *stats;
    uint32_t *err_flags;
    unsigned long long *first_bad;
};
cudaError_t launch_generic_step(const GStepParams &p, int sm_count, cudaStream_t stream);
void generic_step_geometry(int J, uint64_t envs, int sm_count, int *grid, int *block, int *smem_bytes);

// Fills r.a_rcp / r.v_rcp / r.fastdiv.  The normalisation of roboy_robot.py:93-95 divides by a per-joint constant; IEEE
// division costs ~11 instructions and a branch, its in-range core (reciprocal refined once, quotient corrected once) three
// when the reciprocal is known.  Whether that core returns the correctly rounded quotient for EVERY float32 numerator in
// [2^-60, 2^60] is checked on this device for each distinct span (all 2^32 bit patterns, ~3 ms per span, cached per
// process); a span that fails, or one outside [2^-40, 2^40], leaves fastdiv = 0 and the kernel on IEEE division.
cudaError_t prove_generic_fastdiv(RobotSpec &r, int sm_count, cudaStream_t stream);

struct GInitParams {
    uint64_t n, gid_base;
    CallCounter cc;
    PhiloxKeys keys;
    RobotSpec r;
    float *goal;
    uint32_t *step_flags;
    float *held;           // nullptr for reset (the held state becomes the zero state through the flag)
    const uint8_t *mask;   // nullptr: all envs
    float *obs;            // nullptr: do not write observations
};
// init (held != nullptr): RoboyEnv.__init__ / Stub.__init__;  reset (held == nullptr): RoboyEnv.reset
cudaError_t launch_generic_init_or_reset(const GInitParams &p, int sm_count, cudaStream_t stream);

struct GRewardParams {
    uint64_t k, gid_base;
    RobotSpec r;
    int32_t penalty, bonus, check_range;
    const float *q, *qd, *goal_q, *goal_qd;  // [k][J]; goal_qd may be nullptr (the float64 zeros of roboy_env.py:23)
    const uint8_t *feasible;                 // [k] or nullptr
    double *reward;                          // [k]
    uint8_t *reached;                        // [k] or nullptr
    double *stats;
    uint32_t *err_flags;
    unsigned long long *first_bad;
};
cudaError_t launch_generic_compute_reward(const GRewardParams &p, int sm_count, cudaStream_t stream);

struct GScatterParams {
    uint64_t k, n, gid_base;
    RobotSpec r;
    const int64_t *idx;
    // any of the following groups may be null
    const float *goal_q;        // [k][J] -> goal (bounds-checked, roboy_robot.py:76)
    const float *q, *qd;        // [k][J] -> held (+ flags)
    const uint8_t *feasible;
    const int32_t *step;        // -> step_num
    float *goal, *held;
    uint32_t *step_flags;
    uint32_t *err_flags;
    unsigned long long *first_bad;
    float *out_q, *out_qd;      // gather (SimulationClient.read_state): [k][J]
    uint8_t *out_feasible;      // bit 0 is_feasible, bit 1 float64 zero state
};
cudaError_t launch_generic_scatter(const GScatterParams &p, int sm_count, cudaStream_t stream);

// The un-fused plug-in calls of SimulationClient (simulation_client.py:11-23), batched:
//   mode 0  forward_step_command(action in robot units)  -> state      (:36-40)
//   mode 1  forward_reset_command()                      -> zero state (:42-44), masked
//   mode 2  get_new_goal_joint_angles()                  -> goal draw  (:46-47), does not touch env state
struct GSimParams {
    int mode;
    uint64_t n, gid_base;
    CallCounter cc;
    uint32_t sub;
    PhiloxKeys keys;
    RobotSpec r;
    const float *actions;   // mode 0: [n][A] robot units
    const uint8_t *mask;    // mode 1
    uint32_t *step_flags;
    const float *held;
    float *out_q, *out_qd;  // [n][J]; mode 2 writes the goal to out_q
    uint8_t *out_feasible;  // [n] or nullptr
    double *stats;
};
cudaError_t launch_generic_sim(const GSimParams &p, int sm_count, cudaStream_t stream);

// RoboyEnv.step / reset when the states come from an EXTERNAL simulator (the role of RosSimulationClient,
// ros_simulation_client.py:40-60: q, qdot, feasible arrive over the wire and are held as float64 arrays).
struct GExternalParams {
    int reset;                 // 0: step (roboy_env.py:51-70), 1: reset (roboy_env.py:82-87)
    uint64_t n, gid_base;
    CallCounter cc;
    PhiloxKeys keys;
    RobotSpec r;
    int32_t penalty, bonus, max_len;
    const float *q, *qd;       // [n][J]
    const uint8_t *feasible;   // [n] or nullptr
    const uint8_t *mask;       // reset only; nullptr = all
    float *goal;
    uint32_t *step_flags;
    float *obs, *reward;
    uint8_t *done;
    double *stats;
    uint32_t *err_flags;
    unsigned long long *first_bad;
};
cudaError_t launch_generic_external(const GExternalParams &p, int sm_count, cudaStream_t stream);

}  // namespace roboy
