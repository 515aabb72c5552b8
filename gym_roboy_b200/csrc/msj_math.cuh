// Device arithmetic of the env step: normalisation, goal distance, reward, done test.
//
// Written against the reference's operation ORDER and numpy's dtype promotions, because the
// done mask has to be bit-exact (paths relative to gym_roboy/ in Roboy/gym-roboy):
//   normalisation   envs/robots/roboy_robot.py:93-95   (2*v - max - min) / (max - min)
//   _l2_distance    envs/roboy_env.py:137-140          subtract, NaN -> 0, np.linalg.norm
//   compute_reward  envs/roboy_env.py:92-112
//   _did_reach_goal envs/roboy_env.py:125-134
// np.linalg.norm(float32[3]) accumulates the float32 products in a double (OpenBLAS sdot) and
// rounds once to float32 before the float32 sqrt; float64 operands accumulate sequentially with FMA.  All
// arithmetic below uses the round-to-nearest intrinsics so nvcc never contracts a multiply and
// an add into an FMA (numpy does not fuse).
#pragma once
#include <math.h>
#include <stdint.h>

namespace roboy {

struct RobotConsts {
    float a_hi, a_lo, a_span;  // joint angle space (msj_robot.py:9), a_span = fl32(a_hi - a_lo)
    float v_hi, v_lo, v_span;  // joint velocity space (msj_robot.py:10)
    float thr_angle;           // fl32(_MAX_DISTANCE_JOINT_ANGLE / 200)  roboy_env.py:24,127
    float thr_vel;             // fl32(_MAX_DISTANCE_JOINT_VELS / 5)     roboy_env.py:25,130
    float penalty_boundary;    // roboy_env.py:26
    float bonus_goal;          // roboy_env.py:27
    double reward_lo, reward_hi;  // roboy_env.py:30,109
};

__device__ __forceinline__ float normalize32(float v, float hi, float lo, float span) {
    float t = __fmul_rn(2.0f, v);
    t = __fsub_rn(t, hi);
    t = __fsub_rn(t, lo);
    return __fdiv_rn(t, span);
}

__device__ __forceinline__ double normalize64(double v, float hi, float lo, float span) {
    double t = __dmul_rn(2.0, v);
    t = __dsub_rn(t, (double)hi);
    t = __dsub_rn(t, (double)lo);
    return __ddiv_rn(t, (double)span);
}

__device__ __forceinline__ float nan_to_zero(float d) { return (d != d) ? 0.0f : d; }
__device__ __forceinline__ double nan_to_zero(double d) { return (d != d) ? 0.0 : d; }

// ||a - b||_2 for float32 operands, exactly as numpy/OpenBLAS evaluate it.  GUARD: the NaN -> 0 of _l2_distance
// (roboy_env.py:139); the penalty term (:99) calls np.linalg.norm on the difference directly and has none -- a NaN velocity
// makes that reward NaN (tools/soak_api.py found the guarded form returning a finite one for injected NaN velocities).
template <bool GUARD = true>
__device__ __forceinline__ float l2_f32(float a0, float a1, float a2, float b0, float b1, float b2) {
    const float d0 = GUARD ? nan_to_zero(__fsub_rn(a0, b0)) : __fsub_rn(a0, b0);
    const float d1 = GUARD ? nan_to_zero(__fsub_rn(a1, b1)) : __fsub_rn(a1, b1);
    const float d2 = GUARD ? nan_to_zero(__fsub_rn(a2, b2)) : __fsub_rn(a2, b2);
    double s = (double)__fmul_rn(d0, d0);
    s = __dadd_rn(s, (double)__fmul_rn(d1, d1));
    s = __dadd_rn(s, (double)__fmul_rn(d2, d2));
    return __fsqrt_rn((float)s);
}

// ||a - b||_2 once numpy has promoted to float64.
template <bool GUARD = true>
__device__ __forceinline__ double l2_f64(double a0, double a1, double a2, double b0, double b1, double b2) {
    const double d0 = GUARD ? nan_to_zero(__dsub_rn(a0, b0)) : __dsub_rn(a0, b0);
    const double d1 = GUARD ? nan_to_zero(__dsub_rn(a1, b1)) : __dsub_rn(a1, b1);
    const double d2 = GUARD ? nan_to_zero(__dsub_rn(a2, b2)) : __dsub_rn(a2, b2);
    // OpenBLAS ddot's scalar tail (n < 16) is compiled with FMA contraction: s = fma(d, d, s), sequentially -- pinned
    // against numpy in oracle/roboy_oracle.c's header.  (With float32-valued operands the products are exact and the
    // unfused sum gives the same bits; with the float64 normalised zero of an asymmetric velocity space it does not.)
    double s = __dmul_rn(d0, d0);
    s = __fma_rn(d1, d1, s);
    s = __fma_rn(d2, d2, s);
    return __dsqrt_rn(s);
}

// ---------------------------------------------------------------------------------------------
// Hot path: state freshly sampled (float32, feasible, finite), goal angles float32 inside the
// angle space, goal velocities the float64 zeros of roboy_env.py:23.
//
// Three exactness-preserving shortcuts keep this path short (it is issue-bound otherwise):
//  * FASTDIV: x / c as  q0 = x*rc; r = fma(-q0, c, x); q = fma(r, rc, q0)  -- bit-identical to the
//    IEEE division for every numerator this path can produce with the MSJ constants (proved by
//    exhaustion: oracle/verify_fastdiv.c, tests/test_fastdiv_proof.py): kDivProved.  An MSJ-shaped
//    robot with OTHER limits gets the same three instructions with the reciprocal derived and the
//    identity checked on the device when the handle is created (prove_generic_fastdiv: all 2^32
//    numerators, valid for 2^-60 <= |x| <= 2^60), plus a range test of the numerators that sends
//    the rare env outside it (x == 0) through __fdiv_rn: kDivChecked.  Spans that fail: kDivIeee.
//  * the done test's angle distance is first bounded with a 3-instruction float32 estimate
//    against a threshold widened by 1e-5 (the estimate is within 4e-7 of the exact sum); the
//    exact numpy-order evaluation runs only when that cannot exclude "close".
//  * NaN -> 0 of _l2_distance (roboy_env.py:139) cannot trigger: all operands are finite.
// ---------------------------------------------------------------------------------------------
// float32 evaluation of the velocity penalty (roboy_env.py:98-100) on the sampled-state path.  The reference evaluates
//   (||nv - gz||_2 + 1) * (r - exp(r))   in float64 (gz, the goal's normalised zero velocity, is float64) and returns a
// float; only two things are observable: the reward to 1e-6 relative (north_star) and whether it lies inside reward_range
// (:109, exact).  The float32 chain  e = nv - gz_f, s = fma(e, e, ...), (sqrt_rn(s) + 1) * (r - exp(r))  differs from the
// rounded float64 result by at most (J/2 + 4) roundings of 2^-24 (3.3e-7 at 3 joints; allowed up to 8 joints), so it
// decides the range test everywhere except within 1e-5 (relative) of a bound -- there, and for an env that reached its
// goal, the float64 expression runs as before.  Enabled on the host only when gz is a float32 value (symmetric velocity
// spaces: gz = 0) and no normalised velocity can exceed 1e9 (float32 sum of squares stays finite).
struct PenaltyF32 {
    int32_t on;
    float lo_c;     // (float)reward_lo
    float band;     // 1e-5 |reward_lo|, rounded up:  |r - lo_c| > band  =>  r and the float64 result lie on the same side of
                    // reward_lo (r differs from it by < 1e-6 relative, lo_c from reward_lo by 6e-8)
    float hi_in;    // reward_hi - 1e-5 |reward_hi|, rounded down:  r < hi_in  =>  float64 result <= reward_hi
};

// sqrt of the float32 penalty sum: MUFU.SQRT directly (sqrt.approx.ftz: 2^-23 relative error, one rounding more than the
// correctly rounded __fsqrt_rn and ~7 instructions fewer -- the penalty kernels are issue-bound: 0.909 -> 0.918 of HBM peak).
__device__ __forceinline__ float penalty_sqrt(float s) {
    float v;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(v) : "f"(s));
    return v;
}

struct FastConsts {
    float a_rc, v_rc;        // RN(1 / a_span), RN(1 / v_span)
    float thr_angle_sq_hi;   // (thr_angle^2) * (1 + 1e-5), rounded up
    float a_span24;          // a_span * 2^-24 (exact): goal draws,  v = low + a_span24 * float(x >> 8)
    float a_span21;          // a_span * 2^-21 (exact): state draws, v = low + a_span21 * float(k), k < 2^21
    float reward_lo_f, reward_hi_f;  // reward range rounded INWARD to float32: for a float32 reward
                                     // r,  lo <= r <= hi  <=>  reward_lo_f <= r <= reward_hi_f
    double v_gz;             // the normalised float64 zero velocity of the goal (roboy_env.py:23,95):
                             // ((2*0.0 - v_hi) - v_lo) / v_span in float64 -- a constant of the robot, derived on the host
                             // (in the kernel it was a double-precision division per env-step)
    float v_gz_f;            // (float)v_gz, used when pen.on (then exact)
    PenaltyF32 pen;
};

constexpr int kDivIeee = 0, kDivProved = 1, kDivChecked = 2;
constexpr float kDivCheckedLo = 0x1p-60f, kDivCheckedHi = 0x1p60f;

template <int FASTDIV>
__device__ __forceinline__ float div_span(float t, float span, float rc) {
    if (FASTDIV != kDivIeee) {
        const float q0 = __fmul_rn(t, rc);
        const float r = fmaf(-q0, span, t);
        return fmaf(r, rc, q0);
    }
    return __fdiv_rn(t, span);
}

// one value (the rare callers: a goal normalised when it is drawn or loaded)
template <int FASTDIV>
__device__ __forceinline__ float normalize32_hot(float v, float hi, float lo, float span, float rc) {
    const float t = __fsub_rn(__fsub_rn(__fmul_rn(2.0f, v), hi), lo);
    if (FASTDIV == kDivChecked) {
        const float at = fabsf(t);
        if (!(at >= kDivCheckedLo && at <= kDivCheckedHi)) return __fdiv_rn(t, span);
    }
    return div_span<FASTDIV>(t, span, rc);
}

// three values of one space (the hot callers): under kDivChecked the three numerators are range-tested together
template <int FASTDIV>
__device__ __forceinline__ void normalize32_hot3(float v0, float v1, float v2, float hi, float lo, float span, float rc,
                                                 float &n0, float &n1, float &n2) {
    const float t0 = __fsub_rn(__fsub_rn(__fmul_rn(2.0f, v0), hi), lo);
    const float t1 = __fsub_rn(__fsub_rn(__fmul_rn(2.0f, v1), hi), lo);
    const float t2 = __fsub_rn(__fsub_rn(__fmul_rn(2.0f, v2), hi), lo);
    n0 = div_span<FASTDIV>(t0, span, rc);
    n1 = div_span<FASTDIV>(t1, span, rc);
    n2 = div_span<FASTDIV>(t2, span, rc);
    if (FASTDIV == kDivChecked) {
        const float mn = fminf(fminf(fabsf(t0), fabsf(t1)), fabsf(t2)), mx = fmaxf(fmaxf(fabsf(t0), fabsf(t1)), fabsf(t2));
        if (!(mn >= kDivCheckedLo && mx <= kDivCheckedHi)) {
            n0 = __fdiv_rn(t0, span);
            n1 = __fdiv_rn(t1, span);
            n2 = __fdiv_rn(t2, span);
        }
    }
}

template <bool PENALTY, bool BONUS, int FASTDIV>
__device__ __forceinline__ void reward_reached_sampled_ng(float q0, float q1, float q2, float qd0, float qd1, float qd2,
                                                          float g0, float g1, float g2, float ng0, float ng1,
                                                          float ng2, const RobotConsts &c, const FastConsts &f,
                                                          float &reward_out, bool &reached, bool &violation) {
    // ng0..2: the goal already normalised (normalize32_hot) -- the open-loop kernel keeps it in registers
    // _did_reach_goal (:125-134): angles in float32, velocities in float64 -- evaluated exactly
    // only when the cheap bound cannot rule "close" out.
    reached = false;
    {
        const float e0 = __fsub_rn(q0, g0), e1 = __fsub_rn(q1, g1), e2 = __fsub_rn(q2, g2);
        const float est = fmaf(e2, e2, fmaf(e1, e1, __fmul_rn(e0, e0)));
        if (est <= f.thr_angle_sq_hi) {
            double s = (double)__fmul_rn(e0, e0);
            s = __dadd_rn(s, (double)__fmul_rn(e1, e1));
            s = __dadd_rn(s, (double)__fmul_rn(e2, e2));
            if (__fsqrt_rn((float)s) < c.thr_angle)
                reached = l2_f64((double)qd0, (double)qd1, (double)qd2, 0.0, 0.0, 0.0) < (double)c.thr_vel;
        }
    }
    // compute_reward :94-96
    float nq0, nq1, nq2;
    normalize32_hot3<FASTDIV>(q0, q1, q2, c.a_hi, c.a_lo, c.a_span, f.a_rc, nq0, nq1, nq2);
    const float d0 = __fsub_rn(nq0, ng0), d1 = __fsub_rn(nq1, ng1), d2 = __fsub_rn(nq2, ng2);
    double s = (double)__fmul_rn(d0, d0);                    // OpenBLAS sdot: float products, double sum
    s = __dadd_rn(s, (double)__fmul_rn(d1, d1));
    s = __dadd_rn(s, (double)__fmul_rn(d2, d2));
    float r32 = -expf(__fsqrt_rn((float)s));
    if (PENALTY) {  // :98-100, float64 because the goal velocities are
        // (every operand is finite on this path, so the NaN -> 0 of _l2_distance cannot trigger -- and :99 has none anyway)
        float nv0, nv1, nv2;
        normalize32_hot3<FASTDIV>(qd0, qd1, qd2, c.v_hi, c.v_lo, c.v_span, f.v_rc, nv0, nv1, nv2);
        const float diff = __fsub_rn(r32, expf(r32));
        bool exact = true;
        if (f.pen.on) {   // float32 chain + band test (PenaltyF32)
            // kDivProved is MSJ's instantiation: its velocity space is symmetric, gz = +0 and nv - gz = nv
            const bool gz0 = FASTDIV == kDivProved;
            const float e0 = gz0 ? nv0 : __fsub_rn(nv0, f.v_gz_f), e1 = gz0 ? nv1 : __fsub_rn(nv1, f.v_gz_f),
                        e2 = gz0 ? nv2 : __fsub_rn(nv2, f.v_gz_f);
            const float r = __fmul_rn(__fadd_rn(penalty_sqrt(fmaf(e2, e2, fmaf(e1, e1, __fmul_rn(e0, e0)))), 1.0f), diff);
            // an env that reached its goal takes the float64 expression: a NaN fails both comparisons below
            const float rt = reached ? __int_as_float(0x7fc00000) : r;
            const float t = __fsub_rn(rt, f.pen.lo_c);
            if (fabsf(t) > f.pen.band && rt < f.pen.hi_in) {
                reward_out = r;
                violation = t < 0.0f;  // :109
                exact = false;
            }
        }
        if (exact) {
            const double gz = f.v_gz;
            const double e0 = __dsub_rn((double)nv0, gz), e1 = __dsub_rn((double)nv1, gz), e2 = __dsub_rn((double)nv2, gz);
            const double v = __dsqrt_rn(__fma_rn(e2, e2, __fma_rn(e1, e1, __dmul_rn(e0, e0))));
            double r64 = __dmul_rn(__dadd_rn(v, 1.0), (double)diff);
            if (BONUS && reached) r64 = __dadd_rn(r64, (double)c.bonus_goal);  // :105-107
            reward_out = (float)r64;
            violation = !(c.reward_lo <= r64 && r64 <= c.reward_hi);  // :109
        }
    } else {
        if (BONUS && reached) r32 = __fadd_rn(r32, c.bonus_goal);
        reward_out = r32;
        violation = !(r32 >= f.reward_lo_f && r32 <= f.reward_hi_f);  // :109
    }
}

template <bool PENALTY, bool BONUS, int FASTDIV>
__device__ __forceinline__ void reward_reached_sampled(float q0, float q1, float q2, float qd0, float qd1, float qd2,
                                                       float g0, float g1, float g2, const RobotConsts &c,
                                                       const FastConsts &f, float &reward_out, bool &reached,
                                                       bool &violation) {
    reward_reached_sampled_ng<PENALTY, BONUS, FASTDIV>(
        q0, q1, q2, qd0, qd1, qd2, g0, g1, g2, normalize32_hot<FASTDIV>(g0, c.a_hi, c.a_lo, c.a_span, f.a_rc),
        normalize32_hot<FASTDIV>(g1, c.a_hi, c.a_lo, c.a_span, f.a_rc),
        normalize32_hot<FASTDIV>(g2, c.a_hi, c.a_lo, c.a_span, f.a_rc), c, f, reward_out, reached, violation);
}

// ---------------------------------------------------------------------------------------------
// General path: any state dtype the reference can hold (float32 sample / injected state, or the
// float64 zero state), feasibility flag, optional float32 goal velocities.  Used by the hold
// branch of the step, and by the stand-alone compute_reward kernel.
// ---------------------------------------------------------------------------------------------
struct HeldState {
    double q[3], qd[3];  // float32-valued unless is64
    bool is64;           // numpy dtype of the arrays: float64 zero state vs float32
    bool feasible;
};

static __device__ __noinline__ void reward_reached_general(const HeldState &s, const float g[3], bool has_goal_qd,
                                                    const float gqd[3], bool penalty, bool bonus,
                                                    const RobotConsts &c, double &reward_out, bool &reached,
                                                    bool &violation) {
    bool angles_close, vels_close;
    if (!s.is64) {
        angles_close = l2_f32((float)s.q[0], (float)s.q[1], (float)s.q[2], g[0], g[1], g[2]) < c.thr_angle;
    } else {
        angles_close = l2_f64(s.q[0], s.q[1], s.q[2], (double)g[0], (double)g[1], (double)g[2]) < (double)c.thr_angle;
    }
    if (!s.is64 && has_goal_qd) {
        vels_close = l2_f32((float)s.qd[0], (float)s.qd[1], (float)s.qd[2], gqd[0], gqd[1], gqd[2]) < c.thr_vel;
    } else {
        const double v0 = has_goal_qd ? (double)gqd[0] : 0.0, v1 = has_goal_qd ? (double)gqd[1] : 0.0,
                     v2 = has_goal_qd ? (double)gqd[2] : 0.0;
        vels_close = l2_f64(s.qd[0], s.qd[1], s.qd[2], v0, v1, v2) < (double)c.thr_vel;
    }
    reached = angles_close && vels_close;

    float ng[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) ng[k] = normalize32(g[k], c.a_hi, c.a_lo, c.a_span);
    float r32 = 0.0f;
    double r = 0.0;
    bool r_is64;
    if (!s.is64) {
        const float n0 = normalize32((float)s.q[0], c.a_hi, c.a_lo, c.a_span);
        const float n1 = normalize32((float)s.q[1], c.a_hi, c.a_lo, c.a_span);
        const float n2 = normalize32((float)s.q[2], c.a_hi, c.a_lo, c.a_span);
        r32 = -expf(l2_f32(n0, n1, n2, ng[0], ng[1], ng[2]));
        r = (double)r32;
        r_is64 = false;
    } else {
        const double n0 = normalize64(s.q[0], c.a_hi, c.a_lo, c.a_span);
        const double n1 = normalize64(s.q[1], c.a_hi, c.a_lo, c.a_span);
        const double n2 = normalize64(s.q[2], c.a_hi, c.a_lo, c.a_span);
        r = -exp(l2_f64(n0, n1, n2, (double)ng[0], (double)ng[1], (double)ng[2]));
        r_is64 = true;
    }
    if (penalty) {
        if (!s.is64 && has_goal_qd) {  // everything float32 (roboy_env.py:40-49 path)
            const float v = l2_f32<false>(normalize32((float)s.qd[0], c.v_hi, c.v_lo, c.v_span),
                                   normalize32((float)s.qd[1], c.v_hi, c.v_lo, c.v_span),
                                   normalize32((float)s.qd[2], c.v_hi, c.v_lo, c.v_span),
                                   normalize32(gqd[0], c.v_hi, c.v_lo, c.v_span),
                                   normalize32(gqd[1], c.v_hi, c.v_lo, c.v_span),
                                   normalize32(gqd[2], c.v_hi, c.v_lo, c.v_span));
            r32 = __fmul_rn(__fadd_rn(v, 1.0f), __fsub_rn(r32, expf(r32)));
            r = (double)r32;
        } else {
            double nv[3], ngv[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                nv[k] = s.is64 ? normalize64(s.qd[k], c.v_hi, c.v_lo, c.v_span)
                               : (double)normalize32((float)s.qd[k], c.v_hi, c.v_lo, c.v_span);
                ngv[k] = has_goal_qd ? (double)normalize32(gqd[k], c.v_hi, c.v_lo, c.v_span)
                                     : normalize64(0.0, c.v_hi, c.v_lo, c.v_span);
            }
            const double v = l2_f64<false>(nv[0], nv[1], nv[2], ngv[0], ngv[1], ngv[2]);   // :99: no NaN guard
            const double diff = r_is64 ? __dsub_rn(r, exp(r)) : (double)__fsub_rn(r32, expf(r32));
            r = __dmul_rn(__dadd_rn(v, 1.0), diff);
            r_is64 = true;
        }
    }
    if (!s.feasible) {  // :102-103  float32 - int64 scalar promotes to float64
        r = __dsub_rn(r, (double)c.penalty_boundary);
        r_is64 = true;
    }
    if (reached && bonus) {  // :105-107
        if (r_is64) r = __dadd_rn(r, (double)c.bonus_goal);
        else r = (double)__fadd_rn((float)r, c.bonus_goal);
    }
    violation = !(c.reward_lo <= r && r <= c.reward_hi);
    reward_out = r;
}

}  // namespace roboy
