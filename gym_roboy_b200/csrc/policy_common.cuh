// Pieces shared by the fused policy rollout kernels (float32 FFMA2: roboy_policy.cu and, for every other robot,
// roboy_policy_generic.cu; tcgen05 TF32: roboy_policy_tc.cu): the 64-wide dense layer, the Gaussian sample, the clip and
// ONE env's RoboyEnv.step on the action just produced -- the MSJ step kernel's arithmetic, instruction for instruction
// (roboy_kernels.cu, process_chunk).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/roboy_b200.h"
#include "roboy_kernels.cuh"
#include "roboy_policy.cuh"
#include "step_rare.cuh"

namespace roboy {
namespace {

constexpr uint32_t kFullMask = 0xffffffffu;

__device__ __forceinline__ float tanh_mufu(float x) {
    // tanh x = 1 - 2 / (e^{2x} + 1); ex2.approx and rcp.approx are accurate to ~1 ulp, so the
    // absolute error is a few 1e-7 everywhere (the cancellation near 0 costs relative, not absolute,
    // accuracy).  e = inf gives 1, e = 0 gives -1, NaN propagates.
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__fmul_rn(x, 2.885390081777927f)));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fadd_rn(e, 1.0f)));
    return fmaf(-2.0f, r, 1.0f);
}

// acc[e][j2] (outputs 2*j2, 2*j2+1 of env e) += sum_k x_e[k] * W[k][.]; W is [K][64] in shared memory
// (every lane reads the same 16 bytes: a broadcast), x_e[k] sits at x[k * ks + e * es] (thread-private).
template <int E>
__device__ __forceinline__ void dense64(const float *__restrict__ W, const float *__restrict__ x, int K, int ks, int es,
                                        float2 (&acc)[E][32]) {
#pragma unroll 2
    for (int k = 0; k < K; ++k) {
        float2 hh[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const float h = x[k * ks + e * es];
            hh[e] = make_float2(h, h);
        }
        const float4 *w4 = reinterpret_cast<const float4 *>(W + k * ROBOY_POLICY_HIDDEN);
#pragma unroll
        for (int jb = 0; jb < 16; ++jb) {
            const float4 w = w4[jb];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                acc[e][2 * jb] = __ffma2_rn(make_float2(w.x, w.y), hh[e], acc[e][2 * jb]);
                acc[e][2 * jb + 1] = __ffma2_rn(make_float2(w.z, w.w), hh[e], acc[e][2 * jb + 1]);
            }
        }
    }
}

template <int E>
__device__ __forceinline__ void load_bias64(const float *__restrict__ b, float2 (&acc)[E][32]) {
#pragma unroll
    for (int jb = 0; jb < 16; ++jb) {
        const float4 v = reinterpret_cast<const float4 *>(b)[jb];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            acc[e][2 * jb] = make_float2(v.x, v.y);
            acc[e][2 * jb + 1] = make_float2(v.z, v.w);
        }
    }
}

// Two standard normals from two 32-bit words (Box-Muller on the MUFU unit).
__device__ __forceinline__ float2 box_muller(uint32_t x, uint32_t y) {
    const float u1 = fmaf(__uint2float_rn(x >> 8), 0x1p-24f, 0x1p-25f);  // (0, 1)
    const float u2 = __fmul_rn(__uint2float_rn(y >> 8), 0x1p-24f);        // [0, 1)
    const float r = __fsqrt_rn(__fmul_rn(-2.0f, __logf(u1)));
    float s, c;
    __sincosf(__fmul_rn(6.283185307179586f, u2), &s, &c);
    return make_float2(__fmul_rn(r, c), __fmul_rn(r, s));
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

struct EnvRegs {
    float g0, g1, g2, ng0, ng1, ng2;
    uint32_t sf;
};

// The env flags are run-time here (the kernel is FMA-bound in the networks; 2 instantiations instead of 32).
template <bool FASTDIV>
__device__ __forceinline__ void reward_reached_rt(bool penalty, bool bonus, float q0, float q1, float q2, float qd0,
                                                  float qd1, float qd2, const EnvRegs &s, const RobotConsts &c,
                                                  const FastConsts &f, float &reward, bool &reached, bool &violation) {
    if (penalty) {
        if (bonus) reward_reached_sampled_ng<true, true, FASTDIV>(q0, q1, q2, qd0, qd1, qd2, s.g0, s.g1, s.g2, s.ng0, s.ng1, s.ng2, c, f, reward, reached, violation);
        else reward_reached_sampled_ng<true, false, FASTDIV>(q0, q1, q2, qd0, qd1, qd2, s.g0, s.g1, s.g2, s.ng0, s.ng1, s.ng2, c, f, reward, reached, violation);
    } else {
        if (bonus) reward_reached_sampled_ng<false, true, FASTDIV>(q0, q1, q2, qd0, qd1, qd2, s.g0, s.g1, s.g2, s.ng0, s.ng1, s.ng2, c, f, reward, reached, violation);
        else reward_reached_sampled_ng<false, false, FASTDIV>(q0, q1, q2, qd0, qd1, qd2, s.g0, s.g1, s.g2, s.ng0, s.ng1, s.ng2, c, f, reward, reached, violation);
    }
}

template <bool FASTDIV>
__device__ __forceinline__ void normalize_goal(EnvRegs &s, const RobotConsts &c, const FastConsts &f) {
    s.ng0 = normalize32_hot<FASTDIV>(s.g0, c.a_hi, c.a_lo, c.a_span, f.a_rc);
    s.ng1 = normalize32_hot<FASTDIV>(s.g1, c.a_hi, c.a_lo, c.a_span, f.a_rc);
    s.ng2 = normalize32_hot<FASTDIV>(s.g2, c.a_hi, c.a_lo, c.a_span, f.a_rc);
}

// One env: a = mean + std * N(0, 1) (stored un-clipped, with its log-density), clipped to the action space as
// PPO2's runner does before env.step, then RoboyEnv.step (roboy_env.py:51-70) on it.  `row` is the env's row of
// the obs stage in shared memory: on return it holds the observation the policy sees next.
__device__ __forceinline__ void sample_and_step(const StepParams &p, const PolicyParams &q, const float *__restrict__ sd,
                                                float lognorm, const float (&mean)[8], EnvRegs &s, bool live, uint32_t env,
                                                uint32_t tt, uint64_t t, float *__restrict__ row, unsigned int *s_cnt,
                                                float &sum_reward) {
    const bool PENALTY = q.penalty, BONUS = q.bonus, AUTO_RESET = q.auto_reset, FASTDIV = q.fastdiv;
    const size_t n = (size_t)p.n;
    const uint64_t gid = p.gid_base + env;
    // ---- a = mean + std * N(0, 1); the runner clips it to the action space for env.step ----
    const uint4 r0 = philox_draw(gid, t, kStreamNoise, q.noise_keys, 0);
    const uint4 r1 = philox_draw(gid, t, kStreamNoise, q.noise_keys, 1);
    const float2 z01 = box_muller(r0.x, r0.y), z23 = box_muller(r0.z, r0.w);
    const float2 z45 = box_muller(r1.x, r1.y), z67 = box_muller(r1.z, r1.w);
    const float z[8] = {z01.x, z01.y, z23.x, z23.y, z45.x, z45.y, z67.x, z67.y};
    float u[8], a[8], zz = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        u[k] = fmaf(sd[k], z[k], mean[k]);
        const float c = fminf(fmaxf(u[k], p.act_in_lo), p.act_in_hi);
        a[k] = (u[k] != u[k]) ? u[k] : c;  // a NaN stays a NaN (and trips the :52 assert below)
        zz = fmaf(z[k], z[k], zz);
    }
    const float logp = fmaf(-0.5f, zz, lognorm);
    if (live) {
        float4 *ap = reinterpret_cast<float4 *>(q.actions + ((size_t)tt * n + env) * kActDim);
        ap[0] = make_float4(u[0], u[1], u[2], u[3]);
        ap[1] = make_float4(u[4], u[5], u[6], u[7]);
        q.logp[(size_t)tt * n + env] = logp;
        if (q.noise) {
            float4 *np = reinterpret_cast<float4 *>(q.noise + ((size_t)tt * n + env) * kActDim);
            np[0] = make_float4(z[0], z[1], z[2], z[3]);
            np[1] = make_float4(z[4], z[5], z[6], z[7]);
        }
    }

    // ---- RoboyEnv.step on that action: same arithmetic as step_kernel ----
    bool act_ok = true, hold = live;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        act_ok = act_ok && fabsf(a[k]) <= p.act_in_hi;        // roboy_env.py:52
        hold = hold && a[k] >= p.hold_lo && a[k] <= p.hold_hi;  // simulation_client.py:38
    }
    const float g0 = s.g0, g1 = s.g1, g2 = s.g2;
    const uint32_t sf = s.sf;
    float q0, q1, q2, qd0, qd1, qd2, reward;
    bool reached, violation;
    if (!hold) {
        const Draw6 d = split6x21(philox_draw(gid, t, kStreamState, p.keys));
        q0 = uniform_in21(d.k[0], p.c.a_lo, p.f.a_span21);
        q1 = uniform_in21(d.k[1], p.c.a_lo, p.f.a_span21);
        q2 = uniform_in21(d.k[2], p.c.a_lo, p.f.a_span21);
        qd0 = uniform_in21(d.k[3], p.c.a_lo, p.f.a_span21);
        qd1 = uniform_in21(d.k[4], p.c.a_lo, p.f.a_span21);
        qd2 = uniform_in21(d.k[5], p.c.a_lo, p.f.a_span21);
        if (FASTDIV) reward_reached_rt<true>(PENALTY, BONUS, q0, q1, q2, qd0, qd1, qd2, s, p.c, p.f, reward, reached, violation);
        else reward_reached_rt<false>(PENALTY, BONUS, q0, q1, q2, qd0, qd1, qd2, s, p.c, p.f, reward, reached, violation);
    } else {
        const HoldOut h = hold_branch(p, env, sf, g0, g1, g2, PENALTY, BONUS);
        q0 = h.q0; q1 = h.q1; q2 = h.q2; qd0 = h.qd0; qd1 = h.qd1; qd2 = h.qd2;
        reward = h.reward;
        reached = h.flags & 1u;
        violation = h.flags & 2u;
        atomicAdd(&s_cnt[2], 1u);
    }
    uint32_t step = sf & ROBOY_STEP_MASK;
    step += step < ROBOY_STEP_MASK;                          // roboy_env.py:60
    const bool done = reached || (int32_t)step > p.max_len;  // :65-66, :72-73
    uint32_t word = step | (sf & ~ROBOY_STEP_MASK);
    // obs = [q, qd, goal], :75-80
    row[0] = q0; row[1] = q1; row[2] = q2; row[3] = qd0; row[4] = qd1; row[5] = qd2;
    row[6] = g0; row[7] = g1; row[8] = g2;
    if (done && live) {
        const uint32_t r = finish_episode(episode_end(p, t, env, step, reached, AUTO_RESET, row, s_cnt));
        word = (r & 0x80000000u) ? word : (r | ROBOY_F_HELD_ZERO64);
        s.g0 = p.goal[env];   // the new goal was stored by finish_episode (same thread)
        s.g1 = p.goal1[env];
        s.g2 = p.goal2[env];
        if (FASTDIV) normalize_goal<true>(s, p.c, p.f);
        else normalize_goal<false>(s, p.c, p.f);
    }
    if (live && (violation || !act_ok)) {
        atomicOr(p.err_flags, (violation ? ROBOY_ERR_REWARD_RANGE : 0u) | (!act_ok ? ROBOY_ERR_ACTION : 0u));
        atomicMin(p.first_bad, (unsigned long long)gid);
        atomicAdd(&s_cnt[3], 1u);
    }
    s.sf = word;
    if (live) {
        p.reward[(size_t)tt * n + env] = reward;
        p.done[(size_t)tt * n + env] = (uint8_t)done;
        sum_reward += reward;
    }
}

// Episode statistics of a launch: one set of atomics per CTA (as in step_kernel); call with all threads.
// P: StepParams (the MSJ kernels) or GStepParams (the generic rollout).
template <class P>
__device__ __forceinline__ void policy_stats_tail(const P &p, uint32_t T, uint64_t t_first, float sum_reward,
                                                  double *s_red, unsigned int *s_cnt) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const double w_reward = warp_sum_d((double)sum_reward);
    if (lane == 0) s_red[warp] = w_reward;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
        for (int w = 0; w < n_warps; ++w) r += s_red[w];
        const double done = (double)s_cnt[0], succ = (double)s_cnt[1];
        const double steps = blockIdx.x == 0 ? (double)(p.e_end - p.e_begin) * (double)T : 0.0;
        const double v[ROBOY_STAT_COUNT] = {steps, done, succ, done - succ, r, (double)*eplen_counter(s_cnt),
                                            (double)s_cnt[2], (double)s_cnt[3]};
#pragma unroll
        for (int k = 0; k < ROBOY_STAT_COUNT; ++k)
            if (v[k] != 0.0) atomicAdd(p.stats + k, v[k]);
        counter_end(p.cc, t_first);
    }
}

}  // namespace
}  // namespace roboy
