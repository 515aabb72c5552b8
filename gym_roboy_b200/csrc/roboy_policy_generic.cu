// sm_100a kernel of the closed-loop rollout for every robot the generic kernels take (J = 1..15 joints, A = 1..64
// tendons, one bound per component): the float32 policy inside the generic env step.
//
// The shape is the MSJ kernel's (roboy_policy.cu): one launch runs T steps of [MlpPolicy forward -> Gaussian sample ->
// clip -> RoboyEnv.step] for every env; a thread owns one env and keeps its observation row (shared memory), goal and
// step word on chip for the T steps; both networks run in float32 FFMA2 with the weights broadcast from shared memory
// (dense64, policy_common.cuh) and the hidden activations in a thread-private shared-memory column.  The frame around
// the loop body -- shared memory, state draw, action tests, the observation stage's rows -- is policy_generic.cuh's,
// shared with the evaluator (roboy_policy_eval.cu).  What changes with the robot:
//   * the first layer has D = 3J inputs;
//   * the output layer has A8 = 8 * ceil(A / 8) columns.  Its 64 inputs tanh(h2) are written back into the hidden column
//     and it runs in groups of 8 columns, each sampled, stored, clipped and action-tested before the next, so no more
//     than 8 outputs are ever in registers.  Every output is b3 + sum_j tanh(h2_j) * W3[j] with j ascending, the
//     operation order of the MSJ kernel: for MSJ the two give the same bits;
//   * normal k (k < A) is Box-Muller on word pair (k mod 4) / 2 of Philox block (stream 4, sub = k / 4) keyed by the
//     noise seed, the first or second value by k mod 2 -- for A = 8 exactly the MSJ kernel's draws;
//   * the env step is generic_env_step (generic_env.cuh), the per-env body of generic_step_kernel: given the clipped
//     actions this kernel stores, T roboy_step calls reproduce its env outputs bit for bit.
// Per env-step the kernel writes actions 4A + logp 4 + value 4 + obs 12J + reward 4 + done 1 = 4A + 12J + 13 bytes and
// evaluates 64 * (2D + 128 + 8 + A8) FMAs.
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/roboy_b200.h"
#include "generic_env.cuh"
#include "policy_common.cuh"
#include "policy_generic.cuh"
#include "roboy_generic.cuh"
#include "roboy_policy.cuh"

namespace roboy {

namespace {

constexpr int kGPolicySmemBudget = 227 * 1024;

}  // namespace

template <int JM>
__global__ void __launch_bounds__(kGPolicyMaxBlock, 1) generic_policy_rollout_kernel(const __grid_constant__ GStepParams p,
                                                                                      const __grid_constant__ GPolicyParams q) {
    constexpr int J = JM, D = 3 * J, S = g_stage_stride(J);
    const RobotSpec &r = p.r;
    const int A = r.A, A8 = (A + 7) & ~7;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int n_warps = blockDim.x >> 5;
    const GPolicySmem m = g_policy_smem<J>(smem, q.off[ROBOY_POLICY_LAYOUT_FLOATS]);   // the whole image
    g_policy_smem_fill(m, q.image, q.off[ROBOY_POLICY_LAYOUT_FLOATS]);
    const float *img = m.image;

    const uint64_t t_first = counter_begin(p.cc);
    const uint32_t n_end = (uint32_t)p.e_end, n_envs = (uint32_t)p.n;
    const size_t n = (size_t)p.n;
    const uint32_t n_chunks = (n_end + 31) / 32;
    const uint32_t warp_stride = gridDim.x * n_warps;
    const float *vf_net = img + q.off[ROBOY_POLICY_LAYOUT_VF], *pi_net = img + q.off[ROBOY_POLICY_LAYOUT_PI];
    const float *sd = img + q.off[ROBOY_POLICY_LAYOUT_STD];
    const float lognorm = img[q.off[ROBOY_POLICY_LAYOUT_LOGNORM]];
    const bool fastdiv = r.fastdiv != 0;   // the step kernel's choice (launch_generic_step)
    const bool act_vec = (A & 3) == 0;   // rows of actions / noise are 16-byte aligned (the buffers are)
    float *row = m.stage + lane * S;
    float sum_reward = 0.0f;

    for (uint32_t chunk = blockIdx.x * n_warps + warp; chunk < n_chunks; chunk += warp_stride) {
        const uint32_t base = chunk * 32;
        const bool full = base + 32 <= n_end;
        const uint32_t env = base + lane;
        const bool live = env < n_end;
        const uint64_t gid = p.gid_base + env;
        float g[JM];
        uint32_t sf = live ? p.step_flags[env] : 0u;
#pragma unroll
        for (int k = 0; k < JM; ++k) g[k] = live ? p.goal[(size_t)k * n + env] : 0.f;
        __syncwarp();
        // the observation the rollout starts from: slot 0 of the obs buffer
#pragma unroll
        for (int k = 0; k < D; ++k) row[k] = live ? q.obs[(size_t)env * D + k] : 0.f;

        for (uint32_t tt = 0;; ++tt) {
            // ---- value network on obs[tt] (also the bootstrap value at tt == T) ----
            mlp_hidden<D>(vf_net, q.off, row, m.hs);
            {
                float v[8];
                mlp_out8(vf_net + q.off[ROBOY_POLICY_LAYOUT_W3], vf_net + q.off[ROBOY_POLICY_LAYOUT_VF_B3], 8, 0, m.hs, v);
                if (live) q.values[(size_t)tt * n + env] = v[0];
            }
            if (tt == q.T) break;
            // ---- policy network, 8 output columns at a time: mean -> a = mean + std * z -> clip -> action tests ----
            mlp_hidden<D>(pi_net, q.off, row, m.hs);
            const uint64_t t = t_first + tt;
            const size_t slot = (size_t)tt * n + env;
            float zz = 0.0f;
            bool act_ok = true, hold = live;
            for (int c = 0; c < A8 / 8; ++c) {
                float mean[8];
                mlp_out8(pi_net + q.off[ROBOY_POLICY_LAYOUT_W3], pi_net + q.off[ROBOY_POLICY_LAYOUT_PI_B3], A8, c, m.hs, mean);
                const uint4 r0 = philox_draw(gid, t, kStreamNoise, q.noise_keys, 2 * c);
                const uint4 r1 = philox_draw(gid, t, kStreamNoise, q.noise_keys, 2 * c + 1);
                const float2 z01 = box_muller(r0.x, r0.y), z23 = box_muller(r0.z, r0.w);
                const float2 z45 = box_muller(r1.x, r1.y), z67 = box_muller(r1.z, r1.w);
                const float z[8] = {z01.x, z01.y, z23.x, z23.y, z45.x, z45.y, z67.x, z67.y};
                float u[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int k = 8 * c + i;
                    u[i] = fmaf(sd[k], z[i], mean[i]);
                    if (k < A) {
                        zz = fmaf(z[i], z[i], zz);
                        g_clip_test(r, k, u[i], act_ok, hold);
                    }
                }
                if (live) {
                    float *ap = q.actions + slot * A + 8 * c;
                    float *np = q.noise ? q.noise + slot * A + 8 * c : nullptr;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        if (act_vec) {
                            if (8 * c + 4 * h < A) {
                                reinterpret_cast<float4 *>(ap)[h] = make_float4(u[4 * h], u[4 * h + 1], u[4 * h + 2], u[4 * h + 3]);
                                if (np) reinterpret_cast<float4 *>(np)[h] = make_float4(z[4 * h], z[4 * h + 1], z[4 * h + 2], z[4 * h + 3]);
                            }
                        } else {
#pragma unroll
                            for (int i = 4 * h; i < 4 * h + 4; ++i)
                                if (8 * c + i < A) {
                                    ap[i] = u[i];
                                    if (np) np[i] = z[i];
                                }
                        }
                    }
                }
            }
            if (live) q.logp[slot] = fmaf(-0.5f, zz, lognorm);

            // ---- RoboyEnv.step on the clipped action: the generic step kernel's per-env body ----
            float qs[JM], qds[JM];
            g_draw_step_state<JM>(r, p.keys, live, gid, t, qs, qds);
            const bool done = generic_env_step<JM>(p, fastdiv, live, hold, act_ok, qs, qds, g, sf, gid, t, env, n_envs, m.s_cnt,
                                                   eplen_counter(m.s_cnt), sum_reward, [&](uint32_t word, float rf, bool d, bool) {
                                                       sf = word;
                                                       p.reward[slot] = rf;
                                                       p.done[slot] = (uint8_t)d;
                                                   });
            // ---- obs[tt + 1] = [q, qd, goal] into the stage, then the chunk's 32 rows out coalesced ----
            g_stage_obs<JM>(row, qs, qds, g);
            if (done) {   // the goal of the next step (done without auto-reset: the observation above shows the old one)
#pragma unroll
                for (int k = 0; k < JM; ++k) g[k] = p.goal[(size_t)k * n + env];
            }
            __syncwarp();
            float *dst = q.obs + ((size_t)(tt + 1) * n + base) * D;
            if (full && q.obs_aligned) {   // 32 rows = 8D float4s
                float4 *dst4 = reinterpret_cast<float4 *>(dst);
                for (int i4 = lane; i4 < 8 * D; i4 += 32) {
                    float v[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const int i = 4 * i4 + c;
                        v[c] = m.stage[(i / D) * S + i % D];
                    }
                    dst4[i4] = make_float4(v[0], v[1], v[2], v[3]);
                }
            } else {
                const uint32_t rows = full ? 32u : n_end - base;
                for (uint32_t i = lane; i < rows * D; i += 32) dst[i] = m.stage[(i / D) * S + i % D];
            }
            __syncwarp();
        }
        if (live) p.step_flags[env] = sf;
    }

    policy_stats_tail(p, q.T, t_first, sum_reward, m.s_red, m.s_cnt);
}

PolicyGeom generic_policy_geometry(int J, uint32_t image_floats, uint64_t n_envs, int sm_count) {
    PolicyGeom g;
    g.envs_per_thread = 1;
    const int fixed = g_policy_smem_bytes(J, image_floats, 0);
    const int per_warp = g_policy_smem_bytes(J, image_floats, 1) - fixed;
    int max_warps = (kGPolicySmemBudget - fixed) / per_warp;
    if (max_warps > kGPolicyMaxBlock / 32) max_warps = kGPolicyMaxBlock / 32;
    const uint64_t n_chunks = (n_envs + 31) / 32;
    // spread the warps over the SMs first, then fill the CTAs (one CTA per SM)
    g.grid = (int)(n_chunks < (uint64_t)sm_count ? n_chunks : (uint64_t)sm_count);
    uint64_t wpb = (n_chunks + g.grid - 1) / g.grid;
    if (wpb > (uint64_t)max_warps) wpb = (uint64_t)max_warps;
    g.block = (int)wpb * 32;
    g.smem = g_policy_smem_bytes(J, image_floats, (int)wpb);
    return g;
}

cudaError_t launch_generic_policy_rollout(const GStepParams &p, const GPolicyParams &q, int sm_count, cudaStream_t stream) {
    if (p.e_end <= p.e_begin) return cudaSuccess;
    switch (p.r.J) {
#define ROBOY_GPOLICY_CASE(JJ) \
        case JJ: return launch_generic_policy(generic_policy_rollout_kernel<JJ>, p, q, q.off[ROBOY_POLICY_LAYOUT_FLOATS], sm_count, stream);
        ROBOY_GENERIC_JOINT_COUNTS(ROBOY_GPOLICY_CASE)
#undef ROBOY_GPOLICY_CASE
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace roboy
