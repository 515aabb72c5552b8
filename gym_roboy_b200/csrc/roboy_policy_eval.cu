// sm_100a kernel of the deterministic policy evaluation for every robot the generic kernels take (J = 1..15 joints,
// A = 1..64 tendons), MSJ-shaped ones included: what stable-baselines' evaluate_policy(deterministic=True) measures, in
// one launch.
//
// The loop is the generic rollout's (roboy_policy_generic.cu) with the action clip(mean(obs), -1, 1) -- the rollout's
// action under std 0 -- and three differences:
//   * no value network, no sampling and no per-step store: only the policy net of the image is staged in shared memory;
//   * each thread keeps its env's episode bookkeeping in registers (the float64 return of the episode in progress,
//     whether that episode counts, how many records it wrote, how many counted episodes finished) and writes a record
//     [return, length, reached] when a counted episode ends; unfilled records are set to [NaN, 0, 0] at the end;
//   * the observation after the last step is stored once, coalesced through the warp's stage.
// The frame around the loop body and the policy mean are the rollout's (policy_generic.cuh) and the env step is
// generic_env_step (generic_env.cuh): the env outputs are those of T roboy_step calls on the clipped means, bit for bit.
// An episode counts when it starts inside the launch: at the first step for an env whose step counter is 1, and at the
// step after every done (auto-reset on).  Per env-step the kernel evaluates 64 * (D + 64 + A8) FMAs and writes nothing
// but the records of finished episodes and the goals drawn on done.
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/roboy_b200.h"
#include "generic_env.cuh"
#include "policy_common.cuh"
#include "policy_generic.cuh"
#include "roboy_generic.cuh"
#include "roboy_policy.cuh"

namespace roboy {

template <int JM>
__global__ void __launch_bounds__(kGPolicyMaxBlock, 1) generic_policy_evaluate_kernel(const __grid_constant__ GStepParams p,
                                                                                      const __grid_constant__ GEvalParams q) {
    constexpr int J = JM, D = 3 * J, S = g_stage_stride(J);
    const RobotSpec &r = p.r;
    const int A = r.A, A8 = (A + 7) & ~7;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int n_warps = blockDim.x >> 5;
    // the policy net only; launch_generic_policy_evaluate sizes shared memory from the same difference
    const uint32_t net_floats = q.off[ROBOY_POLICY_LAYOUT_STD] - q.off[ROBOY_POLICY_LAYOUT_PI];
    const GPolicySmem m = g_policy_smem<J>(smem, net_floats);
    g_policy_smem_fill(m, q.image + q.off[ROBOY_POLICY_LAYOUT_PI], net_floats);
    const float *pi_net = m.image;

    const uint64_t t_first = counter_begin(p.cc);
    const uint32_t n_end = (uint32_t)p.e_end, n_envs = (uint32_t)p.n;
    const size_t n = (size_t)p.n;
    const uint32_t n_chunks = (n_end + 31) / 32;
    const uint32_t warp_stride = gridDim.x * n_warps;
    const bool fastdiv = r.fastdiv != 0;   // the step kernel's choice (launch_generic_step)
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
#pragma unroll
        for (int k = 0; k < D; ++k) row[k] = live ? q.obs[(size_t)env * D + k] : 0.f;

        // the episode in progress counts if it starts inside the launch: step counter at its reset value
        bool counting = (sf & ROBOY_STEP_MASK) == 1u;
        double ret = 0.0;
        uint32_t n_rec = 0, n_done = 0;

        for (uint32_t tt = 0; tt < q.T; ++tt) {
            // ---- policy network, 8 output columns at a time: mean -> clip -> action tests ----
            mlp_hidden<D>(pi_net, q.off, row, m.hs);
            const uint64_t t = t_first + tt;
            bool act_ok = true, hold = live;
            for (int c = 0; c < A8 / 8; ++c) {
                float mean[8];
                mlp_out8(pi_net + q.off[ROBOY_POLICY_LAYOUT_W3], pi_net + q.off[ROBOY_POLICY_LAYOUT_PI_B3], A8, c, m.hs, mean);
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (8 * c + i < A) g_clip_test(r, 8 * c + i, mean[i], act_ok, hold);
            }

            // ---- RoboyEnv.step on the clipped mean: the generic step kernel's per-env body ----
            float qs[JM], qds[JM];
            g_draw_step_state<JM>(r, p.keys, live, gid, t, qs, qds);
            const uint32_t step_in = sf & ROBOY_STEP_MASK;
            const uint32_t ep_len = step_in + (step_in < ROBOY_STEP_MASK) - 1u;   // step_num - 1 at a done (:60)
            generic_env_step<JM>(p, fastdiv, live, hold, act_ok, qs, qds, g, sf, gid, t, env, n_envs, m.s_cnt,
                                 eplen_counter(m.s_cnt), sum_reward, [&](uint32_t word, float rf, bool d, bool reached) {
                                     sf = word;
                                     if (counting) {
                                         ret = __dadd_rn(ret, (double)rf);
                                         if (d) {
                                             if (n_rec < q.episodes) {
                                                 const uint64_t slot = (uint64_t)n_rec * n + env;
                                                 q.returns[slot] = ret;
                                                 q.lengths[slot] = ep_len;
                                                 q.reached[slot] = (uint8_t)reached;
                                                 ++n_rec;
                                             }
                                             ++n_done;
                                         }
                                     }
                                     if (d) {   // auto-reset: the next episode starts at the next step
                                         counting = true;
                                         ret = 0.0;
                                     }
                                 });
            // ---- the next observation [q, qd, goal] (after a done, g already holds the reset()'s goal) ----
            g_stage_obs<JM>(row, qs, qds, g);
        }
        if (live) {
            p.step_flags[env] = sf;
            q.completed[env] = n_done;
            for (uint32_t k = n_rec; k < q.episodes; ++k) {
                const uint64_t slot = (uint64_t)k * n + env;
                q.returns[slot] = __longlong_as_double(0x7ff8000000000000ll);   // NaN: no such episode
                q.lengths[slot] = 0u;
                q.reached[slot] = 0u;
            }
        }
        // ---- the final observation: the chunk's 32 rows out coalesced ----
        __syncwarp();
        float *dst = q.obs + (size_t)base * D;
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

    policy_stats_tail(p, q.T, t_first, sum_reward, m.s_red, m.s_cnt);
}

cudaError_t launch_generic_policy_evaluate(const GStepParams &p, const GEvalParams &q, int sm_count, cudaStream_t stream) {
    if (p.e_end <= p.e_begin) return cudaSuccess;
    switch (p.r.J) {
#define ROBOY_GEVAL_CASE(JJ) \
        case JJ: return launch_generic_policy(generic_policy_evaluate_kernel<JJ>, p, q, \
                                              q.off[ROBOY_POLICY_LAYOUT_STD] - q.off[ROBOY_POLICY_LAYOUT_PI], sm_count, stream);
        ROBOY_GENERIC_JOINT_COUNTS(ROBOY_GEVAL_CASE)
#undef ROBOY_GEVAL_CASE
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace roboy
