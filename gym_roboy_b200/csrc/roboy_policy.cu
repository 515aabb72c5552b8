// sm_100a kernel of the closed-loop rollout: the policy INSIDE the env-step kernel.
//
// The reference collects rollouts with stable-baselines' PPO2 runner over a SubprocVecEnv
// (gym_roboy/train_parallel.py:28-35): per step the MlpPolicy (two 64-64 tanh networks, Gaussian
// with a state-independent log-std) runs in the trainer process, the action is clipped to the action
// space and crosses a pipe to every env process, and obs / reward / done come back the same way.
// Here ONE launch runs T such steps for every env: a thread owns E envs, keeps their observation,
// goal and step word in registers across the T steps, evaluates both networks in float32
// (weights in shared memory, FFMA2 = fma.rn.f32x2), draws the Gaussian noise from Philox, clips, and
// runs the same env step as step_kernel (RoboyEnv.step, roboy_env.py:51-70, with the Stub update,
// reward, done test, goal resampling and reset-on-done) on the action it just produced.  Nothing
// is read from HBM per step; what is written is what a PPO update consumes:
// action 32 + logp 4 + value 4 + obs 36 + reward 4 + done 1 = 81 B per env-step.
//
// Unlike the env step this kernel is bound by float32 FMA throughput (10,368 FMA per env-step for
// the two networks, i.e. ~21 kflop against 81 B), not by HBM.  The matrix products are done per
// thread ("one env = one row"), with the weight row broadcast from shared memory as LDS.128 and
// the activations of the previous layer read back from a thread-private shared-memory column, so
// that the 64 accumulators per env stay in registers; E = 2 envs per thread halves the
// shared-memory traffic per FMA (17 LDS per 64 FFMA2), which is what keeps the FMA pipe fed.
//
// The env arithmetic (done mask, observations, rewards) is the step kernel's, instruction for
// instruction: given the actions this kernel stores, T roboy_step calls reproduce its env outputs
// bit for bit (tests/test_gpu_policy_rollout.py).  The policy arithmetic is float32 with FMA and a
// tanh evaluated as 1 - 2/(exp2(2x*log2 e) + 1) on the MUFU unit (absolute error ~3e-7); it agrees
// with the torch float32 MlpPolicy to ~1e-6.
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/roboy_b200.h"
#include "roboy_kernels.cuh"
#include "roboy_policy.cuh"
#include "policy_common.cuh"

namespace roboy {

namespace {

constexpr int kHid = ROBOY_POLICY_HIDDEN;  // 64

// One 9 -> 64 -> 64 -> 8 tanh network (the value network's output layer is zero-padded from 1 to 8
// columns so both networks run the same code).  `row` is the envs' observation rows in the obs stage
// (stride 9), `hs` the thread-private column of the hidden-activation scratch [64][32*E].
template <int E>
__device__ __forceinline__ void mlp_forward(const float *__restrict__ net, const float *__restrict__ row, float *__restrict__ hs,
                                            float2 (&out)[E][4]) {
    float2 acc[E][32];
    load_bias64<E>(net + ROBOY_POLICY_OFF_B1, acc);
    dense64<E>(net + ROBOY_POLICY_OFF_W1, row, kObsDim, 1, 32 * kObsDim, acc);
#pragma unroll
    for (int j2 = 0; j2 < 32; ++j2) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
            hs[(2 * j2) * (32 * E) + 32 * e] = tanh_mufu(acc[e][j2].x);
            hs[(2 * j2 + 1) * (32 * E) + 32 * e] = tanh_mufu(acc[e][j2].y);
        }
    }
    load_bias64<E>(net + ROBOY_POLICY_OFF_B2, acc);
    dense64<E>(net + ROBOY_POLICY_OFF_W2, hs, kHid, 32 * E, 32, acc);
    // output layer fused into the activation of the second: out[e][0..7] += tanh(acc[e][j]) * W3[j][0..7]
    {
        const float4 b0 = reinterpret_cast<const float4 *>(net + ROBOY_POLICY_OFF_B3)[0];
        const float4 b1 = reinterpret_cast<const float4 *>(net + ROBOY_POLICY_OFF_B3)[1];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            out[e][0] = make_float2(b0.x, b0.y);
            out[e][1] = make_float2(b0.z, b0.w);
            out[e][2] = make_float2(b1.x, b1.y);
            out[e][3] = make_float2(b1.z, b1.w);
        }
    }
    const float4 *w3 = reinterpret_cast<const float4 *>(net + ROBOY_POLICY_OFF_W3);
#pragma unroll
    for (int j = 0; j < kHid; ++j) {
        const float4 wa = w3[2 * j], wb = w3[2 * j + 1];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const float t = tanh_mufu((j & 1) ? acc[e][j >> 1].y : acc[e][j >> 1].x);
            const float2 tt = make_float2(t, t);
            out[e][0] = __ffma2_rn(make_float2(wa.x, wa.y), tt, out[e][0]);
            out[e][1] = __ffma2_rn(make_float2(wa.z, wa.w), tt, out[e][1]);
            out[e][2] = __ffma2_rn(make_float2(wb.x, wb.y), tt, out[e][2]);
            out[e][3] = __ffma2_rn(make_float2(wb.z, wb.w), tt, out[e][3]);
        }
    }
}

}  // namespace

template <int E>
__global__ void __launch_bounds__(kPolicyMaxBlock, 1) policy_rollout_kernel(const __grid_constant__ StepParams p,
                                                                             const __grid_constant__ PolicyParams q) {
    const bool FASTDIV = q.fastdiv;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int n_warps = blockDim.x >> 5;
    // shared memory: policy image | per warp: hidden scratch [64][32E], obs stage [32E][9] | counters
    float *img = smem;
    float *hs = smem + ROBOY_POLICY_IMAGE_FLOATS + warp * (kHid * 32 * E) + lane;
    float *stage = smem + ROBOY_POLICY_IMAGE_FLOATS + n_warps * (kHid * 32 * E) + warp * (32 * E * kObsDim);
    double *s_red = reinterpret_cast<double *>(smem + ROBOY_POLICY_IMAGE_FLOATS + n_warps * (kHid * 32 * E + 32 * E * kObsDim));
    unsigned int *s_cnt = reinterpret_cast<unsigned int *>(s_red + n_warps);
    for (int i = threadIdx.x; i < ROBOY_POLICY_IMAGE_FLOATS / 4; i += blockDim.x)
        reinterpret_cast<float4 *>(img)[i] = reinterpret_cast<const float4 *>(q.image)[i];
    if (threadIdx.x < kCntWords) s_cnt[threadIdx.x] = 0;
    __syncthreads();

    const uint64_t t_first = counter_begin(p.cc);
    const uint32_t n_end = (uint32_t)p.e_end;
    const size_t n = (size_t)p.n;
    const uint32_t n_chunks = (n_end + 32 * E - 1) / (32 * E);
    const uint32_t warp_stride = gridDim.x * n_warps;
    const float *vf_net = img + ROBOY_POLICY_OFF_VF, *pi_net = img + ROBOY_POLICY_OFF_PI;
    float sum_reward = 0.0f;

    for (uint32_t chunk = blockIdx.x * n_warps + warp; chunk < n_chunks; chunk += warp_stride) {
        const uint32_t base = chunk * (32 * E);
        const bool full = base + 32 * E <= n_end;
        EnvRegs s[E];
        bool live[E];
        __syncwarp();
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const uint32_t env = base + 32 * e + lane;
            live[e] = env < n_end;
            s[e].g0 = live[e] ? p.goal[env] : 0.f;
            s[e].g1 = live[e] ? p.goal1[env] : 0.f;
            s[e].g2 = live[e] ? p.goal2[env] : 0.f;
            s[e].sf = live[e] ? p.step_flags[env] : 1u;
            if (FASTDIV) normalize_goal<true>(s[e], p.c, p.f);
            else normalize_goal<false>(s[e], p.c, p.f);
            // the observation the rollout starts from: slot 0 of the obs buffer
            float *row = stage + (32 * e + lane) * kObsDim;
#pragma unroll
            for (int k = 0; k < kObsDim; ++k) row[k] = live[e] ? q.obs[(size_t)env * kObsDim + k] : 0.f;
        }

        for (uint32_t tt = 0;; ++tt) {
            // ---- value network on obs[tt] (also the bootstrap value at tt == T) ----
            float2 out[E][4];
            mlp_forward<E>(vf_net, stage + lane * kObsDim, hs, out);
#pragma unroll
            for (int e = 0; e < E; ++e)
                if (live[e]) q.values[(size_t)tt * n + base + 32 * e + lane] = out[e][0].x;
            if (tt == q.T) break;
            // ---- policy network: mean of the Gaussian ----
            mlp_forward<E>(pi_net, stage + lane * kObsDim, hs, out);
            const uint64_t t = t_first + tt;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const float mean[8] = {out[e][0].x, out[e][0].y, out[e][1].x, out[e][1].y,
                                       out[e][2].x, out[e][2].y, out[e][3].x, out[e][3].y};
                sample_and_step(p, q, img + ROBOY_POLICY_OFF_STD, img[ROBOY_POLICY_OFF_LOGNORM], mean, s[e], live[e],
                                base + 32 * e + lane, tt, t, stage + (32 * e + lane) * kObsDim, s_cnt, sum_reward);
            }
            // ---- obs[tt + 1]: the stage now holds the chunk's 32E rows; store them coalesced ----
            __syncwarp();
            float *dst = q.obs + ((size_t)(tt + 1) * n + base) * kObsDim;
            if (full && q.obs_aligned) {
                const float4 *src = reinterpret_cast<const float4 *>(stage);
#pragma unroll
                for (int i = 0; i < (32 * E * kObsDim) / 4 / 32; ++i)
                    reinterpret_cast<float4 *>(dst)[i * 32 + lane] = src[i * 32 + lane];
                if (lane < ((32 * E * kObsDim) / 4) % 32)
                    reinterpret_cast<float4 *>(dst)[((32 * E * kObsDim) / 4 / 32) * 32 + lane] =
                        src[((32 * E * kObsDim) / 4 / 32) * 32 + lane];
            } else {
                const uint32_t rows = full ? 32u * E : n_end - base;
                for (uint32_t i = lane; i < rows * kObsDim; i += 32) dst[i] = stage[i];
            }
            __syncwarp();
        }
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (live[e]) p.step_flags[base + 32 * e + lane] = s[e].sf;
    }

    policy_stats_tail(p, q.T, t_first, sum_reward, s_red, s_cnt);
}

PolicyGeom policy_geometry(uint64_t n_envs, int sm_count, int envs_per_thread) {
    PolicyGeom g;
    const uint64_t resident = (uint64_t)sm_count * (kPolicyMaxBlock / 32) * 32;  // envs with one env per thread
    g.envs_per_thread = envs_per_thread ? envs_per_thread : (n_envs <= resident ? 1 : 2);
    const uint64_t n_chunks = (n_envs + 32 * g.envs_per_thread - 1) / (32 * g.envs_per_thread);
    // spread the warps over the SMs first, then fill the CTAs (up to kPolicyMaxBlock threads, 1 CTA per SM)
    g.grid = (int)(n_chunks < (uint64_t)sm_count ? n_chunks : (uint64_t)sm_count);
    uint64_t wpb = (n_chunks + g.grid - 1) / g.grid;
    if (wpb > kPolicyMaxBlock / 32) wpb = kPolicyMaxBlock / 32;
    g.block = (int)wpb * 32;
    g.smem = (int)(sizeof(float) * (ROBOY_POLICY_IMAGE_FLOATS + wpb * (kHid * 32 * g.envs_per_thread + 32 * g.envs_per_thread * kObsDim)) +
                   sizeof(double) * wpb + sizeof(unsigned int) * kCntWords);
    return g;
}

cudaError_t launch_policy_rollout(const StepParams &p, const PolicyParams &q, bool penalty, bool bonus, bool auto_reset,
                                  bool fastdiv, int sm_count, int envs_per_thread, cudaStream_t stream) {
    if (p.e_end <= p.e_begin) return cudaSuccess;
    PolicyParams qq = q;
    qq.penalty = penalty;
    qq.bonus = bonus;
    qq.auto_reset = auto_reset;
    qq.fastdiv = fastdiv;
    const PolicyGeom g = policy_geometry(p.e_end, sm_count, envs_per_thread);
    void (*fn)(const StepParams, const PolicyParams) =
        g.envs_per_thread == 1 ? policy_rollout_kernel<1> : policy_rollout_kernel<2>;
    cudaError_t err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem);
    if (err != cudaSuccess) return err;
    fn<<<g.grid, g.block, g.smem, stream>>>(p, qq);
    return cudaGetLastError();
}

}  // namespace roboy
