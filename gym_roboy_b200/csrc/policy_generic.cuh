// The frame of the generic fused policy kernels, shared by the rollout (roboy_policy_generic.cu) and the evaluator
// (roboy_policy_eval.cu): the shared-memory layout, the sampled state and the action tests of one env-step, and the row
// an env writes into the observation stage.  Both evaluate the policy mean with the same float32 MlpPolicy instructions
// here: given the same observation they compute the same bits.
//
// A warp owns a chunk of 32 envs at a time, a thread one env.  Each env's observation row sits in the warp's stage
// [32][S], S = 3J rounded up to odd, so that the 32 lanes' reads of one input fall in 32 different banks; the warp copies
// the stage out to [n][3J] coalesced, skipping the pad column.  The start of a chunk and that copy-out are written out
// in each kernel: as shared functions they changed both kernels' code, and the evaluator ran 0.5 % slower on
// 15 joints / 64 tendons at 1,048,576 envs (one B200, 1,000 W power limit).
#pragma once
#include <cuda_runtime.h>

#include "../../include/roboy_b200.h"
#include "generic_env.cuh"
#include "policy_common.cuh"
#include "roboy_generic.cuh"
#include "roboy_policy.cuh"

namespace roboy {
namespace {

constexpr int kGHid = ROBOY_POLICY_HIDDEN;  // 64

__host__ __device__ constexpr int g_stage_stride(int J) { return (3 * J) | 1; }

// The dynamic shared memory of a generic policy kernel with n_warps warps per CTA:
//   staged image [staged_floats] | hidden columns [n_warps][64][32] | observation stages [n_warps][32][S] |
//   reduction double[n_warps] | counters [kCntWords]
// staged_floats is a multiple of 4 (16-byte image rows), so the reduction is 8-byte aligned.  g_policy_smem carves it.
__host__ __device__ constexpr int g_policy_smem_bytes(int J, uint32_t staged_floats, int n_warps) {
    return (int)sizeof(float) * ((int)staged_floats + n_warps * (kGHid * 32 + 32 * g_stage_stride(J))) +
           (int)sizeof(double) * n_warps + (int)sizeof(unsigned int) * kCntWords;
}

// This thread's pieces of that layout
struct GPolicySmem {
    float *image;          // the staged image [staged_floats]
    float *hs;             // the thread's hidden column: hs[j * 32], j = 0..63
    float *stage;          // the warp's observation stage [32][S]
    double *s_red;         // [n_warps]
    unsigned int *s_cnt;   // [kCntWords]
};

template <int J>
__device__ __forceinline__ GPolicySmem g_policy_smem(float *smem, uint32_t staged_floats) {
    constexpr int S = g_stage_stride(J);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    GPolicySmem m;
    m.image = smem;
    m.hs = smem + staged_floats + warp * (kGHid * 32) + lane;
    m.stage = smem + staged_floats + n_warps * (kGHid * 32) + warp * (32 * S);
    m.s_red = reinterpret_cast<double *>(smem + staged_floats + n_warps * (kGHid * 32 + 32 * S));
    m.s_cnt = reinterpret_cast<unsigned int *>(m.s_red + n_warps);
    return m;
}

// The staged_floats floats of the image at src into m.image, the counters zeroed.  Call with all threads, after
// g_policy_smem (src read before the carve changes the kernels' code).
__device__ __forceinline__ void g_policy_smem_fill(const GPolicySmem &m, const float *src, uint32_t staged_floats) {
    for (uint32_t i = threadIdx.x; i < staged_floats / 4; i += blockDim.x)
        reinterpret_cast<float4 *>(m.image)[i] = reinterpret_cast<const float4 *>(src)[i];
    if (threadIdx.x < kCntWords) m.s_cnt[threadIdx.x] = 0;
    __syncthreads();
}

// The state the Stub draws for env-step t (roboy_robot.py:35-39), as generic_step_kernel draws it; zeros on a dead lane
template <int JM>
__device__ __forceinline__ void g_draw_step_state(const RobotSpec &r, const PhiloxKeys &keys, bool live, uint64_t gid,
                                                  uint64_t t, float (&qs)[JM], float (&qds)[JM]) {
#pragma unroll
    for (int k = 0; k < JM; ++k) qs[k] = qds[k] = 0.0f;
    if (live) {
        DrawCursor cur;
        cur.block = 0xffffffffu;
#pragma unroll
        for (int k = 0; k < JM; ++k) qs[k] = g_draw_value(r, keys, gid, t, cur, k, k);
#pragma unroll
        for (int k = 0; k < JM; ++k) qds[k] = g_draw_value(r, keys, gid, t, cur, JM + k, k);
    }
}

// Action component k: u clipped to [-1, 1] as PPO2's runner does before env.step, then the range assert and the hold
// test of that component
__device__ __forceinline__ void g_clip_test(const RobotSpec &r, int k, float u, bool &act_ok, bool &hold) {
    const float cl = fminf(fmaxf(u, -1.0f), 1.0f);
    const float a = (u != u) ? u : cl;   // a NaN stays a NaN (and fails the assert)
    act_ok = act_ok && (a >= -1.0f && a <= 1.0f);                      // roboy_env.py:52
    hold = hold && (a >= r.hold_lo[k] && a <= r.hold_hi[k]);           // simulation_client.py:38
}

// The observation [q, qd, goal] (roboy_env.py:75-80) into the env's stage row
template <int JM>
__device__ __forceinline__ void g_stage_obs(float *row, const float (&qs)[JM], const float (&qds)[JM], const float (&g)[JM]) {
#pragma unroll
    for (int k = 0; k < JM; ++k) {
        row[k] = qs[k];
        row[JM + k] = qds[k];
        row[2 * JM + k] = g[k];
    }
}

// tanh(h2) of one network into the thread's hidden column hs[j * 32] (j = 0..63); `row` is the env's observation row
template <int D>
__device__ __forceinline__ void mlp_hidden(const float *__restrict__ net, const uint32_t (&off)[ROBOY_POLICY_LAYOUT_WORDS],
                                           const float *__restrict__ row, float *__restrict__ hs) {
    float2 acc[1][32];
    load_bias64<1>(net + off[ROBOY_POLICY_LAYOUT_B1], acc);
    dense64<1>(net + off[ROBOY_POLICY_LAYOUT_W1], row, D, 1, 0, acc);
#pragma unroll
    for (int j2 = 0; j2 < 32; ++j2) {
        hs[(2 * j2) * 32] = tanh_mufu(acc[0][j2].x);
        hs[(2 * j2 + 1) * 32] = tanh_mufu(acc[0][j2].y);
    }
    load_bias64<1>(net + off[ROBOY_POLICY_LAYOUT_B2], acc);
    dense64<1>(net + off[ROBOY_POLICY_LAYOUT_W2], hs, kGHid, 32, 0, acc);
#pragma unroll
    for (int j2 = 0; j2 < 32; ++j2) {
        hs[(2 * j2) * 32] = tanh_mufu(acc[0][j2].x);
        hs[(2 * j2 + 1) * 32] = tanh_mufu(acc[0][j2].y);
    }
}

// Output columns 8c .. 8c + 7 of the last layer: b3 + sum_j tanh(h2_j) * W3[j] (W3 is [64][W], b3 [W])
__device__ __forceinline__ void mlp_out8(const float *__restrict__ w3, const float *__restrict__ b3, int W, int c,
                                         const float *__restrict__ hs, float (&out)[8]) {
    const float4 b0 = reinterpret_cast<const float4 *>(b3 + 8 * c)[0];
    const float4 b1 = reinterpret_cast<const float4 *>(b3 + 8 * c)[1];
    float2 o[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y), make_float2(b1.z, b1.w)};
    const float *w = w3 + 8 * c;
#pragma unroll 8
    for (int j = 0; j < kGHid; ++j) {
        const float4 wa = reinterpret_cast<const float4 *>(w + j * W)[0], wb = reinterpret_cast<const float4 *>(w + j * W)[1];
        const float t = hs[j * 32];
        const float2 tt = make_float2(t, t);
        o[0] = __ffma2_rn(make_float2(wa.x, wa.y), tt, o[0]);
        o[1] = __ffma2_rn(make_float2(wa.z, wa.w), tt, o[1]);
        o[2] = __ffma2_rn(make_float2(wb.x, wb.y), tt, o[2]);
        o[3] = __ffma2_rn(make_float2(wb.z, wb.w), tt, o[3]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        out[2 * k] = o[k].x;
        out[2 * k + 1] = o[k].y;
    }
}

// One launch of a generic policy kernel over p's envs with staged_floats of the image in shared memory
template <class Q>
cudaError_t launch_generic_policy(void (*fn)(const GStepParams, const Q), const GStepParams &p, const Q &q,
                                  uint32_t staged_floats, int sm_count, cudaStream_t stream) {
    const PolicyGeom g = generic_policy_geometry(p.r.J, staged_floats, p.e_end, sm_count);
    cudaError_t err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem);
    if (err != cudaSuccess) return err;
    fn<<<g.grid, g.block, g.smem, stream>>>(p, q);
    return cudaGetLastError();
}

}  // namespace
}  // namespace roboy
