// The float32 MlpPolicy pieces of the generic fused policy kernels, shared by the rollout (roboy_policy_generic.cu) and
// the evaluator (roboy_policy_eval.cu) so that both evaluate the policy mean with the same instructions: given the same
// observation they compute the same bits.
#pragma once
#include <cuda_runtime.h>

#include "../../include/roboy_b200.h"
#include "policy_common.cuh"

namespace roboy {
namespace {

constexpr int kGHid = ROBOY_POLICY_HIDDEN;  // 64

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

__host__ __device__ constexpr int g_stage_stride(int J) { return (3 * J) | 1; }

}  // namespace
}  // namespace roboy
