// sm_100a kernel of the closed-loop rollout with the policy's matrix products on the 5th-generation
// tensor cores (tcgen05.mma, kind::f16, float32 accumulators in tensor memory).
//
// Same contract as policy_rollout_kernel (roboy_policy.cu): T steps of [MlpPolicy forward -> Gaussian
// sample -> clip -> RoboyEnv.step] per env in ONE launch (train_parallel.py:28-35 is the loop it
// replaces), env state in registers, env outputs bit-identical to T roboy_step calls on the stored
// actions.  What differs is where the 10,368 multiply-adds per env-step of the two 9-64-64-{8,1} networks run:
//
//   * a CTA holds up to four TILES of 128 envs; thread i of a tile owns env i = row i of every matrix
//     = lane i of the tile's 128 tensor-memory columns (48 for the activations A and the input block, packed
//     two float16 per column, 64 for the float32 accumulator D);
//   * per layer the tile's threads write their activation row into TMEM (tcgen05.st), one thread issues
//     K/16 tcgen05.mma (M = 128 envs, N = 64 / 16 outputs, K = 16 per instruction; A from TMEM, the weight
//     matrix B from shared memory in the canonical K-major core-matrix layout, no swizzle) and commits
//     them to the tile's mbarrier; every thread then reads its row of D back (tcgen05.ld) and applies
//     tanh (MUFU.TANH) and packs two results into one float16 pair (F2FP) -- which IS the next layer's A.
//     Biases ride in the product: A carries a constant 1 in an extra K column and W the bias in the
//     matching column, so the activation math is three instructions per two outputs;
//   * four tiles (16 warps) per SM overlap one tile's MMA round trips with the others' activation math.  (A
//     variant in which each group of 128 threads ping-pongs TWO tiles, template parameter U = 2, measured 35 %
//     slower: with the same four tiles in flight it has half the warps to hide TMEM / MUFU latency behind.)
//     Small populations (at most two tiles per SM) run the MERGED form instead: both networks of a tile advance
//     together, three round trips per step instead of six (+11 % at 4,096 envs).
//
// Arithmetic, two modes (template parameter EXACT):
//   fast   float16 operands (10-bit mantissa, the precision of TF32; every operand here is far inside float16's
//          range), float32 accumulation, tanh.approx: action means and values agree with the float32 policy to ~1e-3;
//   exact  every operand split x = hi + lo into two float16 (22 mantissa bits), each product accumulated in float32 as
//          A_hi W_hi + A_hi W_lo + A_lo W_hi (three MMA groups into the same accumulator), and the float32 kernel's
//          tanh (ex2 + rcp): ~1e-6, the accuracy of torch's own float32 forward, at 2.8x the float32 FFMA2 kernel.
// Tensor cores are used HERE because this IS a dense contraction; the env step itself has none and stays off them.
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/roboy_b200.h"
#include "policy_common.cuh"
#include "roboy_kernels.cuh"
#include "roboy_policy.cuh"

namespace roboy {

namespace {

constexpr int kTileEnvs = 128;      // rows of one MMA = TMEM lanes
// TMEM columns of one tile (float16 pairs for A, float32 for D), 128 per tile in both modes -> four tiles per SM:
//   fast : activations [0,32) | constant-1 block [32,40) | input block [40,48) | D [64,128)
//          (biases ride in the product: the constant-1 block multiplies the bias column of W2 / W3)
//   exact: HIGH halves of the activations [0,32) | LOW halves [32,64) | D [64,128); the input block is written over the
//          first 8 columns of each half before every network's first layer, and the biases of the 64-input layers
//          are added in float32 by the epilogue (no room for a constant-1 block)
template <bool EXACT>
struct Cols {
    static constexpr int A = 0;
    static constexpr int Ones = 32;                      // fast only
    static constexpr int ALo = 32;                       // exact only
    static constexpr int In = EXACT ? 0 : 40;
    static constexpr int InLo = 32;                      // exact only
    static constexpr int D = 64;
    static constexpr int Tile = 128;
    static constexpr int KHid = EXACT ? 64 : ROBOY_TC_K_HIDDEN;   // K the 64-input layers' MMAs run over
};
// merged (fast arithmetic, small populations): both networks advance together, one MMA round trip per layer instead of
// two -- activations of the value net [0,32) | of the policy net [32,64) | constant-1 block [64,72) | input block
// [72,80) | D of the value net [128,192) | D of the policy net [192,256): 256 columns per tile, two tiles per SM
struct ColsMerged {
    static constexpr int AVf = 0, APi = 32, Ones = 64, In = 72, DVf = 128, DPi = 192, Tile = 256, MaxGroups = 2;
};
constexpr int kKHid = ROBOY_TC_K_HIDDEN;  // 80: K of the 64-input layers including the bias column block

__device__ __forceinline__ uint32_t smem_u32(const void *ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }

// Shared-memory matrix descriptor, K-major, SWIZZLE_NONE: 8-row x 16-byte core matrices; LBO = byte
// distance between the two core matrices one MMA reads along K, SBO = between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}

// Instruction descriptor: D = F32 (bits 4-5 = 1), A = B = F16 (bits 7-9, 10-12 = 0), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t idesc_f16(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileEnvs >> 4) << 24);
}

__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void mma_commit(uint32_t mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(mbar) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    uint32_t ok = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\tselp.u32 %0, 1, 0, P;\n\t}"
            : "=r"(ok) : "r"(mbar), "r"(parity) : "memory");
        if (ok) break;
        if (clock64() - t0 > 20000000000ll) __trap();  // ~10 s: a lost arrive must not hang the GPU for good
    }
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
          "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
        : "r"(taddr) : "memory");
}

// tcgen05.wait::ld; the loaded registers are threaded through as operands so that no use of them can be
// scheduled ahead of the wait.
__device__ __forceinline__ void tmem_ld_wait16(float (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]),
                   "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
                 :: "memory");
}

template <int N>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&v)[N]);
template <>
__device__ __forceinline__ void tmem_st<8>(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

// two float32 -> packed float16 pair: `lo` in bits 15..0 (the lower K index), `hi` in bits 31..16
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// (tanh.approx.f16x2 is two MUFU.TANH.F16 plus a PRMT in SASS -- no cheaper than two float32 MUFU.TANH,
// and it rounds the argument to float16 first)
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

struct TileCtx {
    uint32_t tmem_a;           // first column of the tile as this warp addresses it: lane quadrant in bits 31..16
    uint32_t mma_a, mma_d;     // first column of the tile / of its accumulator as the issuing thread addresses them (lane 0)
    uint32_t mbar;             // shared-memory address of the tile's mbarrier
    uint32_t parity;
    int bar_id;                // named barrier of the tile's 128 threads
    bool issuer;
};

// One layer's matrix product for a tile, D[128][N] = A[128][K] * W[N][K]^T, split in two so that the threads
// can work on their other tile while it runs.  issue: every thread has written its row of A; the group's
// threads meet, one of them issues the MMAs and commits them to the tile's mbarrier.  wait: D is readable.
// EXACT: every operand is split x = hi + lo with hi = float16(x), lo = float16(x - hi) (22 mantissa bits together), and
// the product is accumulated as A_hi W_hi + A_hi W_lo + A_lo W_hi in float32 -- float32-level accuracy from float16 MMAs.
// a_col / lo_col: first TMEM column of the (high / low) A block.
// K: the K range the MMAs cover; K_LAYOUT: K of W's layout in shared memory (its 8-row groups are K_LAYOUT * 16 bytes apart).
template <int K, int K_LAYOUT, int N, bool EXACT>
__device__ __forceinline__ void gemm_issue(const TileCtx &c, uint32_t a_col, uint32_t lo_col, uint32_t w_saddr) {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.sync %0, 128;" :: "r"(c.bar_id) : "memory");
    if (c.issuer) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // one MMA consumes K = 16: 8 TMEM columns of A, two 16-byte core-matrix columns (256 B) of W
#pragma unroll
        for (int i = 0; i < K / 16; ++i)
            mma_f16_ts(c.mma_d, c.mma_a + a_col + i * 8, smem_desc(w_saddr + i * 256, 128, K_LAYOUT * 16), idesc_f16(N), i > 0);
        if (EXACT) {
#pragma unroll
            for (int i = 0; i < K / 16; ++i)
                mma_f16_ts(c.mma_d, c.mma_a + a_col + i * 8,
                           smem_desc(w_saddr + ROBOY_TC_OFF_LO_BYTES + i * 256, 128, K_LAYOUT * 16), idesc_f16(N), 1);
#pragma unroll
            for (int i = 0; i < K / 16; ++i)
                mma_f16_ts(c.mma_d, c.mma_a + lo_col + i * 8, smem_desc(w_saddr + i * 256, 128, K_LAYOUT * 16), idesc_f16(N), 1);
        }
        mma_commit(c.mbar);
    }
}

__device__ __forceinline__ void gemm_wait(TileCtx &c) {
    mbar_wait(c.mbar, c.parity);
    c.parity ^= 1u;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

__device__ __forceinline__ float f16_lo_to_f32(uint32_t pair) {
    float r;
    asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %1;\n\tcvt.f32.f16 %0, l;\n\t}" : "=f"(r) : "r"(pair));
    return r;
}
__device__ __forceinline__ float f16_hi_to_f32(uint32_t pair) {
    float r;
    asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %1;\n\tcvt.f32.f16 %0, h;\n\t}" : "=f"(r) : "r"(pair));
    return r;
}

// (x0, x1) -> float16 pairs hi = f16(x), lo = f16(x - hi)
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t &hi, uint32_t &lo) {
    hi = pack_f16x2(x0, x1);
    lo = pack_f16x2(__fsub_rn(x0, f16_lo_to_f32(hi)), __fsub_rn(x1, f16_hi_to_f32(hi)));
}

// A[:, 0..63] = tanh(D[:, 0..63] + bias) as float16 pairs.  Fast: MUFU.TANH, the bias is already in D (bias = nullptr);
// exact: the float32 kernel's tanh (ex2 + rcp, abs error ~3e-7), the result split into high and low halves, and the
// float32 bias of a 64-input layer added here.
template <bool EXACT>
__device__ __forceinline__ void tile_activation(const TileCtx &c, const float *__restrict__ bias) {
    using L = Cols<EXACT>;
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
        float v[16];
        tmem_ld16(c.tmem_a + L::D + ch * 16, v);
        tmem_ld_wait16(v);
        if (EXACT && bias) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                const float4 b = *reinterpret_cast<const float4 *>(bias + ch * 16 + i);
                v[i] = __fadd_rn(v[i], b.x); v[i + 1] = __fadd_rn(v[i + 1], b.y);
                v[i + 2] = __fadd_rn(v[i + 2], b.z); v[i + 3] = __fadd_rn(v[i + 3], b.w);
            }
        }
        uint32_t h[8], l[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (EXACT) split_f16x2(tanh_mufu(v[2 * i]), tanh_mufu(v[2 * i + 1]), h[i], l[i]);
            else h[i] = pack_f16x2(tanh_approx(v[2 * i]), tanh_approx(v[2 * i + 1]));
        }
        tmem_st<8>(c.tmem_a + L::A + ch * 8, h);
        if (EXACT) tmem_st<8>(c.tmem_a + L::ALo + ch * 8, l);
    }
}

// K = 16 input block of a tile: obs[0..8], 1 (multiplies the bias column of W1), zeros.
template <bool EXACT>
__device__ __forceinline__ void store_input(const TileCtx &c, const float (&o)[kObsDim]) {
    using L = Cols<EXACT>;
    uint32_t a[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u}, l[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    if (EXACT) {
#pragma unroll
        for (int i = 0; i < 4; ++i) split_f16x2(o[2 * i], o[2 * i + 1], a[i], l[i]);
        split_f16x2(o[8], 1.0f, a[4], l[4]);
        tmem_st<8>(c.tmem_a + L::InLo, l);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = pack_f16x2(o[2 * i], o[2 * i + 1]);
        a[4] = pack_f16x2(o[8], 1.0f);
    }
    tmem_st<8>(c.tmem_a + L::In, a);
}

// One network for the group's U tiles: obs (9) -> 64 -> 64 -> out (first 8 of the 16 padded output columns), biases
// included.  Fast: the input block [obs, 1, 0...] already sits in its own TMEM columns; exact: it is written here, over
// the first columns of the activation blocks.  `bias32`: the float32 biases b2 [64] | b3 [16] of this network (exact).
// With U = 2 the tiles ping-pong: while one tile's MMAs run, the threads do the other tile's activation math.
template <int U, bool EXACT>
__device__ __forceinline__ void group_mlp(TileCtx (&c)[U], const uint16_t *__restrict__ net, const float *__restrict__ bias32,
                                          const float (&o)[U][kObsDim], float (&out)[U][8]) {
    using L = Cols<EXACT>;
    const uint32_t w1 = smem_u32(net + ROBOY_TC_OFF_W1), w2 = smem_u32(net + ROBOY_TC_OFF_W2), w3 = smem_u32(net + ROBOY_TC_OFF_W3);
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (EXACT) store_input<EXACT>(c[u], o[u]);
        gemm_issue<16, 16, 64, EXACT>(c[u], L::In, L::InLo, w1);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        gemm_wait(c[u]);
        tile_activation<EXACT>(c[u], nullptr);                       // b1 rides in the product in both modes
        gemm_issue<L::KHid, kKHid, 64, EXACT>(c[u], L::A, L::ALo, w2);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        gemm_wait(c[u]);
        tile_activation<EXACT>(c[u], bias32);
        gemm_issue<L::KHid, kKHid, 16, EXACT>(c[u], L::A, L::ALo, w3);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        gemm_wait(c[u]);
        float v[16];
        tmem_ld16(c[u].tmem_a + L::D, v);
        tmem_ld_wait16(v);
#pragma unroll
        for (int k = 0; k < 8; ++k) out[u][k] = EXACT ? __fadd_rn(v[k], bias32[64 + k]) : v[k];
    }
}

// ---- merged form: the value and the policy network of one tile advance together ----
// One round trip: for each network K/16 (+1 for the constant-1 block) MMAs into its own accumulator, ONE commit.
template <int N, bool HIDDEN>
__device__ __forceinline__ void merged_issue(const TileCtx &c, uint32_t w_vf, uint32_t w_pi) {
    using M = ColsMerged;
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.sync %0, 128;" :: "r"(c.bar_id) : "memory");
    if (c.issuer) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int net = 0; net < 2; ++net) {
            const uint32_t d = c.mma_a + (net ? M::DPi : M::DVf), a = c.mma_a + (net ? M::APi : M::AVf), w = net ? w_pi : w_vf;
            if (HIDDEN) {   // 64 activations (4 MMAs) + the constant-1 block against the bias columns of W (K layout 80)
#pragma unroll
                for (int i = 0; i < 4; ++i) mma_f16_ts(d, a + i * 8, smem_desc(w + i * 256, 128, kKHid * 16), idesc_f16(N), i > 0);
                mma_f16_ts(d, c.mma_a + M::Ones, smem_desc(w + 4 * 256, 128, kKHid * 16), idesc_f16(N), 1);
            } else {        // the K = 16 input block, shared by both networks
                mma_f16_ts(d, c.mma_a + M::In, smem_desc(w, 128, 16 * 16), idesc_f16(N), 0);
            }
        }
        mma_commit(c.mbar);
    }
}

__device__ __forceinline__ void merged_activation(const TileCtx &c) {
    using M = ColsMerged;
#pragma unroll
    for (int net = 0; net < 2; ++net) {
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            float v[16];
            tmem_ld16(c.tmem_a + (net ? M::DPi : M::DVf) + ch * 16, v);
            tmem_ld_wait16(v);
            uint32_t h[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) h[i] = pack_f16x2(tanh_approx(v[2 * i]), tanh_approx(v[2 * i + 1]));
            tmem_st<8>(c.tmem_a + (net ? M::APi : M::AVf) + ch * 8, h);
        }
    }
}

// value = first output of the value net, mean = the 8 outputs of the policy net; three round trips
__device__ __forceinline__ void merged_mlp(TileCtx &c, const uint16_t *__restrict__ vf, const uint16_t *__restrict__ pi, float &value,
                                           float (&mean)[8]) {
    using M = ColsMerged;
    merged_issue<64, false>(c, smem_u32(vf + ROBOY_TC_OFF_W1), smem_u32(pi + ROBOY_TC_OFF_W1));
    gemm_wait(c);
    merged_activation(c);
    merged_issue<64, true>(c, smem_u32(vf + ROBOY_TC_OFF_W2), smem_u32(pi + ROBOY_TC_OFF_W2));
    gemm_wait(c);
    merged_activation(c);
    merged_issue<16, true>(c, smem_u32(vf + ROBOY_TC_OFF_W3), smem_u32(pi + ROBOY_TC_OFF_W3));
    gemm_wait(c);
    float v[16], m[16];
    tmem_ld16(c.tmem_a + M::DVf, v);
    tmem_ld16(c.tmem_a + M::DPi, m);
    tmem_ld_wait16(v);
    tmem_ld_wait16(m);
    value = v[0];
#pragma unroll
    for (int k = 0; k < 8; ++k) mean[k] = m[k];
}

}  // namespace

// U = tiles per group of 128 threads (thread i of the group owns row i of each of its U tiles); EXACT: split-float16
// operands and the accurate tanh (float32-level accuracy) instead of single float16 operands and tanh.approx.
// MERGED (fast arithmetic, U = 1): both networks of a tile advance together, three MMA round trips per step instead of six.
template <int U, bool EXACT, bool MERGED = false>
__global__ void __launch_bounds__(kPolicyTcMaxBlock / (MERGED ? 2 : U), 1) policy_rollout_tc_kernel(const __grid_constant__ StepParams p,
                                                                                      const __grid_constant__ PolicyParams q) {
    extern __shared__ __align__(128) float smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int n_warps = blockDim.x >> 5;
    const int group = warp >> 2, n_groups = n_warps >> 2;
    const int row_in_tile = (warp & 3) * 32 + lane;
    // shared memory: policy image (float16 weights in UMMA layout, then std / lognorm as float32) | obs stage
    // [32][9] per warp and tile | mbarriers | TMEM base | counters
    float *img = smem;
    const uint16_t *img16 = reinterpret_cast<const uint16_t *>(smem);
    float *stage = smem + kPolicyTcImagePad + warp * (U * 32 * kObsDim);
    uint64_t *mbars = reinterpret_cast<uint64_t *>(smem + kPolicyTcImagePad + n_warps * (U * 32 * kObsDim));
    double *s_red = reinterpret_cast<double *>(mbars + 4);
    unsigned int *s_cnt = reinterpret_cast<unsigned int *>(s_red + n_warps);
    uint32_t *tmem_base_slot = s_cnt + kCntWords;
    using L = Cols<EXACT>;
    // fast: the high halves of the weights and the float32 tail; exact: the whole image
    for (int i = threadIdx.x; i < ROBOY_TC_IMAGE_BYTES / 16; i += blockDim.x)
        if (EXACT || i < ROBOY_TC_OFF_LO_BYTES / 16 || i >= ROBOY_TC_OFF_STD_BYTES / 16)
            reinterpret_cast<float4 *>(img)[i] = reinterpret_cast<const float4 *>(q.image)[i];
    if (threadIdx.x < kCntWords) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        for (int t = 0; t < n_groups * U; ++t)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(mbars + t)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const int n_tiles = n_groups * U;
    constexpr int kTile = MERGED ? ColsMerged::Tile : L::Tile;
    const uint32_t need_cols = (uint32_t)n_tiles * kTile;
    const uint32_t tmem_cols = need_cols <= 128 ? 128u : need_cols <= 256 ? 256u : 512u;   // a power of two >= 32
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(tmem_base_slot)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // the weights were written through the generic proxy; the tensor core reads them through the async proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(tmem_base_slot);

    TileCtx c[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int tile = group * U + u;
        c[u].mma_a = tmem_base + tile * kTile;
        c[u].mma_d = c[u].mma_a + L::D;
        c[u].tmem_a = c[u].mma_a + ((uint32_t)((warp & 3) * 32) << 16);
        c[u].mbar = smem_u32(mbars + tile);
        c[u].parity = 0;
        c[u].bar_id = 1 + group;
        c[u].issuer = row_in_tile == 0;
    }

    const bool FASTDIV = q.fastdiv;
    const uint64_t t_first = counter_begin(p.cc);
    const uint32_t n_end = (uint32_t)p.e_end;
    const size_t n = (size_t)p.n;
    const uint32_t n_chunks = (n_end + U * kTileEnvs - 1) / (U * kTileEnvs);
    const uint16_t *vf_net = img16 + ROBOY_TC_OFF_VF, *pi_net = img16 + ROBOY_TC_OFF_PI;
    const float *sd = img + ROBOY_TC_OFF_STD_BYTES / 4;   // (the image keeps its layout in shared memory)
    const float lognorm = sd[8];
    const float *bias32 = sd + 12;   // float32 b2 | b3 per network (exact mode)
    float sum_reward = 0.0f;

    // all threads of a group walk the same chunks of U * 128 envs (the group's named barrier needs every one of them)
    for (uint32_t chunk = blockIdx.x * n_groups + group; chunk < n_chunks; chunk += gridDim.x * n_groups) {
        uint32_t env[U], wbase[U];   // this thread's env in tile u; first env of this warp's 32 rows of tile u
        bool live[U];
        EnvRegs s[U];
        float o[U][kObsDim];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            wbase[u] = (chunk * U + u) * kTileEnvs + (warp & 3) * 32;
            env[u] = wbase[u] + lane;
            live[u] = env[u] < n_end;
            s[u].g0 = live[u] ? p.goal[env[u]] : 0.f;
            s[u].g1 = live[u] ? p.goal1[env[u]] : 0.f;
            s[u].g2 = live[u] ? p.goal2[env[u]] : 0.f;
            s[u].sf = live[u] ? p.step_flags[env[u]] : 1u;
            if (FASTDIV) normalize_goal<true>(s[u], p.c, p.f);
            else normalize_goal<false>(s[u], p.c, p.f);
#pragma unroll
            for (int k = 0; k < kObsDim; ++k) o[u][k] = live[u] ? q.obs[(size_t)env[u] * kObsDim + k] : 0.f;
            if (!EXACT) {   // the constant K block behind the 64 activations: 1 (multiplies the bias column of W2 / W3), then zeros
                const uint32_t ones[8] = {pack_f16x2(1.0f, 0.0f), 0u, 0u, 0u, 0u, 0u, 0u, 0u};
                tmem_st<8>(c[u].tmem_a + (MERGED ? ColsMerged::Ones : L::Ones), ones);
            }
        }

        for (uint32_t tt = 0;; ++tt) {
            float out[U][8];
            if constexpr (MERGED) {
                {
                    const uint32_t a[8] = {pack_f16x2(o[0][0], o[0][1]), pack_f16x2(o[0][2], o[0][3]), pack_f16x2(o[0][4], o[0][5]),
                                           pack_f16x2(o[0][6], o[0][7]), pack_f16x2(o[0][8], 1.0f), 0u, 0u, 0u};
                    tmem_st<8>(c[0].tmem_a + ColsMerged::In, a);
                }
                float value;
                merged_mlp(c[0], vf_net, pi_net, value, out[0]);
                if (live[0]) q.values[(size_t)tt * n + env[0]] = value;
                if (tt == q.T) break;
            } else {
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (!EXACT) store_input<EXACT>(c[u], o[u]);   // (exact: written per network, it shares columns with the activations)
            if constexpr (EXACT) {
                // one copy of the network code for both nets: the exact kernel is three times the size of the fast one
                // and instruction-cache misses showed in its profile (measured +12 %; the fast kernel loses 1 % this way)
                bool last = false;
#pragma unroll 1
                for (int net = 0; net < 2; ++net) {
                    group_mlp<U, EXACT>(c, net == 0 ? vf_net : pi_net, bias32 + net * ROBOY_TC_BIAS32_NET_FLOATS, o, out);   // value of obs[tt], then the mean
                    if (net == 0) {
#pragma unroll
                        for (int u = 0; u < U; ++u)
                            if (live[u]) q.values[(size_t)tt * n + env[u]] = out[u][0];
                        if (tt == q.T) { last = true; break; }                  // (the bootstrap value of obs[T])
                    }
                }
                if (last) break;
            } else {
                group_mlp<U, EXACT>(c, vf_net, bias32, o, out);           // value of obs[tt] (bootstrap value at tt == T)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (live[u]) q.values[(size_t)tt * n + env[u]] = out[u][0];
                if (tt == q.T) break;
                group_mlp<U, EXACT>(c, pi_net, bias32 + ROBOY_TC_BIAS32_NET_FLOATS, o, out);   // mean of the Gaussian
            }
            }   // !MERGED
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float *row = stage + (u * 32 + lane) * kObsDim;
                sample_and_step(p, q, sd, lognorm, out[u], s[u], live[u], env[u], tt, t_first + tt, row, s_cnt, sum_reward);
#pragma unroll
                for (int k = 0; k < kObsDim; ++k) o[u][k] = row[k];   // (finish_episode may have replaced the row)
            }
            // ---- obs[tt + 1]: this warp's 32 rows of each tile, stored coalesced ----
            __syncwarp();
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool full = wbase[u] + 32 <= n_end;
                float *dst = q.obs + ((size_t)(tt + 1) * n + wbase[u]) * kObsDim;
                const float *st = stage + u * 32 * kObsDim;
                if (full && q.obs_aligned) {
                    const float4 *src = reinterpret_cast<const float4 *>(st);
                    reinterpret_cast<float4 *>(dst)[lane] = src[lane];
                    reinterpret_cast<float4 *>(dst)[32 + lane] = src[32 + lane];
                    if (lane < 8) reinterpret_cast<float4 *>(dst)[64 + lane] = src[64 + lane];
                } else if (wbase[u] < n_end) {
                    const uint32_t rows = full ? 32u : n_end - wbase[u];
                    for (uint32_t i = lane; i < rows * kObsDim; i += 32) dst[i] = st[i];
                }
            }
            __syncwarp();
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (live[u]) p.step_flags[env[u]] = s[u].sf;
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    policy_stats_tail(p, q.T, t_first, sum_reward, s_red, s_cnt);   // contains a __syncthreads()
    if (warp == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

PolicyGeom policy_tc_geometry(uint64_t n_envs, int sm_count, int variant, bool exact) {
    PolicyGeom g;
    const uint64_t n_tiles = (n_envs + kTileEnvs - 1) / kTileEnvs;
    // variant 0 = choose: small populations (at most two 128-env tiles per SM) are bound by the MMA round trips of
    // a step, so both networks advance together (3, "merged": three round trips instead of six; fast arithmetic only);
    // otherwise one tile per thread group (1): four groups (16 warps) per SM hide the round trips and the TMEM / MUFU
    // latencies better than two groups ping-ponging two tiles each (2; measured at 1,048,576 envs: 1.09e10 vs 7.1e9
    // env-steps/s), which stays selectable for experiments.
    if (variant == 0) variant = (!exact && n_tiles <= 2ull * sm_count) ? 3 : 1;
    if (exact) variant = 1;
    const int U = variant == 2 ? 2 : 1;
    g.envs_per_thread = variant;
    const uint64_t n_chunks = (n_envs + U * kTileEnvs - 1) / (U * kTileEnvs);
    const uint64_t max_groups = variant == 3 ? ColsMerged::MaxGroups : 4 / U;   // TMEM: 512 columns per SM
    uint64_t groups = (n_chunks + sm_count - 1) / sm_count;          // spread the groups over the SMs first
    if (groups > max_groups) groups = max_groups;
    const uint64_t grid = (n_chunks + groups - 1) / groups;
    g.grid = (int)(grid < (uint64_t)sm_count ? grid : (uint64_t)sm_count);
    g.block = (int)groups * kTileEnvs;
    const uint64_t warps = groups * 4;
    g.smem = (int)(sizeof(float) * (kPolicyTcImagePad + warps * U * 32 * kObsDim) + 4 * sizeof(uint64_t) + sizeof(double) * warps +
                   sizeof(unsigned int) * (kCntWords + 2));   // counters, TMEM base, pad
    return g;
}

cudaError_t launch_policy_rollout_tc(const StepParams &p, const PolicyParams &q, bool penalty, bool bonus, bool auto_reset,
                                     bool fastdiv, int sm_count, int variant, bool exact, cudaStream_t stream) {
    if (p.e_end <= p.e_begin) return cudaSuccess;
    PolicyParams qq = q;
    qq.penalty = penalty;
    qq.bonus = bonus;
    qq.auto_reset = auto_reset;
    qq.fastdiv = fastdiv;
    const PolicyGeom g = policy_tc_geometry(p.e_end, sm_count, variant, exact);
    void (*fn)(const StepParams, const PolicyParams) =
        exact ? policy_rollout_tc_kernel<1, true>
              : g.envs_per_thread == 3 ? policy_rollout_tc_kernel<1, false, true>
              : g.envs_per_thread == 2 ? policy_rollout_tc_kernel<2, false> : policy_rollout_tc_kernel<1, false>;
    cudaError_t err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem);
    if (err != cudaSuccess) return err;
    fn<<<g.grid, g.block, g.smem, stream>>>(p, qq);
    return cudaGetLastError();
}

}  // namespace roboy
