// Robot-generic sm_100a kernels (see roboy_generic.cuh): runtime joint / tendon counts, one bound per component.
// Arithmetic follows the reference's operation order and numpy's dtype promotions exactly as
// msj_math.cuh does (paths relative to gym_roboy/ in Roboy/gym-roboy):
//   normalisation   envs/robots/roboy_robot.py:93-95   (2*v - max_k - min_k) / (max_k - min_k), per component
//   _l2_distance    envs/roboy_env.py:137-140          subtract, NaN -> 0, np.linalg.norm
//   np.linalg.norm  float32[n < 32]: float products summed sequentially in a double, rounded to float32, float32 sqrt;
//                   float64[n < 16]: sequential FMA (both pinned in oracle/roboy_oracle.c's header)
//   compute_reward  envs/roboy_env.py:92-112;   _did_reach_goal  :125-134;   Stub  envs/simulations/simulation_client.py:26-47
// The fused step (generic_step_kernel) is bound by HBM at 4A + 16J + 13 algorithmic bytes per env-step and keeps every
// access of its hot path coalesced; the other kernels here (construction, injection, the un-fused plug-in calls, the
// external feed) are one thread per env and not on anybody's hot path.  The MSJ hot step has its own kernel
// (roboy_kernels.cu).
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <map>
#include <mutex>
#include <utility>

#include "../../include/roboy_b200.h"
#include "roboy_generic.cuh"
#include "generic_env.cuh"

namespace roboy {
namespace {

constexpr uint32_t kFullMask = 0xffffffffu;
constexpr int kGenericBlock = 256;

__device__ __forceinline__ double g_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

int g_grid(uint64_t items, int sm_count) {
    const uint64_t want = (items + kGenericBlock - 1) / kGenericBlock;
    const uint64_t cap = (uint64_t)sm_count * 8;
    return (int)(want < cap ? want : cap);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// Fused step: RoboyEnv.step (roboy_env.py:51-70) over the Stub (simulation_client.py:36-40), reward, done, goal
// resampling and -- under auto_reset -- the vec-env worker's reset-on-done, for any robot.
//
// A warp walks 32 consecutive envs per iteration (so the done mask is one ballot word) and every global access of the
// hot path is coalesced although rows are A and 3J floats wide:
//   * actions [n][A]: each lane reads its own row, eight floats at a time (float4 when A % 4 == 0); the 32 rows of a warp
//     are contiguous, so each line comes from DRAM once and L1 serves the rest;
//   * goal rows are SoA (one coalesced load per joint);
//   * obs [n][3J]: each lane writes its row into a shared-memory stage, the warp copies the chunk's 32*3J contiguous
//     floats out as float4.
// One instantiation per joint count (1..15): the per-env vectors live in registers, the loops over joints are fully unrolled.
// ---------------------------------------------------------------------------------------------
namespace {

// Threads per CTA of the fused step: up to 10 joints fit 128 registers (two CTAs of 256 per SM, 16 warps); beyond that a
// thread needs ~160, and three CTAs of 128 keep 12 warps on the SM where one of 256 kept 8 (15 joints: 0.73 -> 0.76).
__host__ __device__ constexpr int g_step_block(int J) { return J <= 10 ? 256 : 128; }
__host__ __device__ constexpr int g_min_blocks(int J) { return J <= 10 ? 2 : 3; }   // 3 x 256 per SM spills even at one joint (measured: 0.46 vs 0.51)

}  // namespace

// max(m, |x|, |y|, |z|, |w|) that PROPAGATES NaN (fmaxf would drop it): the range assert of roboy_env.py:52 for four
// actions and the running maximum in two FMNMX
__device__ __forceinline__ float g_maxabs4_nan(float m, const float4 &v) {
    float o;
    asm("{\n\t.reg .f32 ax, ay, az, aw, t;\n\t"
        "abs.f32 ax, %1;\n\tabs.f32 ay, %2;\n\tabs.f32 az, %3;\n\tabs.f32 aw, %4;\n\t"
        "max.NaN.f32 t, az, aw, %5;\n\t"
        "max.NaN.f32 %0, ax, ay, t;\n\t}"
        : "=f"(o)
        : "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "f"(m));
    return o;
}
// min(m, |x - c|, |y - c|, |z - c|, |w - c|): how close four actions come to the centre of the hold intervals
__device__ __forceinline__ float g_mindist4(float m, const float4 &v, float c) {
    float o;
    asm("{\n\t.reg .f32 dx, dy, dz, dw, t;\n\t"
        "sub.rn.f32 dx, %1, %5;\n\tsub.rn.f32 dy, %2, %5;\n\tsub.rn.f32 dz, %3, %5;\n\tsub.rn.f32 dw, %4, %5;\n\t"
        "abs.f32 dx, dx;\n\tabs.f32 dy, dy;\n\tabs.f32 dz, dz;\n\tabs.f32 dw, dw;\n\t"
        "min.f32 t, dz, dw, %6;\n\t"
        "min.f32 %0, dx, dy, t;\n\t}"
        : "=f"(o)
        : "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "f"(c), "f"(m));
    return o;
}

template <int JM, bool FASTDIV>
__global__ void __launch_bounds__(g_step_block(JM), g_min_blocks(JM)) generic_step_kernel(const __grid_constant__ GStepParams p) {
    constexpr int kGenericWarps = g_step_block(JM) / 32;
    extern __shared__ __align__(16) float s_stage[];          // [kGenericWarps][32 * 3J] observation rows of a chunk
    __shared__ double s_sum_reward;
    __shared__ unsigned long long s_eplen;
    __shared__ unsigned int s_cnt[4];   // episodes, successes, holds, violations: rare events, counted where they happen
    const RobotSpec &r = p.r;
    constexpr int J = JM;   // one instantiation per joint count: the per-env vectors are registers, loops have no predicates
    const int A = r.A;
    constexpr int D = 3 * J;
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x == 4) s_eplen = 0;
    if (threadIdx.x == 5) s_sum_reward = 0.0;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    __syncthreads();
    const uint64_t t = counter_begin(p.cc);
    float *stage = s_stage + (size_t)wib * 32 * D;
    // Env indices are 32-bit (a handle holds fewer than 2^31 envs -- roboy_create checks; 2^31 envs of the smallest robot
    // would be 70 GB of observations alone): half the integer instructions of 64-bit counters.  ELEMENT offsets (env * A,
    // env * 3J, joint * n + env) pass 2^32 and are formed with widening multiplies.
    const uint32_t e_begin = (uint32_t)p.e_begin, e_end = (uint32_t)p.e_end, n_envs = (uint32_t)p.n;
    const uint32_t warp = blockIdx.x * kGenericWarps + wib;
    const uint32_t stride = gridDim.x * kGenericWarps * 32;
    const bool obs_vec = (((uintptr_t)p.obs) & 15) == 0;
    const bool act_al16 = (((uintptr_t)p.actions) & 15) == 0;
    const bool act_vec = (A & 3) == 0 && act_al16;
    const uint32_t row_bytes = (uint32_t)A * 4;
    const int n4 = 8 * A;                                     // float4s in the 32 action rows of a full chunk
    const char *pf_act = reinterpret_cast<const char *>(p.actions) + (size_t)lane * 128;
    // lanes 0..J-1 prefetch the line of their goal row, lane J the step words (one pointer per lane)
    const float *pf_goal = lane < J ? p.goal + (size_t)lane * n_envs : reinterpret_cast<const float *>(p.step_flags);
    // Episode statistics cost the hot loop ONE register: the reward sum of this thread (float, like the tuned kernels; the
    // warps' sums are added in double).  Episode ends, holds and violations are rare and go to shared-memory counters
    // where they happen; the step count is the size of the range.
    float sum_reward = 0.0f;

    for (uint32_t base = e_begin + warp * 32; base < e_end; base += stride) {
        const uint32_t e = base + lane;
        const bool live = e < e_end;
        const uint32_t rows = e_end - base < 32 ? e_end - base : 32u;
        {   // the warp's NEXT chunk into L2 (no registers held): its action lines, one line per goal row, the step words
            const uint32_t nb = base + stride;
            if (nb + 32 <= e_end) {
                const char *ap = pf_act + (uint64_t)nb * row_bytes;     // 32 rows = A lines of 128 bytes
                if (lane < A) asm volatile("prefetch.global.L2 [%0];" ::"l"(ap));
                if (lane + 32 < A) asm volatile("prefetch.global.L2 [%0];" ::"l"(ap + 4096));
                if (lane <= J) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf_goal + nb));
            }
        }

        // ---- actions: roboy_env.py:52 assert + the hold test of simulation_client.py:38 ----
        // Fast test, whole chunk at once: the 32 rows are 32*A contiguous floats, read coalesced as float4 (a chunk starts
        // at a multiple of 128*A bytes).  If every |x| <= 1 (NaN fails) nobody trips the assert; if no x lies inside the hull
        // of the hold intervals nobody holds.  That settles almost every chunk in ~11 instructions per float4; otherwise
        // each lane examines its own row (the lines are in L1 by then).
        bool act_ok = true, hold = false;
        bool settled = false;
        // Every load of the chunk is issued before the Philox draws (which depend on no memory), so the ~150 instructions
        // of the draws cover the latency of the loads instead of following it.
        const bool whole = rows == 32 && act_al16;
        const float4 *a4 = reinterpret_cast<const float4 *>(p.actions + (uint64_t)base * (uint32_t)A);
        const float pad = r.hold_pad;
        float4 v[4];
        if (whole) {
#pragma unroll
            for (int u = 0; u < 4; ++u)
                v[u] = lane + 32 * u < n4 ? a4[lane + 32 * u] : make_float4(pad, pad, pad, pad);
        }
        float q[JM], qd[JM], g[JM];
#pragma unroll
        for (int k = 0; k < JM; ++k) q[k] = qd[k] = g[k] = 0.0f;
        uint32_t sf = 0;
        const uint64_t gid = p.gid_base + e;
        if (live) {
            sf = p.step_flags[e];
#pragma unroll
            for (int k = 0; k < JM; ++k)
                g[k] = p.goal[(size_t)k * n_envs + e];
            // simulation_client.py:40 -> roboy_robot.py:35-39: fresh sample, not stored; velocities from the ANGLE space
            // (drawn before the hold test is known: a held env, rare, discards them)
            DrawCursor cur;
            cur.block = 0xffffffffu;
#pragma unroll
            for (int k = 0; k < JM; ++k)
                q[k] = g_draw_value(r, p.keys, gid, t, cur, k, k);
#pragma unroll
            for (int k = 0; k < JM; ++k)
                qd[k] = g_draw_value(r, p.keys, gid, t, cur, J + k, k);
        }
        if (whole) {
            float mx = 0.0f, near = INFINITY;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                mx = g_maxabs4_nan(mx, v[u]);
                near = g_mindist4(near, v[u], r.hold_c);
            }
            for (int i0 = lane + 128; i0 < n4; i0 += 128) {   // more than 16 tendons
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    v[u] = i0 + 32 * u < n4 ? a4[i0 + 32 * u] : make_float4(pad, pad, pad, pad);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    mx = g_maxabs4_nan(mx, v[u]);
                    near = g_mindist4(near, v[u], r.hold_c);
                }
            }
            settled = __all_sync(kFullMask, mx <= 1.0f) && !__any_sync(kFullMask, near <= r.hold_h);
        }
        if (!settled && live) {
            hold = true;
            const float *a = p.actions + (uint64_t)e * (uint32_t)A;
            if (act_vec) {
                for (int k0 = 0; k0 < A; k0 += 8) {
                    const float4 v0 = *reinterpret_cast<const float4 *>(a + k0);
                    const float4 v1 = k0 + 4 < A ? *reinterpret_cast<const float4 *>(a + k0 + 4) : make_float4(0.5f, 0.5f, 0.5f, 0.5f);
                    const float x[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (k0 + u < A) {
                            act_ok = act_ok && (x[u] >= -1.0f && x[u] <= 1.0f);
                            hold = hold && (x[u] >= r.hold_lo[k0 + u] && x[u] <= r.hold_hi[k0 + u]);
                        }
                    }
                }
            } else {
                for (int k0 = 0; k0 < A; k0 += 8) {
                    float x[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) x[u] = k0 + u < A ? a[k0 + u] : 0.5f;
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (k0 + u < A) {
                            act_ok = act_ok && (x[u] >= -1.0f && x[u] <= 1.0f);
                            hold = hold && (x[u] >= r.hold_lo[k0 + u] && x[u] <= r.hold_hi[k0 + u]);
                        }
                    }
                }
            }
        }

        const bool done = generic_env_step<JM>(p, FASTDIV, live, hold, act_ok, q, qd, g, sf, gid, t, e, n_envs, s_cnt, &s_eplen,
                                               sum_reward, [&](uint32_t word, float rf, bool d, bool) {
                                                   p.step_flags[e] = word;
                                                   p.reward[e] = rf;
                                                   p.done[e] = (uint8_t)d;
                                               });
        // ---- obs = [q, qd, goal] (:62 -> :75-80): rows staged in shared memory, copied out coalesced ----
        {
            float *row = stage + lane * D;
#pragma unroll
            for (int k = 0; k < JM; ++k)
                { row[k] = q[k]; row[J + k] = qd[k]; row[2 * J + k] = g[k]; }
            __syncwarp();
            float *dst = p.obs + (uint64_t)base * (uint32_t)D;
            if (obs_vec && rows == 32) {   // 32 * 3J floats = 24J float4s, 16-byte aligned at every chunk
                constexpr int N4 = 24 * J;
                float4 *dst4 = reinterpret_cast<float4 *>(dst);
                const float4 *src4 = reinterpret_cast<const float4 *>(stage);
#pragma unroll
                for (int i = 0; i < (N4 + 31) / 32; ++i)
                    if (i * 32 + 31 < N4 || i * 32 + lane < N4) dst4[i * 32 + lane] = src4[i * 32 + lane];
            } else {
                const uint32_t n_el = rows * (uint32_t)D;
                for (uint32_t i = lane; i < n_el; i += 32u) dst[i] = stage[i];
            }
            __syncwarp();
        }
        if (p.done_bits != nullptr) {
            const uint32_t dm = __ballot_sync(kFullMask, done);
            if (lane == 0) p.done_bits[base >> 5] = dm;
        }
    }
    // episode statistics: reward sums warp-reduced in double -> shared -> one set of atomics per CTA
    {
        const double w = g_warp_sum((double)sum_reward);
        if (lane == 0 && w != 0.0) atomicAdd(&s_sum_reward, w);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double episodes = (double)s_cnt[0], successes = (double)s_cnt[1];
        double st[ROBOY_STAT_COUNT];
        st[ROBOY_STAT_STEPS] = blockIdx.x == 0 ? (double)(e_end - e_begin) : 0.0;
        st[ROBOY_STAT_EPISODES] = episodes;
        st[ROBOY_STAT_SUCCESSES] = successes;
        st[ROBOY_STAT_TIMEOUTS] = episodes - successes;
        st[ROBOY_STAT_SUM_REWARD] = s_sum_reward;
        st[ROBOY_STAT_SUM_EPLEN] = (double)s_eplen;
        st[ROBOY_STAT_HOLDS] = (double)s_cnt[2];
        st[ROBOY_STAT_VIOLATIONS] = (double)s_cnt[3];
#pragma unroll
        for (int k = 0; k < ROBOY_STAT_COUNT; ++k)
            if (st[k] != 0.0) atomicAdd(p.stats + k, st[k]);
        counter_end(p.cc, t);
    }
}

// ---------------------------------------------------------------------------------------------
// Create-time proof of the fast division (see roboy_generic.cuh)
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void fastdiv_prove_kernel(float span, float *rcp_out, unsigned long long *mismatches) {
    const float rcp = g_refined_rcp(span);
    unsigned long long bad = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const float t = __uint_as_float((uint32_t)i);
        const float at = fabsf(t);
        if (at >= kFastDivLo && at <= kFastDivHi)
            bad += __float_as_uint(g_div_core(t, span, rcp)) != __float_as_uint(__fdiv_rn(t, span));
    }
    if (bad) atomicAdd(mismatches, bad);
    if (blockIdx.x == 0 && threadIdx.x == 0) *rcp_out = rcp;
}
}  // namespace

cudaError_t prove_generic_fastdiv(RobotSpec &r, int sm_count, cudaStream_t stream) {
    struct Proof { float rcp; bool ok; };
    static std::mutex mu;
    static std::map<std::pair<int, uint32_t>, Proof> cache;   // (device, span bits) -> proof
    int device = 0;
    cudaError_t err = cudaGetDevice(&device);
    if (err != cudaSuccess) return err;
    r.fastdiv = 1;
    float *rcp_dev = nullptr;
    unsigned long long *bad_dev = nullptr;
    for (int which = 0; which < 2 * r.J && err == cudaSuccess; ++which) {
        const int k = which % r.J;
        const float span = which < r.J ? r.a_span[k] : r.v_span[k];
        uint32_t bits;
        memcpy(&bits, &span, 4);
        Proof pr{0.0f, false};
        bool have = false;
        {
            std::lock_guard<std::mutex> lock(mu);
            auto it = cache.find({device, bits});
            if (it != cache.end()) { pr = it->second; have = true; }
        }
        if (!have) {
            if (span >= 0x1p-40f && span <= 0x1p40f) {
                if (!rcp_dev) {
                    err = cudaMalloc(&rcp_dev, sizeof(float));
                    if (err == cudaSuccess) err = cudaMalloc(&bad_dev, sizeof(unsigned long long));
                    if (err != cudaSuccess) break;
                }
                err = cudaMemsetAsync(bad_dev, 0, sizeof(unsigned long long), stream);
                if (err != cudaSuccess) break;
                fastdiv_prove_kernel<<<sm_count * 8, 256, 0, stream>>>(span, rcp_dev, bad_dev);
                unsigned long long bad = 1;
                err = cudaMemcpyAsync(&bad, bad_dev, sizeof(bad), cudaMemcpyDeviceToHost, stream);
                if (err == cudaSuccess) err = cudaMemcpyAsync(&pr.rcp, rcp_dev, sizeof(float), cudaMemcpyDeviceToHost, stream);
                if (err == cudaSuccess) err = cudaStreamSynchronize(stream);
                if (err != cudaSuccess) break;
                pr.ok = bad == 0;
            }
            std::lock_guard<std::mutex> lock(mu);
            cache[{device, bits}] = pr;
        }
        (which < r.J ? r.a_rcp[k] : r.v_rcp[k]) = pr.rcp;
        if (!pr.ok) r.fastdiv = 0;
    }
    if (rcp_dev) cudaFree(rcp_dev);
    if (bad_dev) cudaFree(bad_dev);
    if (err != cudaSuccess) r.fastdiv = 0;
    return err;
}

void generic_step_geometry(int J, uint64_t envs, int sm_count, int *grid, int *block, int *smem_bytes) {
    const int b = g_step_block(J), warps = b / 32;
    const uint64_t n_chunks = (envs + 31) / 32;
    const uint64_t want = (n_chunks + warps - 1) / warps;
    const uint64_t cap = (uint64_t)sm_count * 4 * (256 / b);
    *grid = (int)(want < cap ? want : cap);
    *block = b;
    *smem_bytes = (int)(sizeof(float) * warps * 32 * 3 * (size_t)J);
}

cudaError_t launch_generic_step(const GStepParams &p, int sm_count, cudaStream_t stream) {
    if (p.e_end <= p.e_begin) return cudaSuccess;
    const int J = p.r.J;
    int grid, block, smem;
    generic_step_geometry(J, p.e_end - p.e_begin, sm_count, &grid, &block, &smem);
    switch (J) {
#define ROBOY_GENERIC_CASE(JJ) \
        case JJ: \
            if (p.r.fastdiv) generic_step_kernel<JJ, true><<<grid, block, smem, stream>>>(p); \
            else generic_step_kernel<JJ, false><<<grid, block, smem, stream>>>(p); \
            break;
        ROBOY_GENERIC_JOINT_COUNTS(ROBOY_GENERIC_CASE)
#undef ROBOY_GENERIC_CASE
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Construction and reset: RoboyEnv.__init__ / reset (roboy_env.py:12-38, :82-87) over the Stub (:29-31, :42-44)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGenericBlock) generic_init_or_reset_kernel(const __grid_constant__ GInitParams p) {
    const uint64_t t = counter_begin(p.cc);
    const RobotSpec &r = p.r;
    const int J = r.J, D = 3 * J;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < p.n; e += stride) {
        if (p.mask && !p.mask[e]) continue;
        const uint64_t gid = p.gid_base + e;
        float g[kJointPad];
        g_draw_goal(r, p.keys, gid, t, 0, g);
        for (int k = 0; k < J; ++k) p.goal[(size_t)k * p.n + e] = g[k];
        if (p.held) {
            // StubSimulationClient.__init__ (simulation_client.py:31): _state = new_random_state()
            float q[kJointPad], qd[kJointPad];
            g_draw_state(r, p.keys, gid, t, q, qd);
            for (int k = 0; k < J; ++k) {
                p.held[(size_t)k * p.n + e] = q[k];
                p.held[(size_t)(J + k) * p.n + e] = qd[k];
            }
            p.step_flags[e] = 1u;  // roboy_env.py:38
        } else {
            // forward_reset_command (simulation_client.py:42-44): _state = float64 zero state
            p.step_flags[e] = 1u | ROBOY_F_HELD_ZERO64;  // roboy_env.py:85
        }
        if (p.obs) {
            float *o = p.obs + e * D;
            for (int k = 0; k < 2 * J; ++k) o[k] = 0.0f;
            for (int k = 0; k < J; ++k) o[2 * J + k] = g[k];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) counter_end(p.cc, t);
}

cudaError_t launch_generic_init_or_reset(const GInitParams &p, int sm_count, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    generic_init_or_reset_kernel<<<g_grid(p.n, sm_count), kGenericBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Stand-alone compute_reward / _did_reach_goal over float32 arrays [k][J]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGenericBlock) generic_compute_reward_kernel(const __grid_constant__ GRewardParams p) {
    const int J = p.r.J;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.k; i += stride) {
        float q[kJointPad], qd[kJointPad], g[kJointPad], gqd[kJointPad];
        for (int k = 0; k < J; ++k) {
            q[k] = p.q[i * J + k];
            qd[k] = p.qd[i * J + k];
            g[k] = p.goal_q[i * J + k];
            gqd[k] = p.goal_qd ? p.goal_qd[i * J + k] : 0.0f;
        }
        const bool feasible = p.feasible ? p.feasible[i] != 0 : true;
        RobotSpec r = p.r;
        if (p.check_range != 1) {
            r.reward_lo = -INFINITY;
            r.reward_hi = INFINITY;
        }
        double rew;
        bool reached, violation;
        g_reward_reached(r, q, qd, false, feasible, g, p.goal_qd ? gqd : nullptr, p.penalty != 0, p.bonus != 0, rew, reached,
                         violation, p.check_range == 2);
        p.reward[i] = rew;
        if (p.reached) p.reached[i] = (uint8_t)reached;
        if (violation && p.check_range == 1) {   // (a NaN reward fails even an infinite range: only when a check was asked for)
            atomicOr(p.err_flags, ROBOY_ERR_REWARD_RANGE);
            atomicMin(p.first_bad, (unsigned long long)(p.gid_base + i));
            atomicAdd(p.stats + ROBOY_STAT_VIOLATIONS, 1.0);
        }
    }
}

cudaError_t launch_generic_compute_reward(const GRewardParams &p, int sm_count, cudaStream_t stream) {
    if (p.k == 0) return cudaSuccess;
    generic_compute_reward_kernel<<<g_grid(p.k, sm_count), kGenericBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Indexed state injection / read-back
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGenericBlock) generic_scatter_kernel(const __grid_constant__ GScatterParams p) {
    const int J = p.r.J;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.k; i += stride) {
        const int64_t e64 = p.idx ? p.idx[i] : (int64_t)i;
        if (e64 < 0 || (uint64_t)e64 >= p.n) continue;
        const uint64_t e = (uint64_t)e64;
        if (p.goal_q) {
            bool inside = true;
            for (int k = 0; k < J; ++k) {
                const float v = p.goal_q[i * J + k];
                inside = inside && (v >= p.r.a_lo[k] && v <= p.r.a_hi[k]);  // roboy_robot.py:76
                p.goal[(uint64_t)k * p.n + e] = v;
            }
            if (!inside) {
                atomicOr(p.err_flags, ROBOY_ERR_GOAL_BOUNDS);
                atomicMin(p.first_bad, (unsigned long long)(p.gid_base + e));
            }
        }
        if (p.q) {
            for (int k = 0; k < J; ++k) {
                p.held[(uint64_t)k * p.n + e] = p.q[i * J + k];
                p.held[(uint64_t)(J + k) * p.n + e] = p.qd[i * J + k];
            }
            uint32_t sf = p.step_flags[e] & ROBOY_STEP_MASK;
            if (p.feasible && !p.feasible[i]) sf |= ROBOY_F_HELD_INFEASIBLE;
            p.step_flags[e] = sf;
        }
        if (p.step) {
            const uint32_t s = (uint32_t)p.step[i] & ROBOY_STEP_MASK;
            p.step_flags[e] = (p.step_flags[e] & ~ROBOY_STEP_MASK) | s;
        }
        if (p.out_q) {  // SimulationClient.read_state
            const uint32_t sf = p.step_flags[e];
            const bool z = sf & ROBOY_F_HELD_ZERO64;
            for (int k = 0; k < J; ++k) {
                p.out_q[i * J + k] = z ? 0.0f : p.held[(uint64_t)k * p.n + e];
                p.out_qd[i * J + k] = z ? 0.0f : p.held[(uint64_t)(J + k) * p.n + e];
            }
            // bit 0: is_feasible; bit 1: the state is the reference's FLOAT64 zero state (roboy_robot.py:41-45)
            if (p.out_feasible) p.out_feasible[i] = z ? 3 : !(sf & ROBOY_F_HELD_INFEASIBLE);
        }
    }
}

cudaError_t launch_generic_scatter(const GScatterParams &p, int sm_count, cudaStream_t stream) {
    if (p.k == 0) return cudaSuccess;
    generic_scatter_kernel<<<g_grid(p.k, sm_count), kGenericBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Un-fused SimulationClient calls (the plug-in API the reference's own RoboyEnv drives)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGenericBlock) generic_sim_kernel(const __grid_constant__ GSimParams p) {
    const uint64_t t = counter_begin(p.cc);
    const RobotSpec &r = p.r;
    const int J = r.J, A = r.A;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < p.n; e += stride) {
        const uint64_t gid = p.gid_base + e;
        float q[kJointPad], qd[kJointPad];
        if (p.mode == 2) {
            g_draw_goal(r, p.keys, gid, t, p.sub, q);
            for (int k = 0; k < J; ++k) p.out_q[e * J + k] = q[k];
            continue;
        }
        uint32_t sf = p.step_flags[e];
        bool hold = true;
        if (p.mode == 1) {
            if (p.mask && !p.mask[e]) continue;
            sf = (sf & ROBOY_STEP_MASK) | ROBOY_F_HELD_ZERO64;  // _state = new_zero_state()
            p.step_flags[e] = sf;
        } else {
            // simulation_client.py:38 np.allclose(action, 0): |a| <= 1e-8 in float64, NaN fails
            for (int k = 0; k < A; ++k) hold = hold && (fabs((double)p.actions[e * A + k]) <= 1e-8);
        }
        bool feasible = true, is64 = false;
        if (hold) {
            const bool z = sf & ROBOY_F_HELD_ZERO64;
            is64 = z;
            for (int k = 0; k < J; ++k) {
                q[k] = z ? 0.0f : p.held[(uint64_t)k * p.n + e];
                qd[k] = z ? 0.0f : p.held[(uint64_t)(J + k) * p.n + e];
            }
            feasible = z || !(sf & ROBOY_F_HELD_INFEASIBLE);
            if (p.mode == 0) atomicAdd(p.stats + ROBOY_STAT_HOLDS, 1.0);
        } else {
            g_draw_state(r, p.keys, gid, t, q, qd);
        }
        if (p.out_q) {
            for (int k = 0; k < J; ++k) {
                p.out_q[e * J + k] = q[k];
                p.out_qd[e * J + k] = qd[k];
            }
            if (p.out_feasible) p.out_feasible[e] = (uint8_t)feasible | (is64 ? 2 : 0);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) counter_end(p.cc, t);
}

cudaError_t launch_generic_sim(const GSimParams &p, int sm_count, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    generic_sim_kernel<<<g_grid(p.n, sm_count), kGenericBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Env step / reset fed by an external simulator.  The wire values are float64 in the reference
// (python floats -> np.array), so the float64 branches of compute_reward / _did_reach_goal apply.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGenericBlock) generic_external_kernel(const __grid_constant__ GExternalParams p) {
    const uint64_t t = counter_begin(p.cc);
    const RobotSpec &r = p.r;
    const int J = r.J, D = 3 * J;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < p.n; e += stride) {
        if (p.reset && p.mask && !p.mask[e]) continue;
        const uint64_t gid = p.gid_base + e;
        float q[kJointPad], qd[kJointPad], g[kJointPad];
        for (int k = 0; k < J; ++k) {
            q[k] = p.q[e * J + k];
            qd[k] = p.qd[e * J + k];
            g[k] = p.goal[(uint64_t)k * p.n + e];
        }
        const bool feasible = p.feasible ? p.feasible[e] != 0 : true;
        // The reference's client builds the state with robot.new_state() (ros_simulation_client.py:40-46), which asserts the
        // angles inside the angle space (roboy_robot.py:76; closed interval, NaN fails; velocities are not checked, :77).
        // Like the other asserts it becomes an error bit and the batch goes on.
        bool bad_state = false;
        for (int k = 0; k < J; ++k) bad_state = bad_state || !(q[k] >= r.a_lo[k] && q[k] <= r.a_hi[k]);
        uint32_t sf = p.step_flags[e];
        bool new_goal = p.reset != 0;
        float *o = p.obs + e * D;
        if (bad_state && p.reset) {
            atomicOr(p.err_flags, ROBOY_ERR_STATE_BOUNDS);
            atomicMin(p.first_bad, (unsigned long long)gid);
        }
        if (!p.reset) {
            double rew;
            bool reached, violation;
            g_reward_reached(r, q, qd, true, feasible, g, nullptr, p.penalty != 0, p.bonus != 0, rew, reached, violation);
            uint32_t step = sf & ROBOY_STEP_MASK;
            step += step < ROBOY_STEP_MASK;                                   // roboy_env.py:60
            const bool done = reached || (int32_t)step > p.max_len;           // :65-66
            sf = step | (sf & ~ROBOY_STEP_MASK);
            p.reward[e] = (float)rew;
            p.done[e] = (uint8_t)done;
            new_goal = done;                                                  // :67-68
            atomicAdd(p.stats + ROBOY_STAT_STEPS, 1.0);
            atomicAdd(p.stats + ROBOY_STAT_SUM_REWARD, (double)(float)rew);
            if (done) {
                atomicAdd(p.stats + ROBOY_STAT_EPISODES, 1.0);
                atomicAdd(p.stats + (reached ? ROBOY_STAT_SUCCESSES : ROBOY_STAT_TIMEOUTS), 1.0);
                atomicAdd(p.stats + ROBOY_STAT_SUM_EPLEN, (double)(step - 1));
            }
            if (violation || bad_state) {
                atomicOr(p.err_flags, (violation ? ROBOY_ERR_REWARD_RANGE : 0u) | (bad_state ? ROBOY_ERR_STATE_BOUNDS : 0u));
                atomicMin(p.first_bad, (unsigned long long)gid);
                atomicAdd(p.stats + ROBOY_STAT_VIOLATIONS, 1.0);
            }
            for (int k = 0; k < J; ++k) { o[k] = q[k]; o[J + k] = qd[k]; o[2 * J + k] = g[k]; }  // :62 the goal in force
        } else {
            sf = 1u | (sf & ~ROBOY_STEP_MASK);                                // :85
        }
        if (new_goal) {
            g_draw_goal(r, p.keys, gid, t, 0, g);
            for (int k = 0; k < J; ++k) p.goal[(uint64_t)k * p.n + e] = g[k];
        }
        if (p.reset)                                                          // :86-87 obs carries the NEW goal
            for (int k = 0; k < J; ++k) { o[k] = q[k]; o[J + k] = qd[k]; o[2 * J + k] = g[k]; }
        p.step_flags[e] = sf;
    }
    __syncthreads();
    if (threadIdx.x == 0) counter_end(p.cc, t);
}

cudaError_t launch_generic_external(const GExternalParams &p, int sm_count, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    generic_external_kernel<<<g_grid(p.n, sm_count), kGenericBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace roboy
