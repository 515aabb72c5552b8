// Rare, divergent paths of one env-step, shared by the step kernels (roboy_kernels.cu) and the fused
// policy rollout kernel (roboy_policy.cu): the Stub's hold branch and the end of an episode.  Both are
// kept out of line so they stay out of the hot paths' register budgets.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/roboy_b200.h"
#include "roboy_kernels.cuh"

namespace roboy {
namespace {

struct HoldOut {
    float q0, q1, q2, qd0, qd1, qd2, reward;
    uint32_t flags;  // bit 0 reached, bit 1 violation
};

// Hold branch of the Stub (simulation_client.py:38-39): the stored state is returned.  Rare and
// divergent, so it is kept out of line and out of the hot path's register budget.
static __device__ __noinline__ HoldOut hold_branch(const StepParams &p, uint32_t e, uint32_t sf, float g0, float g1, float g2,
                                            bool penalty, bool bonus) {
    HeldState s;
    if (sf & ROBOY_F_HELD_ZERO64) {
#pragma unroll
        for (int k = 0; k < 3; ++k) s.q[k] = s.qd[k] = 0.0;
        s.is64 = true;
        s.feasible = true;
    } else {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            s.q[k] = (double)p.held[(size_t)k * p.n + e];
            s.qd[k] = (double)p.held[(size_t)(3 + k) * p.n + e];
        }
        s.is64 = false;
        s.feasible = !(sf & ROBOY_F_HELD_INFEASIBLE);
    }
    double r;
    bool reached, violation;
    const float g[3] = {g0, g1, g2};
    const float no_gqd[3] = {0.f, 0.f, 0.f};
    reward_reached_general(s, g, false, no_gqd, penalty, bonus, p.c, r, reached, violation);
    HoldOut o;
    o.q0 = (float)s.q[0]; o.q1 = (float)s.q[1]; o.q2 = (float)s.q[2];
    o.qd0 = (float)s.qd[0]; o.qd1 = (float)s.qd[1]; o.qd2 = (float)s.qd[2];
    o.reward = (float)r;
    o.flags = (reached ? 1u : 0u) | (violation ? 2u : 0u);
    return o;
}

// A CTA's episode counters in shared memory, 8-byte aligned: unsigned int [0..3] episodes, successes, holds, violations;
// [4..5] the low and high words of the 64-bit sum of episode lengths (one launch's episode ends in one CTA can add up to
// more than 2^32 steps: 257 envs at the 2^24 - 1 cap of the step counter do), read back as one little-endian 64-bit word.
constexpr int kCntWords = 6;
__device__ __forceinline__ unsigned long long *eplen_counter(unsigned int *s_cnt) {
    return reinterpret_cast<unsigned long long *>(s_cnt + 4);
}

// Everything an episode end needs, BY VALUE: the out-of-line function below must not touch the kernel's parameter block.
// (Handed a reference to it, the compiler addressed the block generically -- 25 generic loads for the round keys and the
// pointers plus 44 uniform-register moves, 211 instructions per call; with the values in registers and the round keys
// rebuilt from the two key words it is half that, and 7.7 % of the 32-env chunks make the call in the steady state.)
struct EpisodeEnd {
    uint64_t gid, t;
    uint32_t key0, key1;        // Philox key words (seed); round key r = key + r * W
    float a_lo, a_span24;
    float *goal0, *goal1, *goal2;  // this env's slots of the goal rows
    float *terminal_row;        // this env's row of the terminal-observation side buffer, or nullptr
    float *row;                 // this env's staged observation row (shared memory)
    unsigned int *s_cnt;        // the CTA's counters (layout above)
    uint32_t step;
    uint32_t reached_auto;      // bit 0 reached, bit 1 auto_reset
};

__device__ __forceinline__ EpisodeEnd episode_end(const StepParams &p, uint64_t t, uint32_t e, uint32_t step, bool reached,
                                                  bool auto_reset, float *row, unsigned int *s_cnt) {
    EpisodeEnd a;
    a.gid = p.gid_base + e;
    a.t = t;
    a.key0 = p.keys.k0[0];
    a.key1 = p.keys.k1[0];
    a.a_lo = p.c.a_lo;
    a.a_span24 = p.f.a_span24;
    a.goal0 = p.goal + e;
    a.goal1 = p.goal1 + e;
    a.goal2 = p.goal2 + e;
    a.terminal_row = p.terminal_obs ? p.terminal_obs + (size_t)e * kObsDim : nullptr;
    a.row = row;
    a.s_cnt = s_cnt;
    a.step = step;
    a.reached_auto = (reached ? 1u : 0u) | (auto_reset ? 2u : 0u);
    return a;
}

// Philox4x32-10 with the round keys rebuilt on the fly from the two key words (same bits as philox4x32_10 + PhiloxKeys)
__device__ __forceinline__ uint4 philox4x32_10_seed(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// Rare: an env finished its episode (:65-68) -- new goal, and under auto-reset the worker's
// reset() (:82-87).  Out of line: ~1/400 of env-steps.
static __device__ __noinline__ uint32_t finish_episode(const EpisodeEnd a) {
    // Under auto-reset the reference draws twice (:68 then :86) and only the second goal is ever
    // observable, so a single draw is materialised.
    const uint4 rg = philox4x32_10_seed((uint32_t)a.gid, (uint32_t)(a.gid >> 32), (uint32_t)a.t,
                                        (kStreamGoal << 28) | ((uint32_t)(a.t >> 32) & 0x000fffffu), a.key0, a.key1);
    const float ng0 = uniform_in24(rg.x, a.a_lo, a.a_span24);
    const float ng1 = uniform_in24(rg.y, a.a_lo, a.a_span24);
    const float ng2 = uniform_in24(rg.z, a.a_lo, a.a_span24);
    *a.goal0 = ng0;
    *a.goal1 = ng1;
    *a.goal2 = ng2;
    atomicAdd(&a.s_cnt[0], 1u);
    if (a.reached_auto & 1u) atomicAdd(&a.s_cnt[1], 1u);
    // episode length (steps since reset(): step_num starts at 1) into the 64-bit counter: a 32-bit add and, when it wraps,
    // the carry into the high word (a 64-bit atomicAdd through this generic pointer compiles to a compare-and-swap loop:
    // 193 instructions per call against 182)
    const uint32_t len = a.step - 1, lo = atomicAdd(&a.s_cnt[4], len);
    if (lo + len < lo) atomicAdd(&a.s_cnt[5], 1u);
    if (!(a.reached_auto & 2u)) return a.step | 0x80000000u;  // top bit: keep the flag bits
    float *row = a.row;
    if (a.terminal_row) {
#pragma unroll
        for (int k = 0; k < kObsDim; ++k) a.terminal_row[k] = row[k];
    }
    row[0] = row[1] = row[2] = row[3] = row[4] = row[5] = 0.0f;  // reset(): zero state, :83-84,87
    row[6] = ng0; row[7] = ng1; row[8] = ng2;
    return 1u;                                                   // :85, with the flags replaced
}

}  // namespace
}  // namespace roboy
