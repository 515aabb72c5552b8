// sm_100a kernels of the batched MSJ environment step.
//
// K1 step_kernel   RoboyEnv.step (envs/roboy_env.py:51-70) fused with the Stub simulation update
//                  (envs/simulations/simulation_client.py:36-40), normalisation
//                  (envs/robots/roboy_robot.py:80-95), compute_reward (:92-112), the done test
//                  (:65-66,:125-134), goal resampling (:117-123) and the vec-env reset-on-done.
// K2 construction / reset, the un-fused SimulationClient calls, state injection, stand-alone compute_reward and the
//    external-simulator feed are robot-generic kernels: roboy_generic.cu (this file is the MSJ-shaped hot step).
// K3 episode statistics are folded into K1's tail (warp reduce -> one atomic set per CTA).
//
// The path is elementwise and HBM-bound (93 algorithmic bytes, ~0.6 flop/B): no tensor cores.
// What matters is that every global access is a full-sector coalesced access:
//   * actions [n][8]: each warp reads its 32 envs' 1 KiB as 2 x LDG.128 per lane.  The Stub only
//     ever REDUCES the action (range assert + "all close to zero"), so no transpose is needed:
//     every lane tests the float4 it loaded and two warp ballots hand each env its verdict.
//   * goal / step_flags: structure of arrays, one 128 B line per warp access.
//   * obs [n][9] row-major (36 B rows): staged through shared memory so a warp emits its
//     1152 contiguous bytes as 72 x STG.128.
// The grid is persistent (a multiple of the SM count); statistics live in registers across the
// grid-stride loop, so the atomics are per CTA, not per env.
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>

#include "../../include/roboy_b200.h"
#include "roboy_kernels.cuh"
#include "step_rare.cuh"

namespace roboy {

namespace {

constexpr uint32_t kFull = 0xffffffffu;

// One chunk's state inputs (32 envs): goal and step word.  The chunk's 1 KiB of actions travels separately (Actions2):
// the actions are only ever reduced to two verdicts per env (in range? hold?).
struct ChunkIn {
    float g0, g1, g2;
    uint32_t sf;
    float ng0, ng1, ng2;  // normalised goal; only maintained by the open-loop kernel (KEEP_STATE)
};

// Local env indices are 32-bit (a shard holds < 2^32 envs: 4 Gi envs would need 400 GB of HBM);
// only the Philox counter uses the 64-bit global id.
template <bool TAIL>
__device__ __forceinline__ ChunkIn load_state(const StepParams &p, uint32_t base, int lane) {
    ChunkIn in;
    const uint32_t e = base + lane;
    if (!TAIL) {
        in.g0 = p.goal[e];
        in.g1 = p.goal1[e];
        in.g2 = p.goal2[e];
        in.sf = p.step_flags[e];
    } else {  // ragged tail: out-of-range slots read as neutral values
        const uint32_t n_end = (uint32_t)p.e_end;
        const bool live = e < n_end;
        in.g0 = live ? p.goal[e] : 0.f;
        in.g1 = live ? p.goal1[e] : 0.f;
        in.g2 = live ? p.goal2[e] : 0.f;
        in.sf = live ? p.step_flags[e] : 1u;
    }
    return in;
}

struct Actions2 {
    float4 a0, a1;
};
template <bool TAIL>
__device__ __forceinline__ Actions2 load_actions(const float *actions, uint32_t base, uint32_t n_end, int lane) {
    const float4 *a4 = reinterpret_cast<const float4 *>(actions) + (size_t)base * 2;
    // float4(*(a4 + i)), a by-value load, compiles to the machine code the timings in DESIGN.md were taken with; plain
    // a4[i] (nvcc 12.9) schedules the step and rollout kernels differently
    Actions2 a;
    if (!TAIL) {
        a.a0 = float4(*(a4 + lane));
        a.a1 = float4(*(a4 + 32 + lane));
    } else {
        const float4 z = make_float4(0.5f, 0.5f, 0.5f, 0.5f);  // ragged tail: in range, not "close to zero"
        a.a0 = (base * 2 + lane < n_end * 2) ? float4(*(a4 + lane)) : z;
        a.a1 = (base * 2 + 32 + lane < n_end * 2) ? float4(*(a4 + 32 + lane)) : z;
    }
    return a;
}

// max(|x|, |y|, |z|, |w|) that PROPAGATES NaN (fmaxf would drop it): one value answers both the range assert of
// roboy_env.py:52 (m <= 1; false for NaN) and the pre-filter of the hold test (m <= hold_mag).  Two FMNMX in SASS.
__device__ __forceinline__ float maxabs4_nan(const float4 &v) {
    float m;
    asm("{\n\t.reg .f32 ax, ay, az, aw, t;\n\t"
        "abs.f32 ax, %1;\n\tabs.f32 ay, %2;\n\tabs.f32 az, %3;\n\tabs.f32 aw, %4;\n\t"
        "max.NaN.f32 t, az, aw;\n\t"
        "max.NaN.f32 %0, ax, ay, t;\n\t}"
        : "=f"(m)
        : "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
    return m;
}

// simulation_client.py:38 on the rescaled action, exact: all four components inside [hold_lo, hold_hi]
__device__ __forceinline__ bool action_hold4_exact(const float4 &v, float lo, float hi) {
    return v.x >= lo && v.x <= hi && v.y >= lo && v.y <= hi && v.z >= lo && v.z <= hi && v.w >= lo && v.w <= hi;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// Where one step's outputs go: the handle's / caller's [n] buffers, or slot t of [T][n] rollout buffers.
struct OutPtrs {
    float *obs, *reward;
    uint8_t *done;
    bool obs_aligned;
};

// One env-step for the 32 envs of a chunk.  KEEP_STATE: the caller keeps the step word (and goal) in
// registers across several steps (open-loop rollout) instead of storing it per step.
// roboy_env.py:52 assert + simulation_client.py:38 allclose for the 32 envs of a chunk.
// Each lane tests the two float4 it loaded (float4 i belongs to env i / 2); env `lane` owns float4 2*lane and 2*lane+1
// of the chunk's 64.  The common case -- every action in range, none near zero -- costs two NaN-propagating max-abs,
// four compares and two votes for the whole warp; the per-env ballots run only when a vote says so.
// CENTRED: the hold interval lies around 0 (MSJ: rescaled = 0.05 * (a + 1) - 0.05 ... any tendon range symmetric about 0), so
// the max-abs doubles as its pre-filter.  Otherwise (a one-sided tendon range holds at a = -1) the pre-filter is the
// distance of each float4's first component from the centre of the interval.
template <bool CENTRED = true>
__device__ __forceinline__ void test_actions(const StepParams &p, const Actions2 &act, int lane, bool live, bool &act_ok_out,
                                             bool &hold_out) {
    const float m_a = maxabs4_nan(act.a0), m_b = maxabs4_nan(act.a1);
    bool act_ok = true, hold = false;
    if (!CENTRED) {
        if (!__all_sync(kFull, m_a <= p.act_in_hi && m_b <= p.act_in_hi)) {
            const uint32_t okm0 = __ballot_sync(kFull, m_a <= p.act_in_hi);
            const uint32_t okm1 = __ballot_sync(kFull, m_b <= p.act_in_hi);
            act_ok = (((lane < 16 ? okm0 : okm1) >> ((lane & 15) << 1)) & 3u) == 3u;
        }
        const bool near_a = fabsf(__fsub_rn(act.a0.x, p.hold_c)) <= p.hold_h, near_b = fabsf(__fsub_rn(act.a1.x, p.hold_c)) <= p.hold_h;
        if (__any_sync(kFull, near_a || near_b)) {
            const uint32_t hdm0 = __ballot_sync(kFull, near_a && action_hold4_exact(act.a0, p.hold_lo, p.hold_hi));
            const uint32_t hdm1 = __ballot_sync(kFull, near_b && action_hold4_exact(act.a1, p.hold_lo, p.hold_hi));
            hold = live && (((lane < 16 ? hdm0 : hdm1) >> ((lane & 15) << 1)) & 3u) == 3u;
        }
        act_ok_out = act_ok;
        hold_out = hold;
        return;
    }
    if (!__all_sync(kFull, m_a <= p.act_in_hi && m_b <= p.act_in_hi)) {   // somebody out of range or NaN: who?
        const uint32_t okm0 = __ballot_sync(kFull, m_a <= p.act_in_hi);
        const uint32_t okm1 = __ballot_sync(kFull, m_b <= p.act_in_hi);
        act_ok = (((lane < 16 ? okm0 : okm1) >> ((lane & 15) << 1)) & 3u) == 3u;
    }
    if (__any_sync(kFull, m_a <= p.hold_mag || m_b <= p.hold_mag)) {      // somebody near zero: exact interval test
        const uint32_t hdm0 = __ballot_sync(kFull, m_a <= p.hold_mag && action_hold4_exact(act.a0, p.hold_lo, p.hold_hi));
        const uint32_t hdm1 = __ballot_sync(kFull, m_b <= p.hold_mag && action_hold4_exact(act.a1, p.hold_lo, p.hold_hi));
        hold = live && (((lane < 16 ? hdm0 : hdm1) >> ((lane & 15) << 1)) & 3u) == 3u;
    }
    act_ok_out = act_ok;
    hold_out = hold;
}

template <bool PENALTY, bool BONUS, bool AUTO_RESET, int FASTDIV, bool TAIL, bool KEEP_STATE>
__device__ __forceinline__ uint32_t process_chunk(const StepParams &p, uint64_t t, const ChunkIn &cur, bool act_ok, bool hold,
                                                  uint32_t base, int lane, float *so, unsigned int *s_cnt, float &sum_reward,
                                                  const OutPtrs &out, bool &done_out) {
    const uint32_t e = base + lane;
    const bool live = TAIL ? (e < (uint32_t)p.e_end) : true;

    const float g0 = cur.g0, g1 = cur.g1, g2 = cur.g2;
    const uint32_t sf = cur.sf;
    float q0, q1, q2, qd0, qd1, qd2, reward;
    bool reached, violation;
    if (!hold) {
        // simulation_client.py:40 -> roboy_robot.py:35-39: fresh sample; velocities are drawn
        // from the ANGLE space too (reference quirk, :38)
        const Draw6 d = split6x21(philox_draw(p.gid_base + e, t, kStreamState, p.keys));
        q0 = uniform_in21(d.k[0], p.c.a_lo, p.f.a_span21);
        q1 = uniform_in21(d.k[1], p.c.a_lo, p.f.a_span21);
        q2 = uniform_in21(d.k[2], p.c.a_lo, p.f.a_span21);
        qd0 = uniform_in21(d.k[3], p.c.a_lo, p.f.a_span21);
        qd1 = uniform_in21(d.k[4], p.c.a_lo, p.f.a_span21);
        qd2 = uniform_in21(d.k[5], p.c.a_lo, p.f.a_span21);
        if (KEEP_STATE)
            reward_reached_sampled_ng<PENALTY, BONUS, FASTDIV>(q0, q1, q2, qd0, qd1, qd2, g0, g1, g2, cur.ng0, cur.ng1,
                                                               cur.ng2, p.c, p.f, reward, reached, violation);
        else
            reward_reached_sampled<PENALTY, BONUS, FASTDIV>(q0, q1, q2, qd0, qd1, qd2, g0, g1, g2, p.c, p.f, reward,
                                                            reached, violation);
    } else {
        const HoldOut h = hold_branch(p, e, sf, g0, g1, g2, PENALTY, BONUS);
        q0 = h.q0; q1 = h.q1; q2 = h.q2; qd0 = h.qd0; qd1 = h.qd1; qd2 = h.qd2;
        reward = h.reward;
        reached = h.flags & 1u;
        violation = h.flags & 2u;
        atomicAdd(&s_cnt[2], 1u);
    }

    uint32_t step = sf & ROBOY_STEP_MASK;
    step += step < ROBOY_STEP_MASK;                       // roboy_env.py:60
    const bool done = reached || (int32_t)step > p.max_len;  // :65-66, :72-73
    uint32_t word = step | (sf & ~ROBOY_STEP_MASK);

    // obs = [q, qd, goal] (:75-80), staged in shared memory; stride 9 is bank-conflict-free
    float *row = so + lane * kObsDim;
    row[0] = q0; row[1] = q1; row[2] = q2; row[3] = qd0; row[4] = qd1; row[5] = qd2;
    row[6] = g0; row[7] = g1; row[8] = g2;

    if (done && live) {
        // (tried: the whole warp rewriting its 128-byte goal lines instead of one lane's 4-byte partial-sector stores --
        // 0.9404 against 0.9461 of peak in the steady state, not kept)
        const uint32_t r = finish_episode(episode_end(p, t, e, step, reached, AUTO_RESET, row, s_cnt));
        word = (r & 0x80000000u) ? word : (r | ROBOY_F_HELD_ZERO64);
    }
    if (live && (violation || !act_ok)) {
        atomicOr(p.err_flags, (violation ? ROBOY_ERR_REWARD_RANGE : 0u) | (!act_ok ? ROBOY_ERR_ACTION : 0u));
        atomicMin(p.first_bad, (unsigned long long)(p.gid_base + e));
        atomicAdd(&s_cnt[3], 1u);
    }

    // ---- stores ----
    if (live) {
        if (!KEEP_STATE) p.step_flags[e] = word;
        out.reward[e] = reward;
        out.done[e] = (uint8_t)done;
        sum_reward += reward;
    }
    done_out = done;
    if (!KEEP_STATE && p.done_bits != nullptr) {  // done mask as bits for the done-index list (uniform branch)
        const uint32_t dm = __ballot_sync(kFull, done && live);
        if (lane == 0) p.done_bits[base >> 5] = dm;
    }
    if (!TAIL && out.obs_aligned) {
        // every lane publishes its shared-memory writes to the async proxy, then one lane hands the
        // warp's 1152 contiguous bytes to the bulk-copy engine (SASS: UBLKCP); the staging buffer is
        // double-buffered by the caller, so the copy drains while the next chunk is computed
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(so);
            float *dst = out.obs + (size_t)base * kObsDim;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src),
                         "n"(32 * kObsDim * 4)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        return word;
    }
    __syncwarp();
    if (!TAIL && out.obs_aligned) {
        float4 *dst = reinterpret_cast<float4 *>(out.obs + (size_t)base * kObsDim);  // 1152 B per chunk: 16 B aligned
        const float4 *src = reinterpret_cast<const float4 *>(so);
        dst[lane] = src[lane];
        dst[32 + lane] = src[32 + lane];
        if (lane < 8) dst[64 + lane] = src[64 + lane];
    } else {  // ragged tail, or a caller-supplied obs pointer that is only 4-byte aligned: scalar stores
        const uint32_t rows = TAIL ? (uint32_t)p.e_end - base : 32u;
        const uint32_t n_valid = rows * kObsDim;
        for (uint32_t i = lane; i < n_valid; i += 32) out.obs[(size_t)base * kObsDim + i] = so[i];
    }
    __syncwarp();
    return word;
}

}  // namespace

template <bool PENALTY, bool BONUS, bool AUTO_RESET, int FASTDIV>
__global__ void __launch_bounds__(kStepBlock, kStepMinBlocks) step_kernel(const __grid_constant__ StepParams p) {
    __shared__ __align__(128) float s_obs[2][kWarpsPerBlock][32 * kObsDim];
    __shared__ double s_red[kWarpsPerBlock];
    // rare events (done ~1/400 of env-steps, holds, violations) are counted with shared-memory
    // atomics where they happen instead of tying up registers in the hot loop
    __shared__ __align__(8) unsigned int s_cnt[kCntWords];  // done, success, hold, violation, sum of episode lengths (64-bit)
    if (threadIdx.x < kCntWords) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    // programmatic dependent launch: this grid may have been started while its predecessor in the stream (the policy
    // that produced the actions, or the previous step) was still draining; everything above overlapped with that.
    // From here on the predecessor's writes (actions, state, call counter) are complete and visible.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const uint64_t t = counter_begin(p.cc);
    const uint32_t n_full = (uint32_t)(p.e_end >> 5);  // chunks [chunk0, n_full) are complete
    const uint32_t warp_stride = gridDim.x * kWarpsPerBlock;
    float *so = s_obs[0][warp];
    uint32_t parity = 0;
    // per-thread reward sum: a thread adds at most a few hundred float32 rewards per launch, the
    // cross-thread reduction below is in double
    float sum_reward = 0.0f;
    const OutPtrs out{p.obs, p.reward, p.done, p.obs_aligned != 0};
    bool done_unused;

    uint32_t chunk = (uint32_t)(p.e_begin >> 5) + blockIdx.x * kWarpsPerBlock + warp;
    // Software prefetch into registers: the next chunk's loads are ISSUED FIRST, then this chunk is computed while they are
    // in flight.  (Testing this chunk's actions before issuing the next loads would save the eight-register copy, but the
    // warp then waits for its own data before it has the next request out: measured 1.5 % slower.)
    Actions2 acts;
    ChunkIn in;
    if (chunk < n_full) {
        acts = load_actions<false>(p.actions, chunk << 5, 0, lane);
        in = load_state<false>(p, chunk << 5, lane);
    }
    while (chunk < n_full) {
        const uint32_t next = chunk + warp_stride;
        const ChunkIn cur = in;
        const Actions2 cur_acts = acts;
        if (next < n_full) {
            acts = load_actions<false>(p.actions, next << 5, 0, lane);
            in = load_state<false>(p, next << 5, lane);
        }
        bool act_ok, hold;
        test_actions<FASTDIV != kDivChecked>(p, cur_acts, lane, true, act_ok, hold);
        // the bulk copy issued two chunks ago read this buffer: wait until at most one is still reading
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        so = s_obs[parity][warp];
        parity ^= 1;
        process_chunk<PENALTY, BONUS, AUTO_RESET, FASTDIV, false, false>(p, t, cur, act_ok, hold, chunk << 5, lane, so, s_cnt,
                                                                         sum_reward, out, done_unused);
        chunk = next;
    }
    // all bulk copies of this warp have completed; the ragged tail below stages in buffer 0
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncwarp();
    so = s_obs[0][warp];
    if (chunk == n_full && (p.e_end & 31)) {  // the ragged last chunk belongs to exactly one warp
        const Actions2 tail_acts = load_actions<true>(p.actions, chunk << 5, (uint32_t)p.e_end, lane);
        const ChunkIn cur = load_state<true>(p, chunk << 5, lane);
        bool act_ok, hold;
        test_actions<FASTDIV != kDivChecked>(p, tail_acts, lane, ((chunk << 5) + lane) < (uint32_t)p.e_end, act_ok, hold);
        process_chunk<PENALTY, BONUS, AUTO_RESET, FASTDIV, true, false>(p, t, cur, act_ok, hold, chunk << 5, lane, so, s_cnt,
                                                                        sum_reward, out, done_unused);
    }

    // ---- K3: episode statistics, one set of atomics per CTA ----
    const double w_reward = warp_sum((double)sum_reward);
    if (lane == 0) s_red[warp] = w_reward;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
#pragma unroll
        for (int w = 0; w < kWarpsPerBlock; ++w) r += s_red[w];
        const double done = (double)s_cnt[0], succ = (double)s_cnt[1];
        const double steps = blockIdx.x == 0 ? (double)(p.e_end - p.e_begin) : 0.0;
        const double v[ROBOY_STAT_COUNT] = {steps, done, succ, done - succ, r, (double)*eplen_counter(s_cnt),
                                            (double)s_cnt[2], (double)s_cnt[3]};
#pragma unroll
        for (int k = 0; k < ROBOY_STAT_COUNT; ++k)
            if (v[k] != 0.0) atomicAdd(p.stats + k, v[k]);
        counter_end(p.cc, t);
    }
}

// ---------------------------------------------------------------------------------------------
// Open-loop variant: T consecutive steps on pre-recorded actions.  A warp keeps its 32 envs' goal and
// step word in registers across the T steps, so per env-step only the action is read and obs /
// reward / done are written (73 B instead of 93).  Results are bit-identical to T step_kernel launches.
// ---------------------------------------------------------------------------------------------
// One chunk of 32 envs through T steps; the next step's actions are in flight while a step is computed.  A chunk switch used
// to cost one exposed memory latency (0.73 us per switch: 72 / 80 / 84 % of peak at T = 4 / 16 / 64).  During the LAST step of
// a chunk the action registers have no next step to hold, so the first actions of the warp's NEXT chunk (next_base, or
// kNoChunk) are loaded into them, and the next chunk's goal / step-word lines are prefetched into L2 (no registers).
// (Carrying the next chunk's state in registers as well spilled and lost 1.5 %.)
constexpr uint32_t kNoChunk = 0xffffffffu;

template <bool PENALTY, bool BONUS, bool AUTO_RESET, int FASTDIV, bool TAIL>
__device__ __forceinline__ void rollout_chunk(const StepParams &p, uint32_t T, uint64_t t_first, uint32_t base, int lane,
                                              float (*stage)[kWarpsPerBlock][32 * kObsDim], int warp, uint32_t &parity,
                                              unsigned int *s_cnt, float &sum_reward, Actions2 &acts, uint32_t next_base) {
    const uint32_t n_end = (uint32_t)p.e_end;
    const uint32_t e = base + lane;
    const bool live = TAIL ? e < n_end : true;
    ChunkIn cur = load_state<TAIL>(p, base, lane);
    cur.ng0 = normalize32_hot<FASTDIV>(cur.g0, p.c.a_hi, p.c.a_lo, p.c.a_span, p.f.a_rc);
    cur.ng1 = normalize32_hot<FASTDIV>(cur.g1, p.c.a_hi, p.c.a_lo, p.c.a_span, p.f.a_rc);
    cur.ng2 = normalize32_hot<FASTDIV>(cur.g2, p.c.a_hi, p.c.a_lo, p.c.a_span, p.f.a_rc);
    const size_t n = (size_t)p.n;
    for (uint32_t tt = 0; tt < T; ++tt) {
        const Actions2 cur_acts = acts;
        if (tt + 1 < T) {
            acts = load_actions<TAIL>(p.actions + (size_t)(tt + 1) * n * kActDim, base, n_end, lane);
        } else if (!TAIL && next_base != kNoChunk) {   // hand-over to the warp's next chunk
            acts = load_actions<false>(p.actions, next_base, n_end, lane);
            if (lane < 4) {
                const float *row = lane == 0 ? p.goal : lane == 1 ? p.goal1 : lane == 2 ? p.goal2
                                                                         : reinterpret_cast<const float *>(p.step_flags);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(row + next_base));
            }
        }
        bool act_ok, hold;
        test_actions<FASTDIV != kDivChecked>(p, cur_acts, lane, live, act_ok, hold);
        const OutPtrs out{p.obs + (size_t)tt * n * kObsDim, p.reward + (size_t)tt * n, p.done + (size_t)tt * n,
                          p.obs_aligned != 0};
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        float *so = stage[parity][warp];
        parity ^= 1;
        bool done;
        cur.sf = process_chunk<PENALTY, BONUS, AUTO_RESET, FASTDIV, TAIL, true>(p, t_first + tt, cur, act_ok, hold, base, lane, so,
                                                                                s_cnt, sum_reward, out, done);
        if (done && live) {  // rare: the new goal was stored by finish_episode (same thread)
            cur.g0 = p.goal[e];
            cur.g1 = p.goal1[e];
            cur.g2 = p.goal2[e];
            cur.ng0 = normalize32_hot<FASTDIV>(cur.g0, p.c.a_hi, p.c.a_lo, p.c.a_span, p.f.a_rc);
            cur.ng1 = normalize32_hot<FASTDIV>(cur.g1, p.c.a_hi, p.c.a_lo, p.c.a_span, p.f.a_rc);
            cur.ng2 = normalize32_hot<FASTDIV>(cur.g2, p.c.a_hi, p.c.a_lo, p.c.a_span, p.f.a_rc);
        }
    }
    if (live) p.step_flags[e] = cur.sf;
}

template <bool PENALTY, bool BONUS, bool AUTO_RESET, int FASTDIV>
__global__ void __launch_bounds__(kStepBlock, kStepMinBlocks) rollout_kernel(const __grid_constant__ StepParams p,
                                                                            const uint32_t T) {
    __shared__ __align__(128) float s_obs[2][kWarpsPerBlock][32 * kObsDim];
    __shared__ double s_red[kWarpsPerBlock];
    __shared__ __align__(8) unsigned int s_cnt[kCntWords];
    if (threadIdx.x < kCntWords) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const uint64_t t_first = counter_begin(p.cc);
    const uint32_t n_full = (uint32_t)(p.e_end >> 5);
    const uint32_t warp_stride = gridDim.x * kWarpsPerBlock;
    float sum_reward = 0.0f;
    uint32_t parity = 0;
    uint32_t chunk = (uint32_t)(p.e_begin >> 5) + blockIdx.x * kWarpsPerBlock + warp;
    Actions2 acts;
    if (chunk < n_full) acts = load_actions<false>(p.actions, chunk << 5, (uint32_t)p.e_end, lane);
    for (; chunk < n_full; chunk += warp_stride) {
        const uint32_t next = chunk + warp_stride;
        rollout_chunk<PENALTY, BONUS, AUTO_RESET, FASTDIV, false>(p, T, t_first, chunk << 5, lane, s_obs, warp, parity, s_cnt,
                                                                  sum_reward, acts, next < n_full ? next << 5 : kNoChunk);
    }
    if (chunk == n_full && (p.e_end & 31)) {
        acts = load_actions<true>(p.actions, chunk << 5, (uint32_t)p.e_end, lane);
        rollout_chunk<PENALTY, BONUS, AUTO_RESET, FASTDIV, true>(p, T, t_first, chunk << 5, lane, s_obs, warp, parity, s_cnt,
                                                                 sum_reward, acts, kNoChunk);
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    const double w_reward = warp_sum((double)sum_reward);
    if (lane == 0) s_red[warp] = w_reward;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
#pragma unroll
        for (int w = 0; w < kWarpsPerBlock; ++w) r += s_red[w];
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

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
namespace {

using StepKernelFn = void (*)(const StepParams);

template <int SEL>
StepKernelFn kernel_for() {
    return step_kernel<(SEL & 4) != 0, (SEL & 2) != 0, (SEL & 1) != 0, (SEL >> 3)>;
}

StepKernelFn select_kernel(int sel) {
    switch (sel) {
        case 0: return kernel_for<0>(); case 1: return kernel_for<1>();
        case 2: return kernel_for<2>(); case 3: return kernel_for<3>();
        case 4: return kernel_for<4>(); case 5: return kernel_for<5>();
        case 6: return kernel_for<6>(); case 7: return kernel_for<7>();
        case 8: return kernel_for<8>(); case 9: return kernel_for<9>();
        case 10: return kernel_for<10>(); case 11: return kernel_for<11>();
        case 12: return kernel_for<12>(); case 13: return kernel_for<13>();
        case 14: return kernel_for<14>(); case 15: return kernel_for<15>();
        case 16: return kernel_for<16>(); case 17: return kernel_for<17>();
        case 18: return kernel_for<18>(); case 19: return kernel_for<19>();
        case 20: return kernel_for<20>(); case 21: return kernel_for<21>();
        case 22: return kernel_for<22>(); case 23: return kernel_for<23>();
       
        default: return nullptr;
    }
}

// 24 instantiations: penalty x bonus x auto-reset x division mode (kDivIeee / kDivProved / kDivChecked)
int selector(bool penalty, bool bonus, bool auto_reset, int div_mode) {
    return (div_mode << 3) | (penalty ? 4 : 0) | (bonus ? 2 : 0) | (auto_reset ? 1 : 0);
}

int blocks_per_sm(int sel) {
    static int cached[24] = {0};
    if (!cached[sel]) {
        int b = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, select_kernel(sel), kStepBlock, 0) != cudaSuccess || b < 1)
            b = 1;
        if (b > kStepMinBlocks) b = kStepMinBlocks;
        cached[sel] = b;
    }
    return cached[sel];
}

int grid_for(uint64_t n_range, int per_sm, int sm_count) {
    const uint64_t n_chunks = (n_range + 31) / 32;
    const uint64_t want = (n_chunks + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const uint64_t cap = (uint64_t)sm_count * per_sm;  // persistent: a multiple of the SM count
    return (int)(want < cap ? want : cap);
}

using RolloutKernelFn = void (*)(const StepParams, const uint32_t);

template <int SEL>
RolloutKernelFn rollout_for() {
    return rollout_kernel<(SEL & 4) != 0, (SEL & 2) != 0, (SEL & 1) != 0, (SEL >> 3)>;
}

RolloutKernelFn select_rollout(int sel) {
    switch (sel) {
        case 0: return rollout_for<0>(); case 1: return rollout_for<1>();
        case 2: return rollout_for<2>(); case 3: return rollout_for<3>();
        case 4: return rollout_for<4>(); case 5: return rollout_for<5>();
        case 6: return rollout_for<6>(); case 7: return rollout_for<7>();
        case 8: return rollout_for<8>(); case 9: return rollout_for<9>();
        case 10: return rollout_for<10>(); case 11: return rollout_for<11>();
        case 12: return rollout_for<12>(); case 13: return rollout_for<13>();
        case 14: return rollout_for<14>(); case 15: return rollout_for<15>();
        case 16: return rollout_for<16>(); case 17: return rollout_for<17>();
        case 18: return rollout_for<18>(); case 19: return rollout_for<19>();
        case 20: return rollout_for<20>(); case 21: return rollout_for<21>();
        case 22: return rollout_for<22>(); case 23: return rollout_for<23>();
       
        default: return nullptr;
    }
}

}  // namespace

cudaError_t launch_step_many(const StepParams &p, uint32_t T, bool penalty, bool bonus, bool auto_reset, int fastdiv,
                             int sm_count, cudaStream_t stream) {
    if (p.e_end <= p.e_begin || T == 0) return cudaSuccess;
    const int sel = selector(penalty, bonus, auto_reset, fastdiv);
    static int per_sm[24] = {0};
    if (!per_sm[sel]) {
        int b = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, select_rollout(sel), kStepBlock, 0) != cudaSuccess || b < 1) b = 1;
        if (b > kStepMinBlocks) b = kStepMinBlocks;
        per_sm[sel] = b;
    }
    const int grid = grid_for(p.e_end - p.e_begin, per_sm[sel], sm_count);
    select_rollout(sel)<<<grid, kStepBlock, 0, stream>>>(p, T);
    return cudaGetLastError();
}

LaunchGeom step_geometry(uint64_t n_range, bool penalty, bool bonus, bool auto_reset, int fastdiv, int sm_count) {
    const int sel = selector(penalty, bonus, auto_reset, fastdiv);
    return LaunchGeom{grid_for(n_range, blocks_per_sm(sel), sm_count), kStepBlock,
                      (int)(sizeof(float) * kWarpsPerBlock * 32 * kObsDim + sizeof(double) * kWarpsPerBlock * ROBOY_STAT_COUNT)};
}

cudaError_t launch_step(const StepParams &p, bool penalty, bool bonus, bool auto_reset, int fastdiv, int sm_count,
                        cudaStream_t stream) {
    if (p.e_end <= p.e_begin) return cudaSuccess;
    const int sel = selector(penalty, bonus, auto_reset, fastdiv);
    const int grid = grid_for(p.e_end - p.e_begin, blocks_per_sm(sel), sm_count);
    static const bool pdl = [] {   // ROBOY_B200_PDL=0 in the environment turns the launch attribute off (A/B measurements)
        const char *v = getenv("ROBOY_B200_PDL");
        return !(v && v[0] == '0');
    }();
    if (!pdl) {
        select_kernel(sel)<<<grid, kStepBlock, 0, stream>>>(p);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kStepBlock);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, select_kernel(sel), p);
}

__global__ void counter_bump_kernel(unsigned long long *t_dev, unsigned int advance) { *t_dev += advance; }

cudaError_t launch_counter_bump(unsigned long long *t_dev, unsigned int advance, cudaStream_t stream) {
    counter_bump_kernel<<<1, 1, 0, stream>>>(t_dev, advance);
    return cudaGetLastError();
}

// Measurement only: an EMPTY kernel launched exactly like the step kernel (same grid, block, programmatic-dependent-launch
// attribute) -- the launch floor bench.py prints next to the launch-bound sizes.
__global__ void __launch_bounds__(kStepBlock) null_step_kernel() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

cudaError_t launch_null_step(uint64_t n_range, bool penalty, bool bonus, bool auto_reset, int fastdiv, int sm_count,
                             cudaStream_t stream) {
    const int sel = selector(penalty, bonus, auto_reset, fastdiv);
    const int grid = grid_for(n_range, blocks_per_sm(sel), sm_count);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kStepBlock);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, null_step_kernel);
}

// ---------------------------------------------------------------------------------------------
// Rollout consumer: GAE(lambda) over [T][n] buffers, one thread per env walking t backwards
// (all accesses coalesced across envs).  delta_t = r_t + gamma*V_{t+1}*(1-done_t) - V_t;
// A_t = delta_t + gamma*lam*(1-done_t)*A_{t+1};  R_t = A_t + V_t.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gae_kernel(const __grid_constant__ GaeParams p) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < p.n; e += stride) {
        float next_v = p.last_value[e];
        float gae = 0.0f;
        for (uint64_t t = p.T; t-- > 0;) {
            const size_t i = (size_t)t * p.n + e;
            const float nonterminal = p.done[i] ? 0.0f : 1.0f;
            const float v = p.value[i];
            const float delta = p.reward[i] + p.gamma * next_v * nonterminal - v;
            gae = delta + p.gamma * p.lam * nonterminal * gae;
            p.adv[i] = gae;
            p.ret[i] = gae + v;
            next_v = v;
        }
    }
}

cudaError_t launch_gae(const GaeParams &p, int sm_count, cudaStream_t stream) {
    if (p.n == 0 || p.T == 0) return cudaSuccess;
    const uint64_t want = (p.n + 255) / 256;
    const int grid = (int)(want < (uint64_t)sm_count * 8 ? want : (uint64_t)sm_count * 8);
    gae_kernel<<<grid, 256, 0, stream>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Done-index list: ascending env ids of the envs that finished in the last step (roboy_env.py:65-68),
// from the bit mask the step kernel published.  Two tiny launches (2 MB of mask words at 16,777,216 envs).
// ---------------------------------------------------------------------------------------------
namespace {
constexpr int kDoneBlock = 256;
constexpr int kDoneWordsPerThread = kDoneTileWords / kDoneBlock;  // 4 consecutive words per thread

__device__ __forceinline__ uint32_t done_word(const DoneIndexParams &p, uint32_t w) {
    if (w >= p.n_words) return 0u;
    uint32_t v = p.bits[w];
    const uint32_t rem = p.n_envs - w * 32u;  // envs covered by this word
    if (rem < 32u) v &= (1u << rem) - 1u;
    return v;
}

// exclusive prefix sum of one value per thread over the CTA; `total` gets the CTA sum
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *s_warp, uint32_t &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kDoneBlock / 32; ++w) {
        const uint32_t x = s_warp[w];
        if (w < warp) base += x;
        tot += x;
    }
    __syncthreads();
    total = tot;
    return base + inc - v;
}
}  // namespace

__global__ void __launch_bounds__(kDoneBlock) done_count_kernel(const __grid_constant__ DoneIndexParams p) {
    __shared__ uint32_t s_warp[kDoneBlock / 32];
    __shared__ bool s_last;
    const uint32_t w0 = (blockIdx.x * kDoneBlock + threadIdx.x) * kDoneWordsPerThread;
    uint32_t c = 0;
#pragma unroll
    for (int k = 0; k < kDoneWordsPerThread; ++k) c += __popc(done_word(p, w0 + k));
    uint32_t total;
    block_exclusive_scan(c, s_warp, total);
    if (threadIdx.x == 0) {
        p.tile_off[blockIdx.x] = total;
        __threadfence();
        s_last = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    // last CTA: exclusive scan of the tile sums in place (tile order = env order), total -> *count
    __threadfence();
    uint32_t carry = 0;
    for (uint32_t b = 0; b < gridDim.x; b += kDoneBlock) {
        const uint32_t i = b + threadIdx.x;
        const uint32_t v = i < gridDim.x ? *reinterpret_cast<volatile uint32_t *>(p.tile_off + i) : 0u;
        uint32_t tot;
        const uint32_t ex = block_exclusive_scan(v, s_warp, tot);
        if (i < gridDim.x) p.tile_off[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) {
        p.tile_off[gridDim.x] = carry;
        *p.count = carry;
        *p.ticket = 0;
    }
}

__global__ void __launch_bounds__(kDoneBlock) done_emit_kernel(const __grid_constant__ DoneIndexParams p) {
    __shared__ uint32_t s_warp[kDoneBlock / 32];
    const uint32_t w0 = (blockIdx.x * kDoneBlock + threadIdx.x) * kDoneWordsPerThread;
    uint32_t word[kDoneWordsPerThread];
    uint32_t c = 0;
#pragma unroll
    for (int k = 0; k < kDoneWordsPerThread; ++k) {
        word[k] = done_word(p, w0 + k);
        c += __popc(word[k]);
    }
    uint32_t total;
    uint32_t pos = p.tile_off[blockIdx.x] + block_exclusive_scan(c, s_warp, total);
    if (c == 0) return;
#pragma unroll
    for (int k = 0; k < kDoneWordsPerThread; ++k) {
        uint32_t m = word[k];
        while (m) {
            const uint32_t b = __ffs(m) - 1;
            m &= m - 1;
            if (pos < p.capacity) {
                const uint32_t e = (w0 + k) * 32u + b;
                p.idx[pos] = (int32_t)e;
                if (p.terminal_rows)
                    for (int j = 0; j < p.obs_dim; ++j)
                        p.terminal_rows[(size_t)pos * p.obs_dim + j] = p.terminal_obs[(size_t)e * p.obs_dim + j];
            }
            ++pos;
        }
    }
}

cudaError_t launch_done_index(const DoneIndexParams &p, cudaStream_t stream) {
    if (p.n_words == 0) return cudaSuccess;
    const int grid = (int)((p.n_words + kDoneTileWords - 1) / kDoneTileWords);
    done_count_kernel<<<grid, kDoneBlock, 0, stream>>>(p);
    done_emit_kernel<<<grid, kDoneBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace roboy
