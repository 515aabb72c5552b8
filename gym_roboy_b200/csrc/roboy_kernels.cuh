// Kernel parameter blocks and launcher prototypes shared by roboy_kernels.cu and roboy_capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "msj_math.cuh"
#include "philox.cuh"

namespace roboy {

constexpr int kStepBlock = 256;  // threads per CTA of the step kernel
constexpr int kWarpsPerBlock = kStepBlock / 32;
constexpr int kStepMinBlocks = 3;  // __launch_bounds__ min CTAs/SM (register cap)
constexpr int kObsDim = 9, kActDim = 8;

// The Philox call counter lives in device memory so that launches carry no host state and can be
// captured in CUDA graphs (closed-loop rollouts: policy + step, replayed many times).
//   kFixed    t = t_fixed (host supplied; the multi-stream host-buffer path, construction)
//   kAdvance  t = *t_dev + 1, and the LAST CTA of the launch to finish stores it back
//   kPeek     t = *t_dev (get_new_goal_joint_angles between steps)
//   kPeekNext t = *t_dev + 1 without storing it (the concurrent stages of the host-buffer pipeline; one
//             launch_counter_bump after them advances the counter)
struct CallCounter {
    enum Mode : int { kFixed = 0, kAdvance = 1, kPeek = 2, kPeekNext = 3 };
    unsigned long long *t_dev;
    unsigned int *cta_done;  // CTAs of the current launch that have finished
    unsigned long long t_fixed;
    int mode;
    unsigned int advance;    // how many counter values this launch consumes (T for a T-step rollout; else 1)
};

__device__ __forceinline__ uint64_t counter_begin(const CallCounter &c) {
    if (c.mode == CallCounter::kFixed) return c.t_fixed;
    const unsigned long long t = *reinterpret_cast<const volatile unsigned long long *>(c.t_dev);
    return c.mode == CallCounter::kPeek ? t : t + 1;
}

// Call once per CTA, by one thread, after the CTA's last use of the counter value.  Every CTA read
// *t_dev before it got here, and the store happens only after ALL CTAs got here.
__device__ __forceinline__ void counter_end(const CallCounter &c, uint64_t t) {
    if (c.mode != CallCounter::kAdvance) return;
    __threadfence();
    if (atomicAdd(c.cta_done, 1u) == gridDim.x - 1) {
        *c.cta_done = 0;
        *c.t_dev = t + (c.advance ? c.advance - 1 : 0);   // t is the FIRST value this launch used
    }
}

struct StepParams {
    uint64_t n;         // envs in this shard (= leading dimension of the SoA arrays)
    uint64_t e_begin;   // this launch covers local envs [e_begin, e_end); e_begin % 32 == 0
    uint64_t e_end;
    uint64_t gid_base;  // global id of local env 0
    CallCounter cc;     // Philox call counter of this launch
    PhiloxKeys keys;
    RobotConsts c;
    FastConsts f;
    float hold_mag;              // max(|hold_lo|, |hold_hi|): cheap pre-filter for the hold test
    float hold_c, hold_h;        // centre and (padded) half width of the hold interval: the pre-filter of robots whose
                                 // interval does not lie around 0 (kDivChecked instantiations)
    float hold_lo, hold_hi;      // the float32 interval of action components a for which
                                 // |fl(fl(slope*fl(a - in_hi)) + act_hi)| <= 1e-8, i.e. numpy's
                                 // allclose(rescaled, 0) (roboy_env.py:157-158, simulation_client.py:38)
    float act_in_hi, act_in_lo;  // RoboyEnv.action_space bounds, roboy_env.py:31
    float pad_[2];               // unread; without it the pointers below sit 8 bytes earlier and ptxas pairs their constant
                                 // loads differently in the step and open-loop kernels
    int32_t max_len;             // roboy_env.py:28
    int32_t obs_aligned;         // obs pointer is 16-byte aligned: vector / bulk stores allowed
    // inputs / state / outputs (device pointers)
    const float *__restrict__ actions;  // [n][8]
    float *__restrict__ goal;           // [3][n]
    float *__restrict__ goal1;          // goal + n, goal + 2n (row pointers, so an address is one IMAD.WIDE)
    float *__restrict__ goal2;
    uint32_t *__restrict__ step_flags;  // [n]
    const float *__restrict__ held;     // [6][n]
    float *__restrict__ obs;            // [n][9]
    float *__restrict__ reward;         // [n]
    uint8_t *__restrict__ done;         // [n]
    float *__restrict__ terminal_obs;   // [n][9] or nullptr
    uint32_t *__restrict__ done_bits;   // [ceil(n/32)] or nullptr: the done mask of this step as bits (bit l of word c = env 32c+l)
    double *__restrict__ stats;         // [ROBOY_STAT_COUNT]
    uint32_t *__restrict__ err_flags;
    unsigned long long *__restrict__ first_bad;
};

cudaError_t launch_null_step(uint64_t n_range, bool penalty, bool bonus, bool auto_reset, int fastdiv, int sm_count,
                             cudaStream_t stream);
cudaError_t launch_counter_bump(unsigned long long *t_dev, unsigned int advance, cudaStream_t stream);

struct LaunchGeom {
    int grid, block, smem;
};

LaunchGeom step_geometry(uint64_t n_range, bool penalty, bool bonus, bool auto_reset, int fastdiv, int sm_count);
cudaError_t launch_step(const StepParams &p, bool penalty, bool bonus, bool auto_reset, int fastdiv, int sm_count,
                        cudaStream_t stream);
// T consecutive steps on pre-recorded actions [T][n][8] -> obs [T][n][9], reward / done [T][n], with the
// env state held in registers across the T steps (open loop: 73 B per env-step instead of 93).
cudaError_t launch_step_many(const StepParams &p, uint32_t T, bool penalty, bool bonus, bool auto_reset, int fastdiv,
                             int sm_count, cudaStream_t stream);

// Generalised advantage estimation over rollout buffers [T][n] that the step kernel filled in place
// (the PPO2 runner of train_parallel.py:31-34 does this on the host; stable-baselines is external).
struct GaeParams {
    uint64_t T, n;
    const float *reward, *value;   // [T][n]
    const uint8_t *done;           // [T][n]  done[t] = episode ended AT step t
    const float *last_value;       // [n]     V(obs after the last step)
    float gamma, lam;
    float *adv, *ret;              // [T][n]
};
cudaError_t launch_gae(const GaeParams &p, int sm_count, cudaStream_t stream);

// Done-index list (roboy_env.py:65-68: which envs finished): the step kernel publishes its done mask as bits
// (StepParams::done_bits, one warp ballot per 32-env chunk); these two small kernels turn the words into the
// ascending list of env ids -- deterministic, no atomics on the output order:
//   count: per-tile popcounts (a tile = kDoneTileWords words = 32,768 envs); the last CTA to finish scans the tile sums
//   emit : every set bit writes its env id at tile offset + rank inside the tile, and (optionally) gathers that env's
//          pre-reset observation row into a packed [count][obs_dim] buffer (the vec-env `terminal_observation`s)
constexpr int kDoneTileWords = 1024;
struct DoneIndexParams {
    const uint32_t *bits;      // [n_words]
    uint32_t n_words;
    uint32_t n_envs;           // bits beyond n_envs in the last word are ignored
    uint32_t *tile_off;        // [n_tiles + 1] scratch: tile sums, then exclusive offsets
    unsigned int *ticket;      // zero between launches
    int32_t *idx;              // [capacity] out: ascending local env ids
    uint32_t capacity;
    uint32_t *count;           // out: number of done envs (may exceed capacity; only capacity entries are written)
    const float *terminal_obs; // [n][obs_dim] or nullptr
    float *terminal_rows;      // [capacity][obs_dim] or nullptr
    int obs_dim;
};
cudaError_t launch_done_index(const DoneIndexParams &p, cudaStream_t stream);

}  // namespace roboy
