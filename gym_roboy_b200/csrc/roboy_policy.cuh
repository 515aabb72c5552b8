// Parameter blocks and launchers of the fused policy rollout kernels (roboy_policy.cu, roboy_policy_tc.cu,
// roboy_policy_generic.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/roboy_b200.h"
#include "roboy_generic.cuh"
#include "roboy_kernels.cuh"

namespace roboy {

constexpr int kPolicyMaxBlock = 256;
constexpr int kPolicyTcMaxBlock = 512;      // tensor-core variant: up to four 128-env tiles per CTA
constexpr int kPolicyTcImagePad = 15040;     // ROBOY_TC_IMAGE_BYTES rounded up to 128 bytes, in floats  // threads per CTA at most; one CTA per SM (shared memory bound)

struct PolicyParams {
    const float *__restrict__ image;  // [ROBOY_POLICY_IMAGE_FLOATS] packed policy (include/roboy_b200.h)
    uint32_t T;
    int32_t obs_aligned;              // every obs[t] slice is 16-byte aligned
    float *__restrict__ obs;          // [T+1][n][9]; slot 0 is the input, slots 1..T are written
    float *__restrict__ actions;      // [T][n][8]  un-clipped samples (what PPO2's runner stores)
    float *__restrict__ logp;         // [T][n]
    float *__restrict__ values;       // [T+1][n]
    float *__restrict__ noise;        // [T][n][8] or nullptr
    PhiloxKeys noise_keys;
    bool penalty, bonus, auto_reset, fastdiv;  // env flags, run-time in this kernel (filled by the launcher)
};

struct PolicyGeom {
    int grid, block, smem, envs_per_thread;
};

// envs_per_thread: 0 = choose (1 while every env fits on the chip at once, else 2)
PolicyGeom policy_geometry(uint64_t n_envs, int sm_count, int envs_per_thread);
// p: as for launch_step_many (reward / done are [T][n]; p.actions and p.obs are not used)
cudaError_t launch_policy_rollout(const StepParams &p, const PolicyParams &q, bool penalty, bool bonus, bool auto_reset,
                                  bool fastdiv, int sm_count, int envs_per_thread, cudaStream_t stream);

// tensor-core (tcgen05, TF32) variant: q.image is the ROBOY_TC_* image
// variant: 0 = choose; 1 = one 128-env tile per group of 128 threads; 2 = two tiles per group, ping-pong; 3 = merged
// (both networks of a tile advance together: small populations).  PolicyGeom::envs_per_thread returns the choice.
// exact: split-float16 operands (float32-level accuracy) instead of single float16 operands
PolicyGeom policy_tc_geometry(uint64_t n_envs, int sm_count, int tiles_per_group, bool exact);
cudaError_t launch_policy_rollout_tc(const StepParams &p, const PolicyParams &q, bool penalty, bool bonus, bool auto_reset,
                                     bool fastdiv, int sm_count, int tiles_per_group, bool exact, cudaStream_t stream);

// Float32 rollout for every robot the generic kernels take (roboy_policy_generic.cu): one env per thread, one
// instantiation per joint count; p is as for launch_generic_step (reward / done are [T][n]; p.actions and p.obs are not
// used), q.image is laid out by roboy_policy_layout (include/roboy_b200.h).
constexpr int kGPolicyMaxBlock = 256;
struct GPolicyParams {
    const float *__restrict__ image;
    uint32_t off[ROBOY_POLICY_LAYOUT_WORDS];   // roboy_policy_layout(3J, A)
    uint32_t T;
    int32_t obs_aligned;              // every obs[t] slice is 16-byte aligned
    float *__restrict__ obs;          // [T+1][n][3J]
    float *__restrict__ actions;      // [T][n][A]
    float *__restrict__ logp;         // [T][n]
    float *__restrict__ values;       // [T+1][n]
    float *__restrict__ noise;        // [T][n][A] or nullptr
    PhiloxKeys noise_keys;
};
// warps per CTA: min(8, chunks of 32 envs per SM).  The cap is kGPolicyMaxBlock / 32 = 8 (beyond 256 threads the
// register cap makes every joint count spill).  The shared-memory budget (227 KB minus the image, per warp a 64 x 32
// hidden column and a 32-row stage) is also applied, but never binds under that cap: 15 joints / 64 tendons, the
// largest image, still leaves room for 11 warps.
PolicyGeom generic_policy_geometry(int J, uint32_t image_floats, uint64_t n_envs, int sm_count);
cudaError_t launch_generic_policy_rollout(const GStepParams &p, const GPolicyParams &q, int sm_count, cudaStream_t stream);

// Deterministic policy evaluation for every robot (roboy_policy_eval.cu): the rollout's loop with the action
// clip(mean(obs), -1, 1), no value network and no per-step stores; each env's episodes are recorded as they finish.
// p is as for launch_generic_step (p.actions, p.obs, p.reward and p.done are not used).
struct GEvalParams {
    const float *__restrict__ image;  // the roboy_policy_layout(3J, A) image; only its policy net is read
    uint32_t off[ROBOY_POLICY_LAYOUT_WORDS];
    uint32_t T;
    uint32_t episodes;                // records per env (K)
    int32_t obs_aligned;              // obs is 16-byte aligned
    float *__restrict__ obs;          // [n][3J] in: the observation to start from; out: the one after the last step
    double *__restrict__ returns;     // [K][n]
    uint32_t *__restrict__ lengths;   // [K][n]
    uint8_t *__restrict__ reached;    // [K][n]
    uint32_t *__restrict__ completed; // [n]
};
cudaError_t launch_generic_policy_evaluate(const GStepParams &p, const GEvalParams &q, int sm_count, cudaStream_t stream);

// PPO2 minibatch gradient (roboy_ppo.cu) for every robot: one 64-sample tile at a time per CTA of 128 threads, one CTA per
// slot, slots = min(tiles, kPpoMaxSlots): a function of M only, so the partial sums and their order are too.
constexpr int kPpoTile = 64, kPpoThreads = 128, kPpoMaxSlots = 1184, kPpoAdvBlocks = 256, kPpoAdvThreads = 256;
struct PpoParams {
    const float *__restrict__ image;           // roboy_policy_layout(3J, A) image
    uint32_t off[ROBOY_POLICY_LAYOUT_WORDS];
    uint32_t P;                                // off[ROBOY_POLICY_LAYOUT_FLOATS]
    int J, A;
    uint64_t M, n_rows;
    const int64_t *__restrict__ index;         // [M]
    const float *__restrict__ obs;             // [n_rows][3J]
    const float *__restrict__ actions;         // [n_rows][A]
    const float *__restrict__ logp, *__restrict__ values, *__restrict__ ret;   // [n_rows]
    float clip, clip_vf, ent_coef, vf_coef;    // clip_vf < 0: no value clipping
    float *__restrict__ grad;                  // [P]
    double *__restrict__ stats;                // [ROBOY_PPO_STAT_COUNT]
    double *adv_part, *stat_part;              // workspace, carved by launch_ppo_grad
    float *grad_part;
};
uint32_t ppo_slots(uint64_t M);
uint64_t ppo_workspace_bytes(uint32_t P, uint64_t M);
cudaError_t launch_ppo_grad(PpoParams p, void *workspace, cudaStream_t stream);

}  // namespace roboy
