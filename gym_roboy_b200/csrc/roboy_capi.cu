// C-ABI of the B200-native batched MSJ env step (see include/roboy_b200.h for the contract and
// the reference lines each entry point replaces).  Host side only: handle, HBM allocation,
// launch bookkeeping, the pinned/pipelined host-buffer path and DLPack export.
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <atomic>
#include <new>

#include "../../include/roboy_b200.h"
#include "dlpack_min.h"
#include "roboy_generic.cuh"
#include "roboy_kernels.cuh"
#include "roboy_policy.cuh"

using namespace roboy;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            return fail(ROBOY_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

constexpr int kHostStreamsMax = 8;         // ring of streams for the host-buffer pipeline
constexpr int kHostStreamsDefault = 2;                // ring of two streams, each stage entirely on one of them (measured best)
constexpr uint64_t kHostStageEnvsDefault = 1u << 19;  // 524,288 envs per pipeline stage (16 MiB in, 20.5 MiB out)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
        if (prev == dev) prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// roboy_env.py:24-25 _l2_distance(space.low, space.high) in float32, numpy evaluation order
// (float32 products accumulated in double, rounded to float32, float32 sqrt).
float box_diagonal_f32(const float *lo, const float *hi, int dim) {
    double s = 0.0;
    for (int k = 0; k < dim; ++k) {
        volatile float d = lo[k] - hi[k];
        volatile float p = d * d;
        s += (double)p;
    }
    return sqrtf((float)s);
}

// ---- host-side derivation of the hot path's constants (config time, not the data path) ----
uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
// order-preserving map float32 -> uint32 (for bisection over floats)
uint32_t fkey(float f) { const uint32_t u = f2u(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
float fkey_inv(uint32_t k) { return u2f((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// roboy_env.py:157-158 in float32, unfused: slope*(a - in_hi) + out_hi
float rescale_f32(float a, float in_hi, float slope, float act_hi) {
    volatile float r = a - in_hi;
    r = slope * r;
    r = r + act_hi;
    return r;
}

// The set of action components a whose rescaled value passes numpy's allclose(., 0) (|x| <= 1e-8,
// simulation_client.py:38).  rescale is monotone non-decreasing in a, so the set is an interval of floats; both ends by
// bisection over EVERY finite float32, not just [-1, 1]: an action outside the action space fails the assert of
// roboy_env.py:52 (error word), but the batch goes on, and what the Stub then does with that env is what numpy would do
// under `python -O` -- a one-sided tendon range [0, hi] holds at a = -1, and a = -1.0000001 rescales to within 1e-8 of
// zero as well (tools/soak_parity.py found the oracle holding there and the kernels not).  Empty -> lo > hi.
void hold_interval(float in_hi, float slope, float act_hi, float *lo, float *hi) {
    const double tol = 1e-8;
    const uint32_t a = fkey(-FLT_MAX), b = fkey(FLT_MAX);
    // smallest a with rescale(a) >= -tol
    uint32_t l = a, r = b;
    if (!((double)rescale_f32(FLT_MAX, in_hi, slope, act_hi) >= -tol)) { *lo = 1.f; *hi = -1.f; return; }
    while (l < r) {
        const uint32_t m = l + (r - l) / 2;
        if ((double)rescale_f32(fkey_inv(m), in_hi, slope, act_hi) >= -tol) r = m; else l = m + 1;
    }
    const float first = fkey_inv(l);
    // largest a with rescale(a) <= tol
    l = a; r = b;
    if (!((double)rescale_f32(-FLT_MAX, in_hi, slope, act_hi) <= tol)) { *lo = 1.f; *hi = -1.f; return; }
    while (l < r) {
        const uint32_t m = l + (r - l + 1) / 2;
        if ((double)rescale_f32(fkey_inv(m), in_hi, slope, act_hi) <= tol) l = m; else r = m - 1;
    }
    const float last = fkey_inv(l);
    if (first > last) { *lo = 1.f; *hi = -1.f; return; }
    *lo = first;
    *hi = last;
}

float round_up_f32(double x) {
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
}
float round_down_f32(double x) {
    float f = (float)x;
    if ((double)f > x) f = nextafterf(f, -INFINITY);
    return f;
}

// The 3-instruction division of the sampled-state path is proved bit-exact (oracle/verify_fastdiv.c)
// for the MSJ spans only: 2*pi_f32 (0x40c90fdb) and (pi/3)_f32 (0x3f860a92).
bool spans_are_proved(float a_lo, float a_hi, float v_lo, float v_hi) {
    return f2u(a_hi - a_lo) == 0x40c90fdbu && a_lo == -a_hi && f2u(v_hi - v_lo) == 0x3f860a92u && v_lo == -v_hi;
}

int cfg_dim_joint(const roboy_cfg &c) { return c.dim_joint > 0 ? c.dim_joint : ROBOY_DIM_JOINT; }
int cfg_dim_action(const roboy_cfg &c) { return c.dim_action > 0 ? c.dim_action : ROBOY_DIM_ACTION; }

// The robot's spaces as per-component arrays, whichever way the caller gave them
void fill_robot_spec(const roboy_cfg &c, RobotSpec &r) {
    memset(&r, 0, sizeof(r));
    r.J = cfg_dim_joint(c);
    r.A = cfg_dim_action(c);
    for (int k = 0; k < r.J; ++k) {
        r.a_lo[k] = c.per_component_bounds ? c.angle_low_v[k] : c.angle_low;
        r.a_hi[k] = c.per_component_bounds ? c.angle_high_v[k] : c.angle_high;
        r.v_lo[k] = c.per_component_bounds ? c.vel_low_v[k] : c.vel_low;
        r.v_hi[k] = c.per_component_bounds ? c.vel_high_v[k] : c.vel_high;
    }
    for (int k = 0; k < r.A; ++k) {
        const float lo = c.per_component_bounds ? c.act_low_v[k] : c.act_low;
        const float hi = c.per_component_bounds ? c.act_high_v[k] : c.act_high;
        const float slope = (hi - lo) / (1.0f - (-1.0f));  // roboy_env.py:157, float32, per component
        hold_interval(1.0f, slope, hi, &r.hold_lo[k], &r.hold_hi[k]);
    }
    r.thr_angle = box_diagonal_f32(r.a_lo, r.a_hi, r.J) / 200.0f;  // roboy_env.py:127
    r.thr_vel = box_diagonal_f32(r.v_lo, r.v_hi, r.J) / 5.0f;      // roboy_env.py:130
    r.penalty_boundary = fabsf(c.penalty_boundary);
    r.bonus_goal = c.bonus_goal;
    r.reward_lo = c.reward_lo;
    r.reward_hi = c.reward_hi;
    // constants of the fused generic step, each the value the kernel would otherwise recompute per env-step
    for (int k = 0; k < r.J; ++k) {
        volatile float sa = r.a_hi[k] - r.a_lo[k], sv = r.v_hi[k] - r.v_lo[k];   // float32 - float32 (roboy_robot.py:95)
        r.a_span[k] = sa;
        r.v_span[k] = sv;
        volatile float s21 = sa * 0x1p-21f;
        r.a_span21[k] = s21;
        volatile double t = 2.0 * 0.0;     // (2*0 - max - min) / (max - min) in float64, the goal's zero velocity (roboy_env.py:23)
        t = t - (double)r.v_hi[k];
        t = t - (double)r.v_lo[k];
        r.v_gz[k] = t / (double)sv;
    }
    r.thr_angle_sq_hi = round_up_f32((double)r.thr_angle * (double)r.thr_angle * (1.0 + 1e-5));
    {   // hull of the hold intervals: the whole-chunk pre-filter of the hold test
        float lo = INFINITY, hi = -INFINITY;
        bool possible = true;
        for (int k = 0; k < r.A; ++k) {
            if (!(r.hold_lo[k] <= r.hold_hi[k])) possible = false;
            lo = fminf(lo, r.hold_lo[k]);
            hi = fmaxf(hi, r.hold_hi[k]);
        }
        if (!possible) {
            r.hold_c = 0.0f;
            r.hold_h = -1.0f;
            r.hold_pad = 0.0f;
        } else {
            const double c0 = 0.5 * ((double)lo + (double)hi), h0 = 0.5 * ((double)hi - (double)lo);
            r.hold_c = (float)c0;
            r.hold_h = round_up_f32(h0 * 1.001 + fabs(c0) * 1e-6 + 1e-30);   // covers the rounding of hold_c and of x - hold_c
            r.hold_pad = c0 <= 0.0 ? 1.0f : -1.0f;   // farthest end of [-1, 1]: outside the hull unless the hull spans it
        }
    }
}

// MSJ's dims and the same bounds on every component: the tuned kernels apply
bool is_msj_shaped(const roboy_cfg &c, const RobotSpec &r) {
    if (r.J != ROBOY_DIM_JOINT || r.A != ROBOY_DIM_ACTION) return false;
    for (int k = 1; k < r.J; ++k)
        if (r.a_lo[k] != r.a_lo[0] || r.a_hi[k] != r.a_hi[0] || r.v_lo[k] != r.v_lo[0] || r.v_hi[k] != r.v_hi[0]) return false;
    if (c.per_component_bounds)
        for (int k = 1; k < r.A; ++k)
            if (c.act_low_v[k] != c.act_low_v[0] || c.act_high_v[k] != c.act_high_v[0]) return false;
    return true;
}

const char *check_robot(const roboy_cfg &c) {
    const int J = cfg_dim_joint(c), A = cfg_dim_action(c);
    if (J < 1 || J > ROBOY_MAX_JOINT) return "dim_joint must be 1..15 (numpy sums longer vectors in a CPU-dependent order)";
    if (A < 1 || A > ROBOY_MAX_ACTION) return "dim_action must be 1..64";
    for (int k = 0; k < J; ++k) {
        const float al = c.per_component_bounds ? c.angle_low_v[k] : c.angle_low, ah = c.per_component_bounds ? c.angle_high_v[k] : c.angle_high;
        const float vl = c.per_component_bounds ? c.vel_low_v[k] : c.vel_low, vh = c.per_component_bounds ? c.vel_high_v[k] : c.vel_high;
        if (!(ah > al) || !(vh > vl)) return "empty robot space";
        // ptxas evaluates fl(fl(2*v) - max) of the normalisation (roboy_robot.py:95) as fma(2, v, -max) -- the same bits for
        // every float32 v as long as |max| < 2^103 (oracle/verify_fused_numerator.c); bounds that large are not joint limits
        if (!(fabsf(al) < 0x1p100f && fabsf(ah) < 0x1p100f && fabsf(vl) < 0x1p100f && fabsf(vh) < 0x1p100f))
            return "robot space bounds must be below 2^100 in magnitude";
    }
    for (int k = 0; k < A; ++k) {
        const float tl = c.per_component_bounds ? c.act_low_v[k] : c.act_low, th = c.per_component_bounds ? c.act_high_v[k] : c.act_high;
        if (!(th > tl)) return "empty robot space";
    }
    return nullptr;
}

}  // namespace

struct roboy_env {
    roboy_cfg cfg;
    int device = 0;
    int sm_count = 148;
    std::atomic<int> refs{1};
    // The Philox call counter is DEVICE state (t_dev): kernels read it and the last CTA of an
    // advancing launch bumps it, so launches carry no host state and are CUDA-graph capturable.
    unsigned long long *t_dev = nullptr;
    unsigned int *cta_done = nullptr;
    uint32_t goal_sub = 0;  // goal draws already made at this call counter (un-fused API)
    uint64_t launches = 0;  // kernels launched through this handle
    PhiloxKeys keys;
    RobotSpec spec;         // the robot, per component: the one description of it (tune_step_params reads component 0)
    int J = ROBOY_DIM_JOINT, A = ROBOY_DIM_ACTION, D = ROBOY_DIM_OBS;
    bool msj_shaped = true;  // MSJ's dims with uniform bounds: the tuned step / rollout kernels apply
    int fastdiv = kDivIeee;      // division mode of the tuned MSJ-shaped kernels (msj_math.cuh): IEEE / proved offline / proved at create
    // HBM
    float *goal = nullptr;
    uint32_t *step_flags = nullptr;
    float *held = nullptr;
    float *obs = nullptr;
    float *reward = nullptr;
    uint8_t *done = nullptr;
    double *stats = nullptr;
    uint32_t *err_flags = nullptr;
    unsigned long long *first_bad = nullptr;
    float *terminal_obs = nullptr;  // caller-owned
    // host-buffer pipeline (lazily created)
    float *actions_stage = nullptr;  // device copy of the host actions
    cudaStream_t hs[kHostStreamsMax] = {};
    int host_streams = kHostStreamsDefault;
    uint64_t host_stage_envs = kHostStageEnvsDefault;
    bool host_ready = false;
    cudaEvent_t hev[kHostStreamsMax] = {};
    bool host_ramp = true;  // shorter first stages (pipeline fill)
    int host_pattern = ROBOY_HOST_PATTERN_RING;
    // Stream count of the ring, tuned by measurement unless the caller fixed it (roboy_set_host_pipeline): one GPU on
    // its own PCIe link wants two streams (both copy engines busy), eight GPUs saturating the host's memory path want one
    // (72.5 against 77.3 ms per pass).  Calls 2 and 3 time the two candidates, the faster one is kept.
    bool host_autotune = true;
    int host_calls = 0;
    double host_ms[2] = {0.0, 0.0};
    int host_mode = 0;  // ROBOY_HOST_STAGED / ROBOY_HOST_MAPPED_OUT / ROBOY_HOST_MAPPED_ALL
    // done-index list (lazily allocated by roboy_enable_done_index)
    uint32_t *done_bits = nullptr;
    uint32_t *done_tile_off = nullptr;
    unsigned int *done_ticket = nullptr;
};

namespace {

void free_env(roboy_env *e) {
    DeviceGuard g(e->device);
    cudaFree(e->goal);
    cudaFree(e->step_flags);
    cudaFree(e->held);
    cudaFree(e->obs);
    cudaFree(e->reward);
    cudaFree(e->done);
    cudaFree(e->stats);
    cudaFree(e->err_flags);
    cudaFree(e->first_bad);
    cudaFree(e->t_dev);
    cudaFree(e->cta_done);
    cudaFree(e->actions_stage);
    cudaFree(e->done_bits);
    cudaFree(e->done_tile_off);
    cudaFree(e->done_ticket);
    if (e->host_ready)
        for (int i = 0; i < kHostStreamsMax; ++i) {
            cudaStreamDestroy(e->hs[i]);
            cudaEventDestroy(e->hev[i]);
        }
    delete e;
}

void unref(roboy_env *e) {
    if (e->refs.fetch_sub(1) == 1) free_env(e);
}

// PenaltyF32 (msj_math.cuh): whether the float32 evaluation of roboy_env.py:98-100 applies is a property of the robot;
// its fall-back band follows the current reward_range (roboy_create, roboy_set_reward_range).
// ROBOY_B200_PENALTY_F64=1 keeps every handle on the float64 expression (A/B runs, the bit-equality test).
void set_penalty_f32(roboy_env *e) {
    const RobotSpec &r = e->spec;
    PenaltyF32 pen{};
    const char *off = getenv("ROBOY_B200_PENALTY_F64");
    bool ok = r.J <= 8 && !(off && off[0] == '1');
    for (int k = 0; k < r.J && ok; ++k) {
        ok = ok && (double)(float)r.v_gz[k] == r.v_gz[k];
        // the Stub draws velocities from the ANGLE space (roboy_robot.py:38): bound of the normalised velocity
        const double span = (double)r.v_span[k], hi = (double)r.v_hi[k], lo = (double)r.v_lo[k];
        const double n_lo = (2.0 * (double)r.a_lo[k] - hi - lo) / span, n_hi = (2.0 * (double)r.a_hi[k] - hi - lo) / span;
        ok = ok && fabs(n_lo) < 1e9 && fabs(n_hi) < 1e9 && fabs(r.v_gz[k]) < 1e9;
    }
    const double lo = r.reward_lo, hi = r.reward_hi;
    ok = ok && !(lo != lo) && !(hi != hi);
    if (ok) {
        const double band_lo = fabs(lo) <= DBL_MAX ? 1e-5 * fabs(lo) : 0.0, band_hi = fabs(hi) <= DBL_MAX ? 1e-5 * fabs(hi) : 0.0;
        pen.on = 1;
        pen.lo_c = (float)lo;
        pen.band = round_up_f32(band_lo);
        pen.hi_in = round_down_f32(hi - band_hi);
    }
    e->spec.pen = pen;
    for (int k = 0; k < r.J; ++k) e->spec.v_gz_f[k] = (float)r.v_gz[k];
}

CallCounter counter(roboy_env *e, CallCounter::Mode mode, unsigned long long t_fixed = 0) {
    CallCounter c;
    c.t_dev = e->t_dev;
    c.cta_done = e->cta_done;
    c.t_fixed = t_fixed;
    c.mode = mode;
    c.advance = 1;
    return c;
}

// The fields both step parameter blocks carry (StepParams of the tuned kernels, GStepParams of the generic ones).
template <class P>
void fill_common_step_params(roboy_env *e, P &p, const float *actions, float *obs, float *reward, uint8_t *done) {
    p.n = e->cfg.n_envs;
    p.e_begin = 0;
    p.e_end = e->cfg.n_envs;
    p.gid_base = e->cfg.env_id_base;
    p.cc = counter(e, CallCounter::kAdvance);
    p.keys = e->keys;
    p.max_len = e->cfg.max_episode_len;
    p.actions = actions;
    p.goal = e->goal;
    p.step_flags = e->step_flags;
    p.held = e->held;
    p.obs = obs ? obs : e->obs;
    p.reward = reward ? reward : e->reward;
    p.done = done ? done : e->done;
    p.terminal_obs = e->terminal_obs;
    p.done_bits = e->done_bits;
    p.stats = e->stats;
    p.err_flags = e->err_flags;
    p.first_bad = e->first_bad;
}

// The scalar constants of the tuned MSJ-shaped kernels: component 0 of the finished RobotSpec (an MSJ-shaped robot has
// the same bounds on every component), after prove_generic_fastdiv and set_penalty_f32.  Kept in the parameter block as
// scalars: the tuned step is launch-bound at small sizes, and carrying the whole RobotSpec there made it slower.
void tune_step_params(const RobotSpec &r, int div_mode, StepParams &p) {
    RobotConsts &c = p.c;
    c.a_hi = r.a_hi[0];
    c.a_lo = r.a_lo[0];
    c.a_span = r.a_span[0];
    c.v_hi = r.v_hi[0];
    c.v_lo = r.v_lo[0];
    c.v_span = r.v_span[0];
    c.thr_angle = r.thr_angle;
    c.thr_vel = r.thr_vel;
    c.penalty_boundary = r.penalty_boundary;
    c.bonus_goal = r.bonus_goal;
    c.reward_lo = r.reward_lo;
    c.reward_hi = r.reward_hi;
    FastConsts &f = p.f;
    if (div_mode == kDivChecked) {   // the reciprocals prove_generic_fastdiv checked on this device
        f.a_rc = r.a_rcp[0];
        f.v_rc = r.v_rcp[0];
    } else {                         // kDivProved: the reciprocals oracle/verify_fastdiv.c proved (unused under kDivIeee)
        f.a_rc = (float)(1.0 / (double)r.a_span[0]);
        f.v_rc = (float)(1.0 / (double)r.v_span[0]);
    }
    f.thr_angle_sq_hi = r.thr_angle_sq_hi;
    f.a_span24 = r.a_span[0] * 0x1p-24f;
    f.a_span21 = r.a_span21[0];
    f.reward_lo_f = round_up_f32(r.reward_lo);
    f.reward_hi_f = round_down_f32(r.reward_hi);
    f.v_gz = r.v_gz[0];
    f.v_gz_f = r.v_gz_f[0];
    f.pen = r.pen;
    p.hold_lo = r.hold_lo[0];
    p.hold_hi = r.hold_hi[0];
    p.hold_mag = fmaxf(fabsf(r.hold_lo[0]), fabsf(r.hold_hi[0]));
    p.hold_c = r.hold_c;
    p.hold_h = r.hold_h;
    p.act_in_hi = 1.0f;   // roboy_env.py:31
    p.act_in_lo = -1.0f;
}

void fill_step_params(roboy_env *e, StepParams &p, const float *actions, float *obs, float *reward, uint8_t *done) {
    fill_common_step_params(e, p, actions, obs, reward, done);
    tune_step_params(e->spec, e->fastdiv, p);
    p.goal1 = e->goal + e->cfg.n_envs;
    p.goal2 = e->goal + 2 * e->cfg.n_envs;
    p.obs_aligned = ((uintptr_t)p.obs & 15) == 0;
}

void fill_generic_step_params(roboy_env *e, GStepParams &p, const float *actions, float *obs, float *reward, uint8_t *done) {
    fill_common_step_params(e, p, actions, obs, reward, done);
    p.r = e->spec;
    p.penalty = e->cfg.joint_vel_penalty;
    p.bonus = e->cfg.bonus_for_goal;
    p.auto_reset = e->cfg.auto_reset;
}

// One fused step over local envs [e_begin, e_end): the tuned kernel for MSJ-shaped robots, the generic one otherwise.
// obs / reward / done: full-array base pointers (NULL = the handle's buffers).
cudaError_t launch_env_step(roboy_env *e, const float *actions, float *obs, float *reward, uint8_t *done, uint64_t e_begin,
                            uint64_t e_end, const CallCounter &cc, bool with_done_bits, cudaStream_t stream) {
    if (e->msj_shaped) {
        StepParams p;
        fill_step_params(e, p, actions, obs, reward, done);
        p.e_begin = e_begin;
        p.e_end = e_end;
        p.cc = cc;
        if (!with_done_bits) p.done_bits = nullptr;
        return launch_step(p, e->cfg.joint_vel_penalty, e->cfg.bonus_for_goal, e->cfg.auto_reset, e->fastdiv, e->sm_count, stream);
    }
    GStepParams p;
    fill_generic_step_params(e, p, actions, obs, reward, done);
    p.e_begin = e_begin;
    p.e_end = e_end;
    p.cc = cc;
    if (!with_done_bits) p.done_bits = nullptr;
    return launch_generic_step(p, e->sm_count, stream);
}

int check_env(roboy_env *e) {
    if (!e) return fail(ROBOY_E_ARG, "NULL handle");
    return ROBOY_OK;
}

}  // namespace

extern "C" {

int roboy_abi_version(void) { return ROBOY_B200_ABI_VERSION; }
const char *roboy_last_error(void) { return g_err; }

int roboy_cfg_msj(roboy_cfg *cfg) {
    if (!cfg) return fail(ROBOY_E_ARG, "NULL cfg");
    memset(cfg, 0, sizeof(*cfg));
    const double pi = 3.14159265358979323846;
    cfg->n_envs = 1;
    cfg->angle_high = (float)pi;  // msj_robot.py:9  Box(low=-np.pi, high=np.pi, dtype float32)
    cfg->angle_low = (float)(-pi);
    cfg->vel_high = (float)(pi / 6);  // msj_robot.py:10
    cfg->vel_low = (float)(-pi / 6);
    cfg->act_high = (float)0.3;  // msj_robot.py:15-16
    cfg->act_low = (float)(-0.3);
    cfg->max_episode_len = 400;      // roboy_env.py:28
    cfg->joint_vel_penalty = 0;      // roboy_env.py:13
    cfg->bonus_for_goal = 1;         // roboy_env.py:14
    cfg->auto_reset = 1;
    cfg->penalty_boundary = 1.0f;    // roboy_env.py:26
    cfg->bonus_goal = 1000.0f;       // roboy_env.py:27
    cfg->reward_lo = -INFINITY;
    cfg->reward_hi = INFINITY;
    cfg->dim_joint = ROBOY_DIM_JOINT;    // msj_robot.py:8
    cfg->dim_action = ROBOY_DIM_ACTION;  // msj_robot.py:12
    cfg->per_component_bounds = 0;
    for (int k = 0; k < ROBOY_DIM_JOINT; ++k) {
        cfg->angle_low_v[k] = cfg->angle_low; cfg->angle_high_v[k] = cfg->angle_high;
        cfg->vel_low_v[k] = cfg->vel_low; cfg->vel_high_v[k] = cfg->vel_high;
    }
    for (int k = 0; k < ROBOY_DIM_ACTION; ++k) { cfg->act_low_v[k] = cfg->act_low; cfg->act_high_v[k] = cfg->act_high; }
    return ROBOY_OK;
}

int roboy_hold_intervals(const roboy_cfg *cfg, float *lo, float *hi) {
    if (!cfg || !lo || !hi) return fail(ROBOY_E_ARG, "NULL argument");
    if (const char *why = check_robot(*cfg)) return fail(ROBOY_E_ARG, "%s", why);
    RobotSpec r;
    fill_robot_spec(*cfg, r);
    for (int k = 0; k < r.A; ++k) { lo[k] = r.hold_lo[k]; hi[k] = r.hold_hi[k]; }
    return ROBOY_OK;
}

int roboy_hold_interval(const roboy_cfg *cfg, float *lo, float *hi) {
    if (!cfg || !lo || !hi) return fail(ROBOY_E_ARG, "NULL argument");
    float l[ROBOY_MAX_ACTION], h[ROBOY_MAX_ACTION];
    const int rc = roboy_hold_intervals(cfg, l, h);
    if (rc) return rc;
    *lo = l[0];
    *hi = h[0];
    return ROBOY_OK;
}

int roboy_create(const roboy_cfg *cfg, int device, roboy_env **out) {
    if (!cfg || !out) return fail(ROBOY_E_ARG, "NULL argument");
    *out = nullptr;
    if (cfg->n_envs == 0) return fail(ROBOY_E_ARG, "n_envs must be > 0");
    if (cfg->n_envs > 0x7fffff00ull) return fail(ROBOY_E_ARG, "a shard holds fewer than 2^31 envs");
    if (const char *why = check_robot(*cfg)) return fail(ROBOY_E_ARG, "%s", why);
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(ROBOY_E_CUDA, "no CUDA device: roboy_b200 has no CPU path");
    }
    if (device < 0 || device >= n_dev) return fail(ROBOY_E_ARG, "device %d out of range (%d devices)", device, n_dev);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(ROBOY_E_CUDA, "cudaSetDevice(%d) failed", device);

    roboy_env *e = new (std::nothrow) roboy_env();
    if (!e) return fail(ROBOY_E_ALLOC, "out of host memory");
    e->cfg = *cfg;
    e->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) e->sm_count = prop.multiProcessorCount;
    e->keys = make_philox_keys(cfg->seed);
    fill_robot_spec(*cfg, e->spec);
    const RobotSpec &r = e->spec;
    e->J = r.J;
    e->A = r.A;
    e->D = 3 * r.J;
    e->msj_shaped = is_msj_shaped(*cfg, r);
    if (const char *force = getenv("ROBOY_B200_FORCE_GENERIC"))   // tests: run an MSJ-shaped robot through the generic kernels
        if (force[0] == '1') e->msj_shaped = false;
    e->fastdiv = (e->msj_shaped && spans_are_proved(r.a_lo[0], r.a_hi[0], r.v_lo[0], r.v_hi[0])) ? kDivProved : kDivIeee;
    if (e->fastdiv == kDivIeee) {
        // Any other robot: the division by its spans is checked against IEEE division on this device, over all 2^32
        // numerators (roboy_generic.cuh).  The generic step uses the per-joint reciprocals; an MSJ-shaped robot with other
        // limits runs the tuned kernels in their range-checked instantiation (kDivChecked) with the reciprocal of joint 0.
        const char *off = getenv("ROBOY_B200_GENERIC_FASTDIV");
        if (!(off && off[0] == '0')) {
            const cudaError_t perr = prove_generic_fastdiv(e->spec, e->sm_count, nullptr);
            if (perr != cudaSuccess) {
                free_env(e);
                return fail(ROBOY_E_CUDA, "fast-division proof: %s", cudaGetErrorString(perr));
            }
            if (e->msj_shaped && e->spec.fastdiv) e->fastdiv = kDivChecked;
        }
    }

    set_penalty_f32(e);

    const uint64_t n = cfg->n_envs;
    cudaError_t err = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) {
        if (err == cudaSuccess) err = cudaMalloc(p, bytes);
    };
    alloc((void **)&e->goal, sizeof(float) * e->J * n);
    alloc((void **)&e->step_flags, sizeof(uint32_t) * n);
    alloc((void **)&e->held, sizeof(float) * 2 * e->J * n);
    alloc((void **)&e->obs, sizeof(float) * e->D * n);
    alloc((void **)&e->reward, sizeof(float) * n);
    alloc((void **)&e->done, n);
    alloc((void **)&e->stats, sizeof(double) * ROBOY_STAT_COUNT);
    alloc((void **)&e->err_flags, sizeof(uint32_t));
    alloc((void **)&e->first_bad, sizeof(unsigned long long));
    alloc((void **)&e->t_dev, sizeof(unsigned long long));
    alloc((void **)&e->cta_done, sizeof(unsigned int));
    if (err == cudaSuccess) err = cudaMemset(e->t_dev, 0, sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMemset(e->cta_done, 0, sizeof(unsigned int));
    if (err == cudaSuccess) err = cudaMemset(e->stats, 0, sizeof(double) * ROBOY_STAT_COUNT);
    if (err == cudaSuccess) err = cudaMemset(e->err_flags, 0, sizeof(uint32_t));
    if (err == cudaSuccess) err = cudaMemset(e->first_bad, 0xff, sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMemset(e->done, 0, n);
    if (err == cudaSuccess) {
        GInitParams ip{};
        ip.n = n;
        ip.gid_base = cfg->env_id_base;
        ip.cc = counter(e, CallCounter::kFixed, 0);
        ip.keys = e->keys;
        ip.r = e->spec;
        ip.goal = e->goal;
        ip.step_flags = e->step_flags;
        ip.held = e->held;
        ip.mask = nullptr;
        ip.obs = nullptr;
        err = launch_generic_init_or_reset(ip, e->sm_count, 0);
        e->launches++;
        // Goal draw 0 of counter 0 is the goal the env starts with.  The first get_new_goal_joint_angles() after
        // construction hands out that same draw, so the reference's RoboyEnv.__init__ (roboy_env.py:37), which asks the
        // client for its first goal, starts from the goal the fused env starts from.
        e->goal_sub = 0;
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(0);
    if (err != cudaSuccess) {
        cudaGetLastError();
        int code = err == cudaErrorMemoryAllocation ? ROBOY_E_ALLOC : ROBOY_E_CUDA;
        fail(code, "roboy_create(n_envs=%llu): %s", (unsigned long long)n, cudaGetErrorString(err));
        free_env(e);
        return code;
    }
    *out = e;
    return ROBOY_OK;
}

int roboy_destroy(roboy_env *env) {
    if (check_env(env)) return ROBOY_E_ARG;
    {
        DeviceGuard g(env->device);
        cudaDeviceSynchronize();
    }
    unref(env);
    return ROBOY_OK;
}

int roboy_set_reward_range(roboy_env *env, double lo, double hi) {
    if (check_env(env)) return ROBOY_E_ARG;
    env->cfg.reward_lo = env->spec.reward_lo = lo;
    env->cfg.reward_hi = env->spec.reward_hi = hi;
    set_penalty_f32(env);
    return ROBOY_OK;
}

int roboy_reset(roboy_env *env, const uint8_t *mask_dev, float *obs_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    env->goal_sub = 1;  // the reset itself consumes goal draw 0 of the new counter value
    GInitParams ip{};
    ip.n = env->cfg.n_envs;
    ip.gid_base = env->cfg.env_id_base;
    ip.cc = counter(env, CallCounter::kAdvance);
    ip.keys = env->keys;
    ip.r = env->spec;
    ip.goal = env->goal;
    ip.step_flags = env->step_flags;
    ip.held = nullptr;
    ip.mask = mask_dev;
    ip.obs = obs_dev ? obs_dev : env->obs;
    CUDA_TRY(launch_generic_init_or_reset(ip, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_step(roboy_env *env, const float *actions_dev, float *obs_dev, float *reward_dev, uint8_t *done_dev,
               void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!actions_dev) return fail(ROBOY_E_ARG, "actions_dev is NULL");
    if ((uintptr_t)actions_dev & 15) return fail(ROBOY_E_ARG, "actions must be 16-byte aligned");
    if (obs_dev && ((uintptr_t)obs_dev & 3)) return fail(ROBOY_E_ARG, "obs must be 4-byte aligned");
    DeviceGuard g(env->device);
    env->goal_sub = 1;  // done envs consume goal draw 0 of the new counter value
    CUDA_TRY(launch_env_step(env, actions_dev, obs_dev, reward_dev, done_dev, 0, env->cfg.n_envs,
                             counter(env, CallCounter::kAdvance), true, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_step_many(roboy_env *env, uint32_t T, const float *actions_dev, float *obs_dev, float *reward_dev,
                    uint8_t *done_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!actions_dev || !obs_dev || !reward_dev || !done_dev) return fail(ROBOY_E_ARG, "NULL device pointer");
    if (T == 0) return ROBOY_OK;
    if ((uintptr_t)actions_dev & 15) return fail(ROBOY_E_ARG, "actions must be 16-byte aligned");
    if ((uintptr_t)obs_dev & 3) return fail(ROBOY_E_ARG, "obs must be 4-byte aligned");
    DeviceGuard g(env->device);
    env->goal_sub = 1;
    if (!env->msj_shaped) {
        // other robots: T launches of the generic step kernel over the [t] slices (same results, state through HBM)
        const uint64_t n = env->cfg.n_envs;
        for (uint32_t t = 0; t < T; ++t) {
            CUDA_TRY(launch_env_step(env, actions_dev + (size_t)t * n * env->A, obs_dev + (size_t)t * n * env->D,
                                     reward_dev + (size_t)t * n, done_dev + (size_t)t * n, 0, n,
                                     counter(env, CallCounter::kAdvance), false, (cudaStream_t)stream));
            env->launches++;
        }
        return ROBOY_OK;
    }
    StepParams p;
    fill_step_params(env, p, actions_dev, obs_dev, reward_dev, done_dev);
    p.cc.advance = T;
    p.done_bits = nullptr;  // the done-index list belongs to single steps
    // every [t] slice of obs must be 16-byte aligned for the vector / bulk stores
    p.obs_aligned = (((uintptr_t)obs_dev & 15) == 0) && (T == 1 || (env->cfg.n_envs * ROBOY_DIM_OBS * sizeof(float)) % 16 == 0);
    CUDA_TRY(launch_step_many(p, T, env->cfg.joint_vel_penalty, env->cfg.bonus_for_goal, env->cfg.auto_reset,
                              env->fastdiv, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

// ---- the host-buffer path: H2D(actions) -> step kernel -> D2H(obs, reward, done), pipelined in stages ----
enum { kHostH2D = 1, kHostKernel = 2, kHostD2H = 4, kHostSplitDirections = 8 };

static int host_pipeline(roboy_env *env, const float *actions_host, float *obs_host, float *reward_host,
                         uint8_t *done_host, int what) {
    const uint64_t n = env->cfg.n_envs;
    // The stages run on internal non-blocking streams.  Order them after everything queued on this device before the
    // call (roboy_reset / roboy_set_* / roboy_step on ANY stream, blocking or not): the call is device-synchronous.
    CUDA_TRY(cudaDeviceSynchronize());
    if (!env->host_ready) {
        CUDA_TRY(cudaMalloc((void **)&env->actions_stage, sizeof(float) * env->A * n));
        for (int i = 0; i < kHostStreamsMax; ++i) {
            CUDA_TRY(cudaStreamCreateWithFlags(&env->hs[i], cudaStreamNonBlocking));
            CUDA_TRY(cudaEventCreateWithFlags(&env->hev[i], cudaEventDisableTiming));
        }
        env->host_ready = true;
    }
    const bool run_kernel = (what & kHostKernel) != 0;
    if (run_kernel) env->goal_sub = 1;
    const size_t A = (size_t)env->A, D = (size_t)env->D;
    // All stages of one call use the same counter value *t_dev + 1 (they run concurrently on several streams, so none of
    // them may store it back); a one-thread kernel advances the device counter once they have all finished.
    const CallCounter cc = counter(env, CallCounter::kPeekNext);
    const float *k_actions = env->actions_stage;   // what the stage kernels read and write (full-array base pointers)
    float *k_obs = nullptr, *k_reward = nullptr;
    uint8_t *k_done = nullptr;
    const int mode = run_kernel ? env->host_mode : ROBOY_HOST_STAGED;
    if (mode != ROBOY_HOST_STAGED) {
        // zero-copy: the kernel addresses the caller's page-locked buffers directly over PCIe
        void *o = nullptr, *r = nullptr, *d = nullptr, *a = nullptr;
        if (cudaHostGetDevicePointer(&o, obs_host, 0) != cudaSuccess || cudaHostGetDevicePointer(&r, reward_host, 0) != cudaSuccess ||
            cudaHostGetDevicePointer(&d, done_host, 0) != cudaSuccess ||
            (mode == ROBOY_HOST_MAPPED_ALL && cudaHostGetDevicePointer(&a, (void *)actions_host, 0) != cudaSuccess)) {
            cudaGetLastError();
            return fail(ROBOY_E_ARG, "host mode %d needs page-locked host buffers (cudaHostAlloc / cudaHostRegister / roboy_host_alloc)", mode);
        }
        k_obs = (float *)o;
        k_reward = (float *)r;
        k_done = (uint8_t *)d;
        if (mode == ROBOY_HOST_MAPPED_ALL) {
            if ((uintptr_t)a & 15) return fail(ROBOY_E_ARG, "actions must be 16-byte aligned");
            k_actions = (const float *)a;
        }
    }
    cudaError_t err = cudaSuccess;
#define HOST_TRY(expr) do { if (err == cudaSuccess) err = (expr); } while (0)
    int used = 0;
    if (mode == ROBOY_HOST_MAPPED_ALL) {
        // one launch over the whole shard: PCIe reads and posted writes overlap inside the kernel, no staging at all
        HOST_TRY(launch_env_step(env, k_actions, k_obs, k_reward, k_done, 0, n, cc, true, env->hs[0]));
        env->launches++;
        used = 1;
    } else if (what & kHostSplitDirections) {
        // copy-ceiling probe only: both directions as one monolithic copy each, on two independent streams
        if (what & kHostH2D)
            HOST_TRY(cudaMemcpyAsync(env->actions_stage, actions_host, sizeof(float) * A * n, cudaMemcpyHostToDevice, env->hs[0]));
        if (what & kHostD2H) {
            HOST_TRY(cudaMemcpyAsync(obs_host, env->obs, sizeof(float) * D * n, cudaMemcpyDeviceToHost, env->hs[1]));
            HOST_TRY(cudaMemcpyAsync(reward_host, env->reward, sizeof(float) * n, cudaMemcpyDeviceToHost, env->hs[1]));
            HOST_TRY(cudaMemcpyAsync(done_host, env->done, n, cudaMemcpyDeviceToHost, env->hs[1]));
        }
        used = 2;
    } else {
        // Pipeline over stages of the env range.  ROBOY_HOST_PATTERN_RING (default): stage i runs H2D(actions_i) -> step
        // kernel_i -> D2H(obs_i, reward_i, done_i) on stream i % n_streams, so the copy engines of both directions and the
        // SMs overlap across stages.  ROBOY_HOST_PATTERN_SPLIT: one "up" stream carries every H2D and kernel, a ring of
        // "down" streams the D2H copies behind per-stage events.  Measured on PCIe Gen5 x16 (16,777,216 envs, 1.22 GB per
        // pass; the two directions as one monolithic copy each take 13.4-13.9 ms): ring of 2 streams 14.0-14.2 ms, split
        // with 1 / 2 / 3 down streams 15.9 / 15.3 / 15.4 ms -- an H2D engine that never waits takes link bandwidth from
        // the D2H leg, which is the longer one (41 of the 73 bytes).  The first stages are shorter: the D2H engine idles
        // until the first kernel has run.
        int stage = 0;
        const uint64_t stage_envs = env->host_stage_envs;
        cudaStream_t up = env->hs[0];
        const int n_down = env->host_streams > 1 ? env->host_streams - 1 : 0;   // 0: D2H on the up stream too
        const bool ring = env->host_pattern == ROBOY_HOST_PATTERN_RING && env->host_streams > 1;
        uint64_t b = 0;
        while (b < n && err == cudaSuccess) {
            uint64_t len = stage_envs;
            if (env->host_ramp && stage < 3 && n > 4 * stage_envs) len = (stage_envs >> (3 - stage)) & ~31ull;  // 1/8, 1/4, 1/2
            if (len == 0) len = stage_envs;
            const uint64_t eend = b + len < n ? b + len : n;
            const uint64_t cnt = eend - b;
            if (ring) up = env->hs[stage % env->host_streams];   // ROBOY_HOST_PATTERN_RING: stage i entirely on stream i % n
            if (what & kHostH2D)
                HOST_TRY(cudaMemcpyAsync(env->actions_stage + b * A, actions_host + b * A, sizeof(float) * A * cnt,
                                         cudaMemcpyHostToDevice, up));
            if (run_kernel) {
                HOST_TRY(launch_env_step(env, k_actions, k_obs, k_reward, k_done, b, eend, cc, true, up));
                env->launches++;
            }
            if ((what & kHostD2H) && mode == ROBOY_HOST_STAGED) {
                cudaStream_t down = n_down ? env->hs[1 + stage % n_down] : up;
                if (ring) down = up;
                if (down != up && ((what & kHostH2D) || run_kernel)) {
                    cudaEvent_t ev = env->hev[stage % kHostStreamsMax];   // re-recording an event is fine: waits already
                    HOST_TRY(cudaEventRecord(ev, up));                    // queued keep the record they saw
                    HOST_TRY(cudaStreamWaitEvent(down, ev, 0));
                }
                HOST_TRY(cudaMemcpyAsync(obs_host + b * D, env->obs + b * D, sizeof(float) * D * cnt, cudaMemcpyDeviceToHost, down));
                HOST_TRY(cudaMemcpyAsync(reward_host + b, env->reward + b, sizeof(float) * cnt, cudaMemcpyDeviceToHost, down));
                HOST_TRY(cudaMemcpyAsync(done_host + b, env->done + b, cnt, cudaMemcpyDeviceToHost, down));
            }
            b = eend;
            ++stage;
        }
        used = ring ? env->host_streams : 1 + n_down;
    }
    if (err == cudaSuccess && run_kernel) {
        // all kernels of this call are on stream 0 (mapped modes: one stream per stage ring is not needed either), so the
        // device counter is advanced there, in stream order, without a join
        if (env->host_pattern == ROBOY_HOST_PATTERN_RING && mode != ROBOY_HOST_MAPPED_ALL)
            for (int i = 1; i < used; ++i) {
                HOST_TRY(cudaEventRecord(env->hev[i], env->hs[i]));
                HOST_TRY(cudaStreamWaitEvent(env->hs[0], env->hev[i], 0));
            }
        HOST_TRY(launch_counter_bump(env->t_dev, 1, env->hs[0]));
    }
    // Whatever happened, nothing may still be copying into the caller's buffers when this returns.
    for (int i = 0; i < used; ++i) {
        const cudaError_t e2 = cudaStreamSynchronize(env->hs[i]);
        if (err == cudaSuccess) err = e2;
    }
#undef HOST_TRY
    if (err != cudaSuccess) {
        cudaGetLastError();
        return fail(ROBOY_E_CUDA, "roboy_step_host: %s", cudaGetErrorString(err));
    }
    return ROBOY_OK;
}

int roboy_step_host(roboy_env *env, const float *actions_host, float *obs_host, float *reward_host,
                    uint8_t *done_host) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!actions_host || !obs_host || !reward_host || !done_host) return fail(ROBOY_E_ARG, "NULL host buffer");
    DeviceGuard g(env->device);
    const int what = kHostH2D | kHostKernel | kHostD2H;
    const bool tuning = env->host_autotune && env->host_mode == ROBOY_HOST_STAGED && env->host_calls < 3 &&
                        env->cfg.n_envs > 2 * env->host_stage_envs;   // (a single-stage call has nothing to tune)
    if (!tuning) return host_pipeline(env, actions_host, obs_host, reward_host, done_host, what);
    // call 0: warm-up (stream creation, first touch), ring of 2; call 1: ring of 2, timed; call 2: one stream, timed
    const int call = env->host_calls++;
    env->host_streams = call == 2 ? 1 : 2;
    timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    const int rc = host_pipeline(env, actions_host, obs_host, reward_host, done_host, what);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (call >= 1) env->host_ms[call - 1] = (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6;
    if (call == 2) env->host_streams = env->host_ms[1] < 0.97 * env->host_ms[0] ? 1 : 2;
    return rc;
}

int roboy_host_copy_probe(roboy_env *env, const float *actions_host, float *obs_host, float *reward_host,
                          uint8_t *done_host, int directions, int monolithic, int iters, double *ms_per_pass) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!actions_host || !obs_host || !reward_host || !done_host || !ms_per_pass) return fail(ROBOY_E_ARG, "NULL argument");
    if (!(directions & 3) || iters < 1) return fail(ROBOY_E_ARG, "directions: 1 = H2D, 2 = D2H, 3 = both; iters >= 1");
    DeviceGuard g(env->device);
    const int what = ((directions & 1) ? kHostH2D : 0) | ((directions & 2) ? kHostD2H : 0) | (monolithic ? kHostSplitDirections : 0);
    int rc = host_pipeline(env, actions_host, obs_host, reward_host, done_host, what);  // warm-up (stream creation, page touch)
    if (rc) return rc;
    timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int i = 0; i < iters; ++i) {
        rc = host_pipeline(env, actions_host, obs_host, reward_host, done_host, what);
        if (rc) return rc;
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    *ms_per_pass = ((t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6) / iters;
    return ROBOY_OK;
}

int roboy_set_host_mode(roboy_env *env, int mode) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (mode < ROBOY_HOST_STAGED || mode > ROBOY_HOST_MAPPED_ALL) return fail(ROBOY_E_ARG, "unknown host mode %d", mode);
    env->host_mode = mode;
    return ROBOY_OK;
}

int roboy_host_alloc(uint64_t bytes, int write_combined, void **out_host) {
    if (!out_host || bytes == 0) return fail(ROBOY_E_ARG, "NULL argument / zero size");
    *out_host = nullptr;
    const unsigned flags = cudaHostAllocPortable | cudaHostAllocMapped | (write_combined ? cudaHostAllocWriteCombined : 0u);
    const cudaError_t e = cudaHostAlloc(out_host, bytes, flags);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? ROBOY_E_ALLOC : ROBOY_E_CUDA, "cudaHostAlloc(%llu): %s",
                    (unsigned long long)bytes, cudaGetErrorString(e));
    }
    return ROBOY_OK;
}

int roboy_host_free(void *host) {
    if (!host) return ROBOY_OK;
    CUDA_TRY(cudaFreeHost(host));
    return ROBOY_OK;
}

int roboy_set_host_pipeline(roboy_env *env, uint64_t stage_envs, int n_streams) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (stage_envs == 0 || (stage_envs & 31) || n_streams < 1 || n_streams > kHostStreamsMax)
        return fail(ROBOY_E_ARG, "stage_envs must be a positive multiple of 32 and 1 <= n_streams <= %d", kHostStreamsMax);
    env->host_stage_envs = stage_envs;
    env->host_streams = n_streams;
    env->host_autotune = false;   // the caller fixed the pipeline
    return ROBOY_OK;
}

int roboy_set_host_autotune(roboy_env *env, int enable) {
    if (check_env(env)) return ROBOY_E_ARG;
    env->host_autotune = enable != 0;
    env->host_calls = 0;
    if (enable) {
        env->host_streams = kHostStreamsDefault;
        env->host_stage_envs = kHostStageEnvsDefault;
        env->host_pattern = ROBOY_HOST_PATTERN_RING;
        env->host_ramp = true;
    }
    return ROBOY_OK;
}

int roboy_get_host_pipeline(roboy_env *env, uint64_t *stage_envs, int *n_streams, int *pattern) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (stage_envs) *stage_envs = env->host_stage_envs;
    if (n_streams) *n_streams = env->host_streams;
    if (pattern) *pattern = env->host_pattern;
    return ROBOY_OK;
}

int roboy_set_host_pattern(roboy_env *env, int pattern) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (pattern != ROBOY_HOST_PATTERN_SPLIT && pattern != ROBOY_HOST_PATTERN_RING) return fail(ROBOY_E_ARG, "unknown pattern %d", pattern);
    env->host_pattern = pattern;
    return ROBOY_OK;
}

int roboy_set_host_ramp(roboy_env *env, int enable) {
    if (check_env(env)) return ROBOY_E_ARG;
    env->host_ramp = enable != 0;
    return ROBOY_OK;
}

int roboy_set_terminal_obs(roboy_env *env, float *terminal_obs_dev) {
    if (check_env(env)) return ROBOY_E_ARG;
    env->terminal_obs = terminal_obs_dev;
    return ROBOY_OK;
}

int roboy_compute_reward(roboy_env *env, uint64_t k, const float *q_dev, const float *qd_dev,
                         const uint8_t *feasible_dev, const float *goal_q_dev, const float *goal_qd_dev,
                         double *reward_dev, uint8_t *reached_dev, int check_range, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!q_dev || !qd_dev || !goal_q_dev || !reward_dev) return fail(ROBOY_E_ARG, "NULL device pointer");
    DeviceGuard g(env->device);
    GRewardParams p{};
    p.k = k;
    p.r = env->spec;
    p.penalty = env->cfg.joint_vel_penalty != 0;
    p.bonus = env->cfg.bonus_for_goal != 0;
    p.check_range = check_range;   // 0 no check, 1 check, 2 reward-range probe (no check, correctly rounded float32 exp)
    p.gid_base = env->cfg.env_id_base;
    p.q = q_dev;
    p.qd = qd_dev;
    p.goal_q = goal_q_dev;
    p.goal_qd = goal_qd_dev;
    p.feasible = feasible_dev;
    p.reward = reward_dev;
    p.reached = reached_dev;
    p.stats = env->stats;
    p.err_flags = env->err_flags;
    p.first_bad = env->first_bad;
    CUDA_TRY(launch_generic_compute_reward(p, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

static int scatter_common(roboy_env *env, GScatterParams &p, uint64_t k, const int64_t *idx, void *stream) {
    DeviceGuard g(env->device);
    p.k = k;
    p.n = env->cfg.n_envs;
    p.idx = idx;
    p.r = env->spec;
    p.gid_base = env->cfg.env_id_base;
    p.goal = env->goal;
    p.held = env->held;
    p.step_flags = env->step_flags;
    p.err_flags = env->err_flags;
    p.first_bad = env->first_bad;
    CUDA_TRY(launch_generic_scatter(p, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_set_goal(roboy_env *env, uint64_t k, const int64_t *idx_dev, const float *goal_q_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!goal_q_dev) return fail(ROBOY_E_ARG, "goal_q_dev is NULL");
    GScatterParams p{};
    p.goal_q = goal_q_dev;
    return scatter_common(env, p, k, idx_dev, stream);
}

int roboy_set_state(roboy_env *env, uint64_t k, const int64_t *idx_dev, const float *q_dev, const float *qd_dev,
                    const uint8_t *feasible_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!q_dev || !qd_dev) return fail(ROBOY_E_ARG, "q_dev/qd_dev is NULL");
    GScatterParams p{};
    p.q = q_dev;
    p.qd = qd_dev;
    p.feasible = feasible_dev;
    return scatter_common(env, p, k, idx_dev, stream);
}

int roboy_set_step_num(roboy_env *env, uint64_t k, const int64_t *idx_dev, const int32_t *step_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!step_dev) return fail(ROBOY_E_ARG, "step_dev is NULL");
    GScatterParams p{};
    p.step = step_dev;
    return scatter_common(env, p, k, idx_dev, stream);
}

int roboy_read_state(roboy_env *env, uint64_t k, const int64_t *idx_dev, float *q_dev, float *qd_dev,
                     uint8_t *feasible_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!q_dev || !qd_dev) return fail(ROBOY_E_ARG, "q_dev/qd_dev is NULL");
    GScatterParams p{};
    p.out_q = q_dev;
    p.out_qd = qd_dev;
    p.out_feasible = feasible_dev;
    return scatter_common(env, p, k, idx_dev, stream);
}

static void fill_sim_params(roboy_env *env, GSimParams &p, int mode) {
    p.mode = mode;
    p.n = env->cfg.n_envs;
    p.gid_base = env->cfg.env_id_base;
    p.cc = counter(env, mode == 2 ? CallCounter::kPeek : CallCounter::kAdvance);
    p.sub = env->goal_sub;
    p.keys = env->keys;
    p.r = env->spec;
    p.step_flags = env->step_flags;
    p.held = env->held;
    p.stats = env->stats;
}

int roboy_sim_step(roboy_env *env, const float *actions_dev, float *q_dev, float *qd_dev, uint8_t *feasible_dev,
                   void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!actions_dev || !q_dev || !qd_dev) return fail(ROBOY_E_ARG, "NULL device pointer");
    if ((uintptr_t)actions_dev & 15) return fail(ROBOY_E_ARG, "actions must be 16-byte aligned");
    DeviceGuard g(env->device);
    env->goal_sub = 0;
    GSimParams p{};
    fill_sim_params(env, p, 0);
    p.actions = actions_dev;
    p.out_q = q_dev;
    p.out_qd = qd_dev;
    p.out_feasible = feasible_dev;
    CUDA_TRY(launch_generic_sim(p, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_sim_reset(roboy_env *env, const uint8_t *mask_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    env->goal_sub = 0;
    GSimParams p{};
    fill_sim_params(env, p, 1);
    p.mask = mask_dev;
    CUDA_TRY(launch_generic_sim(p, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_new_goal(roboy_env *env, float *goal_q_dev, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!goal_q_dev) return fail(ROBOY_E_ARG, "goal_q_dev is NULL");
    DeviceGuard g(env->device);
    if (env->goal_sub >= 255) return fail(ROBOY_E_ARG, "more than 255 goal draws without a step or reset in between");
    GSimParams p{};
    fill_sim_params(env, p, 2);
    p.out_q = goal_q_dev;
    CUDA_TRY(launch_generic_sim(p, env->sm_count, (cudaStream_t)stream));
    env->goal_sub += 1;
    env->launches++;
    return ROBOY_OK;
}

int roboy_set_flags(roboy_env *env, int joint_vel_penalty, int bonus_for_goal, int auto_reset) {
    if (check_env(env)) return ROBOY_E_ARG;
    env->cfg.joint_vel_penalty = joint_vel_penalty != 0;
    env->cfg.bonus_for_goal = bonus_for_goal != 0;
    env->cfg.auto_reset = auto_reset != 0;
    return ROBOY_OK;
}

int roboy_set_seed(roboy_env *env, uint64_t seed) {
    if (check_env(env)) return ROBOY_E_ARG;
    env->cfg.seed = seed;
    env->keys = make_philox_keys(seed);
    return ROBOY_OK;
}

int roboy_reseed(roboy_env *env, uint64_t seed) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    env->cfg.seed = seed;
    env->keys = make_philox_keys(seed);
    CUDA_TRY(cudaDeviceSynchronize());
    const unsigned long long zero = 0;
    CUDA_TRY(cudaMemcpy(env->t_dev, &zero, sizeof(zero), cudaMemcpyHostToDevice));
    GInitParams ip{};
    ip.n = env->cfg.n_envs;
    ip.gid_base = env->cfg.env_id_base;
    ip.cc = counter(env, CallCounter::kFixed, 0);
    ip.keys = env->keys;
    ip.r = env->spec;
    ip.goal = env->goal;
    ip.step_flags = env->step_flags;
    ip.held = env->held;
    CUDA_TRY(launch_generic_init_or_reset(ip, env->sm_count, 0));
    env->launches++;
    env->goal_sub = 0;
    CUDA_TRY(cudaStreamSynchronize(0));
    return ROBOY_OK;
}

int roboy_buffer(roboy_env *env, int which, void **dev_ptr, uint64_t *nbytes) {
    if (check_env(env)) return ROBOY_E_ARG;
    const uint64_t n = env->cfg.n_envs;
    void *p = nullptr;
    uint64_t b = 0;
    switch (which) {
        case ROBOY_BUF_GOAL: p = env->goal; b = 4ull * env->J * n; break;
        case ROBOY_BUF_STEP_FLAGS: p = env->step_flags; b = 4 * n; break;
        case ROBOY_BUF_HELD: p = env->held; b = 8ull * env->J * n; break;
        case ROBOY_BUF_OBS: p = env->obs; b = 4ull * env->D * n; break;
        case ROBOY_BUF_REWARD: p = env->reward; b = 4 * n; break;
        case ROBOY_BUF_DONE: p = env->done; b = n; break;
        case ROBOY_BUF_STATS: p = env->stats; b = 8 * ROBOY_STAT_COUNT; break;
        case ROBOY_BUF_TERMINAL_OBS: p = env->terminal_obs; b = env->terminal_obs ? 4ull * env->D * n : 0; break;
        case ROBOY_BUF_DONE_BITS: p = env->done_bits; b = env->done_bits ? 4 * ((n + 31) / 32) : 0; break;
        default: return fail(ROBOY_E_ARG, "unknown buffer id %d", which);
    }
    if (dev_ptr) *dev_ptr = p;
    if (nbytes) *nbytes = b;
    return ROBOY_OK;
}

struct DlCtx {
    roboy_env *env;
    int64_t shape[2];
};

static void dl_deleter(DLManagedTensor *self) {
    DlCtx *ctx = (DlCtx *)self->manager_ctx;
    unref(ctx->env);
    delete ctx;
    delete self;
}

void *roboy_export_dlpack(roboy_env *env, int which) {
    if (check_env(env)) return nullptr;
    const int64_t n = (int64_t)env->cfg.n_envs;
    DLManagedTensor *m = new (std::nothrow) DLManagedTensor();
    DlCtx *ctx = new (std::nothrow) DlCtx();
    if (!m || !ctx) {
        delete m;
        delete ctx;
        fail(ROBOY_E_ALLOC, "out of host memory");
        return nullptr;
    }
    DLTensor &t = m->dl_tensor;
    t.device.device_type = kDLCUDA;
    t.device.device_id = env->device;
    t.strides = nullptr;
    t.byte_offset = 0;
    t.shape = ctx->shape;
    t.dtype.lanes = 1;
    t.dtype.code = kDLFloat;
    t.dtype.bits = 32;
    t.ndim = 2;
    switch (which) {
        case ROBOY_BUF_GOAL: t.data = env->goal; ctx->shape[0] = env->J; ctx->shape[1] = n; break;
        case ROBOY_BUF_HELD: t.data = env->held; ctx->shape[0] = 2 * env->J; ctx->shape[1] = n; break;
        case ROBOY_BUF_OBS: t.data = env->obs; ctx->shape[0] = n; ctx->shape[1] = env->D; break;
        case ROBOY_BUF_REWARD: t.data = env->reward; t.ndim = 1; ctx->shape[0] = n; break;
        case ROBOY_BUF_STEP_FLAGS:
            t.data = env->step_flags; t.ndim = 1; ctx->shape[0] = n;
            t.dtype.code = kDLInt;  // torch has no uint32 arithmetic; the top bits used stay below 2^31
            break;
        case ROBOY_BUF_DONE:
            t.data = env->done; t.ndim = 1; ctx->shape[0] = n;
            t.dtype.code = kDLUInt; t.dtype.bits = 8;
            break;
        case ROBOY_BUF_STATS:
            t.data = env->stats; t.ndim = 1; ctx->shape[0] = ROBOY_STAT_COUNT;
            t.dtype.bits = 64;
            break;
        case ROBOY_BUF_DONE_BITS:
            if (!env->done_bits) {
                delete m;
                delete ctx;
                fail(ROBOY_E_ARG, "the done index is not enabled");
                return nullptr;
            }
            t.data = env->done_bits; t.ndim = 1; ctx->shape[0] = (n + 31) / 32;
            t.dtype.code = kDLInt;
            break;
        default:
            delete m;
            delete ctx;
            fail(ROBOY_E_ARG, "buffer %d cannot be exported", which);
            return nullptr;
    }
    env->refs.fetch_add(1);
    ctx->env = env;
    m->manager_ctx = ctx;
    m->deleter = dl_deleter;
    return m;
}

int roboy_get_counter(roboy_env *env, uint64_t *t) {
    if (check_env(env) || !t) return fail(ROBOY_E_ARG, "NULL argument");
    DeviceGuard g(env->device);
    unsigned long long v = 0;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(&v, env->t_dev, sizeof(v), cudaMemcpyDeviceToHost));
    *t = v;
    return ROBOY_OK;
}

int roboy_set_counter(roboy_env *env, uint64_t t) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    const unsigned long long v = t;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(env->t_dev, &v, sizeof(v), cudaMemcpyHostToDevice));
    env->goal_sub = 1;
    return ROBOY_OK;
}

int roboy_stats(roboy_env *env, double out_host[ROBOY_STAT_COUNT], void *stream) {
    if (check_env(env) || !out_host) return fail(ROBOY_E_ARG, "NULL argument");
    DeviceGuard g(env->device);
    CUDA_TRY(cudaMemcpyAsync(out_host, env->stats, sizeof(double) * ROBOY_STAT_COUNT, cudaMemcpyDeviceToHost,
                             (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return ROBOY_OK;
}

int roboy_clear_stats(roboy_env *env, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    CUDA_TRY(cudaMemsetAsync(env->stats, 0, sizeof(double) * ROBOY_STAT_COUNT, (cudaStream_t)stream));
    CUDA_TRY(cudaMemsetAsync(env->err_flags, 0, sizeof(uint32_t), (cudaStream_t)stream));
    CUDA_TRY(cudaMemsetAsync(env->first_bad, 0xff, sizeof(unsigned long long), (cudaStream_t)stream));
    return ROBOY_OK;
}

int roboy_clear_errors(roboy_env *env, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    CUDA_TRY(cudaMemsetAsync(env->err_flags, 0, sizeof(uint32_t), (cudaStream_t)stream));
    CUDA_TRY(cudaMemsetAsync(env->first_bad, 0xff, sizeof(unsigned long long), (cudaStream_t)stream));
    return ROBOY_OK;
}

int roboy_errors(roboy_env *env, uint32_t *err_flags, uint64_t *first_bad_env, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    uint32_t f = 0;
    unsigned long long b = 0;
    CUDA_TRY(cudaMemcpyAsync(&f, env->err_flags, sizeof(f), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaMemcpyAsync(&b, env->first_bad, sizeof(b), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    if (err_flags) *err_flags = f;
    if (first_bad_env) *first_bad_env = (uint64_t)b;
    return ROBOY_OK;
}

static int external_common(roboy_env *env, int reset, const uint8_t *mask, const float *q, const float *qd,
                           const uint8_t *feasible, float *obs, float *reward, uint8_t *done, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!q || !qd) return fail(ROBOY_E_ARG, "q_dev/qd_dev is NULL");
    DeviceGuard g(env->device);
    env->goal_sub = 1;
    GExternalParams p{};
    p.reset = reset;
    p.n = env->cfg.n_envs;
    p.gid_base = env->cfg.env_id_base;
    p.cc = counter(env, CallCounter::kAdvance);
    p.keys = env->keys;
    p.r = env->spec;
    p.penalty = env->cfg.joint_vel_penalty != 0;
    p.bonus = env->cfg.bonus_for_goal != 0;
    p.max_len = env->cfg.max_episode_len;
    p.q = q;
    p.qd = qd;
    p.feasible = feasible;
    p.mask = mask;
    p.goal = env->goal;
    p.step_flags = env->step_flags;
    p.obs = obs ? obs : env->obs;
    p.reward = reward ? reward : env->reward;
    p.done = done ? done : env->done;
    p.stats = env->stats;
    p.err_flags = env->err_flags;
    p.first_bad = env->first_bad;
    CUDA_TRY(launch_generic_external(p, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_step_external(roboy_env *env, const float *q_dev, const float *qd_dev, const uint8_t *feasible_dev,
                        float *obs_dev, float *reward_dev, uint8_t *done_dev, void *stream) {
    return external_common(env, 0, nullptr, q_dev, qd_dev, feasible_dev, obs_dev, reward_dev, done_dev, stream);
}

int roboy_reset_external(roboy_env *env, const uint8_t *mask_dev, const float *q_dev, const float *qd_dev,
                         float *obs_dev, void *stream) {
    return external_common(env, 1, mask_dev, q_dev, qd_dev, nullptr, obs_dev, nullptr, nullptr, stream);
}

int roboy_gae(uint64_t T, uint64_t n, const float *reward_dev, const float *value_dev, const uint8_t *done_dev,
              const float *last_value_dev, float gamma, float lam, float *adv_dev, float *ret_dev, void *stream) {
    if (!reward_dev || !value_dev || !done_dev || !last_value_dev || !adv_dev || !ret_dev)
        return fail(ROBOY_E_ARG, "NULL device pointer");
    GaeParams p{};
    p.T = T;
    p.n = n;
    p.reward = reward_dev;
    p.value = value_dev;
    p.done = done_dev;
    p.last_value = last_value_dev;
    p.gamma = gamma;
    p.lam = lam;
    p.adv = adv_dev;
    p.ret = ret_dev;
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CUDA_TRY(launch_gae(p, sms, (cudaStream_t)stream));
    return ROBOY_OK;
}

// The env-step block and the image offsets of a T-step fused generic policy launch (the rollout's and the evaluator's)
static int fill_generic_policy_launch(roboy_env *env, uint32_t T, float *reward_dev, uint8_t *done_dev, GStepParams &p,
                                      uint32_t (&off)[ROBOY_POLICY_LAYOUT_WORDS]) {
    fill_generic_step_params(env, p, nullptr, nullptr, reward_dev, done_dev);
    p.cc.advance = T;
    p.done_bits = nullptr;   // the done-index list belongs to single steps
    return roboy_policy_layout(env->D, env->A, off);
}

static int policy_rollout_common(roboy_env *env, bool tensor_cores, bool exact, uint32_t T, const float *image_dev, uint64_t noise_seed,
                                 float *obs_dev, float *actions_dev, float *logp_dev, float *values_dev, float *reward_dev,
                                 uint8_t *done_dev, float *noise_dev, int envs_per_thread, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!image_dev || !obs_dev || !actions_dev || !logp_dev || !values_dev || !reward_dev || !done_dev)
        return fail(ROBOY_E_ARG, "NULL device pointer");
    if (((uintptr_t)image_dev & 15) || ((uintptr_t)actions_dev & 15) || (noise_dev && ((uintptr_t)noise_dev & 15)))
        return fail(ROBOY_E_ARG, "image, actions and noise must be 16-byte aligned");
    if ((uintptr_t)obs_dev & 3) return fail(ROBOY_E_ARG, "obs must be 4-byte aligned");
    if (envs_per_thread < 0 || envs_per_thread > (tensor_cores ? 3 : 2))
        return fail(ROBOY_E_ARG, "envs_per_thread must be 0, 1 or 2 (tensor-core variant: 0..3)");
    if (!env->msj_shaped && tensor_cores)
        return fail(ROBOY_E_ARG, "the tensor-core policy rollout is built for MSJ-shaped robots (3 joints, 8 tendons, uniform "
                                 "bounds); other robots run the float32 rollout, roboy_policy_rollout");
    if (!env->msj_shaped && envs_per_thread > 1)
        return fail(ROBOY_E_ARG, "the policy rollout of robots other than MSJ runs one env per thread (envs_per_thread 0 or 1)");
    if (T == 0) return ROBOY_OK;
    DeviceGuard g(env->device);
    env->goal_sub = 1;
    if (!env->msj_shaped) {
        GStepParams p;
        GPolicyParams q{};
        if (fill_generic_policy_launch(env, T, reward_dev, done_dev, p, q.off) != ROBOY_OK) return ROBOY_E_ARG;
        q.image = image_dev;
        q.T = T;
        q.obs_aligned = (((uintptr_t)obs_dev & 15) == 0) && (env->cfg.n_envs * env->D * sizeof(float)) % 16 == 0;
        q.obs = obs_dev;
        q.actions = actions_dev;
        q.logp = logp_dev;
        q.values = values_dev;
        q.noise = noise_dev;
        q.noise_keys = make_philox_keys(noise_seed);
        CUDA_TRY(launch_generic_policy_rollout(p, q, env->sm_count, (cudaStream_t)stream));
        env->launches++;
        return ROBOY_OK;
    }
    StepParams p;
    fill_step_params(env, p, nullptr, obs_dev, reward_dev, done_dev);
    p.cc.advance = T;
    p.done_bits = nullptr;
    PolicyParams q{};
    q.image = image_dev;
    q.T = T;
    q.obs_aligned = (((uintptr_t)obs_dev & 15) == 0) && (env->cfg.n_envs * ROBOY_DIM_OBS * sizeof(float)) % 16 == 0;
    q.obs = obs_dev;
    q.actions = actions_dev;
    q.logp = logp_dev;
    q.values = values_dev;
    q.noise = noise_dev;
    q.noise_keys = make_philox_keys(noise_seed);
    if (tensor_cores)
        CUDA_TRY(launch_policy_rollout_tc(p, q, env->cfg.joint_vel_penalty, env->cfg.bonus_for_goal, env->cfg.auto_reset,
                                          env->fastdiv == kDivProved, env->sm_count, envs_per_thread, exact, (cudaStream_t)stream));
    else
        CUDA_TRY(launch_policy_rollout(p, q, env->cfg.joint_vel_penalty, env->cfg.bonus_for_goal, env->cfg.auto_reset,
                                       env->fastdiv == kDivProved, env->sm_count, envs_per_thread, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_policy_rollout(roboy_env *env, uint32_t T, const float *image_dev, uint64_t noise_seed, float *obs_dev,
                         float *actions_dev, float *logp_dev, float *values_dev, float *reward_dev, uint8_t *done_dev,
                         float *noise_dev, int envs_per_thread, void *stream) {
    return policy_rollout_common(env, false, true, T, image_dev, noise_seed, obs_dev, actions_dev, logp_dev, values_dev, reward_dev,
                                 done_dev, noise_dev, envs_per_thread, stream);
}

int roboy_policy_rollout_tc(roboy_env *env, uint32_t T, const float *tc_image_dev, uint64_t noise_seed, float *obs_dev,
                            float *actions_dev, float *logp_dev, float *values_dev, float *reward_dev, uint8_t *done_dev,
                            float *noise_dev, int tiles_per_group, int exact, void *stream) {
    return policy_rollout_common(env, true, exact != 0, T, tc_image_dev, noise_seed, obs_dev, actions_dev, logp_dev, values_dev, reward_dev,
                                 done_dev, noise_dev, tiles_per_group, stream);
}

int roboy_policy_evaluate(roboy_env *env, uint32_t T, const float *image_dev, float *obs_dev, uint32_t episodes,
                          double *returns_dev, uint32_t *lengths_dev, uint8_t *reached_dev, uint32_t *completed_dev,
                          void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!env->cfg.auto_reset)
        return fail(ROBOY_E_ARG, "roboy_policy_evaluate needs auto_reset: without it no new episode ever starts");
    if (!image_dev || !obs_dev || !returns_dev || !lengths_dev || !reached_dev || !completed_dev)
        return fail(ROBOY_E_ARG, "NULL device pointer");
    if ((uintptr_t)image_dev & 15) return fail(ROBOY_E_ARG, "image must be 16-byte aligned");
    if ((uintptr_t)obs_dev & 3) return fail(ROBOY_E_ARG, "obs must be 4-byte aligned");
    if (T == 0) return ROBOY_OK;
    DeviceGuard g(env->device);
    env->goal_sub = 1;
    // every robot, MSJ-shaped ones included, on the generic env step
    GStepParams p;
    GEvalParams q{};
    if (fill_generic_policy_launch(env, T, nullptr, nullptr, p, q.off) != ROBOY_OK) return ROBOY_E_ARG;
    q.image = image_dev;
    q.T = T;
    q.episodes = episodes;
    q.obs_aligned = ((uintptr_t)obs_dev & 15) == 0;   // one [n][3J] block: every chunk of 32 rows starts 16-byte aligned
    q.obs = obs_dev;
    q.returns = returns_dev;
    q.lengths = lengths_dev;
    q.reached = reached_dev;
    q.completed = completed_dev;
    CUDA_TRY(launch_generic_policy_evaluate(p, q, env->sm_count, (cudaStream_t)stream));
    env->launches++;
    return ROBOY_OK;
}

int roboy_policy_tc_geometry(roboy_env *env, int tiles_per_group, int exact, int *grid, int *block, int *smem_bytes, int *tpg) {
    if (check_env(env)) return ROBOY_E_ARG;
    const PolicyGeom geo = policy_tc_geometry(env->cfg.n_envs, env->sm_count, tiles_per_group, exact != 0);
    if (grid) *grid = geo.grid;
    if (block) *block = geo.block;
    if (smem_bytes) *smem_bytes = geo.smem;
    if (tpg) *tpg = geo.envs_per_thread;
    return ROBOY_OK;
}

int roboy_policy_layout(int dim_obs, int dim_action, uint32_t *offsets) {
    if (!offsets) return fail(ROBOY_E_ARG, "NULL offsets");
    if (dim_obs < 3 || dim_obs > 3 * kMaxJoint || dim_obs % 3 != 0 || dim_action < 1 || dim_action > kMaxAction)
        return fail(ROBOY_E_ARG, "policy dims must be dim_obs = 3J with J in 1..%d and dim_action in 1..%d", kMaxJoint,
                    kMaxAction);
    const uint32_t D = (uint32_t)dim_obs, A8 = ((uint32_t)dim_action + 7) / 8 * 8, H = ROBOY_POLICY_HIDDEN;
    uint32_t *o = offsets;
    o[ROBOY_POLICY_LAYOUT_W1] = 0;
    o[ROBOY_POLICY_LAYOUT_B1] = H * D;
    o[ROBOY_POLICY_LAYOUT_W2] = H * D + H;
    o[ROBOY_POLICY_LAYOUT_B2] = H * D + H + H * H;
    o[ROBOY_POLICY_LAYOUT_W3] = H * D + 2 * H + H * H;
    o[ROBOY_POLICY_LAYOUT_VF_B3] = o[ROBOY_POLICY_LAYOUT_W3] + H * 8;
    o[ROBOY_POLICY_LAYOUT_PI_B3] = o[ROBOY_POLICY_LAYOUT_W3] + H * A8;
    o[ROBOY_POLICY_LAYOUT_VF] = 0;
    o[ROBOY_POLICY_LAYOUT_PI] = o[ROBOY_POLICY_LAYOUT_VF_B3] + 8;
    o[ROBOY_POLICY_LAYOUT_STD] = o[ROBOY_POLICY_LAYOUT_PI] + o[ROBOY_POLICY_LAYOUT_PI_B3] + A8;
    o[ROBOY_POLICY_LAYOUT_LOGNORM] = o[ROBOY_POLICY_LAYOUT_STD] + A8;
    o[ROBOY_POLICY_LAYOUT_FLOATS] = (o[ROBOY_POLICY_LAYOUT_LOGNORM] + 1 + 3) / 4 * 4;
    return ROBOY_OK;
}

// Bytes from dev_ptr to the end of the device allocation holding it (cuMemGetAddressRange through the runtime's
// driver entry point: no link against libcuda).  false if dev_ptr is not in a device allocation.
static bool allocation_room(const void *dev_ptr, uint64_t *room) {
    typedef int (*GetRange)(unsigned long long *base, size_t *size, unsigned long long ptr);
    static GetRange get_range = nullptr;
    if (!get_range) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess || !fn)
            return false;
        get_range = (GetRange)fn;
    }
    unsigned long long base = 0;
    size_t size = 0;
    if (get_range(&base, &size, (unsigned long long)(uintptr_t)dev_ptr) != 0) return false;
    *room = base + size - (uint64_t)(uintptr_t)dev_ptr;
    return true;
}

int roboy_ppo_workspace_bytes(int dim_obs, int dim_action, uint64_t M, uint64_t *bytes) {
    if (!bytes) return fail(ROBOY_E_ARG, "NULL bytes");
    uint32_t off[ROBOY_POLICY_LAYOUT_WORDS];
    if (roboy_policy_layout(dim_obs, dim_action, off) != ROBOY_OK) return ROBOY_E_ARG;
    if (M == 0) return fail(ROBOY_E_ARG, "the minibatch is empty (M == 0)");
    *bytes = ppo_workspace_bytes(off[ROBOY_POLICY_LAYOUT_FLOATS], M);
    return ROBOY_OK;
}

int roboy_ppo_grad(int dim_obs, int dim_action, const float *image_dev, uint64_t M, const int64_t *index_dev,
                   uint64_t n_rows, const float *obs_dev, const float *actions_dev, const float *logp_dev,
                   const float *values_dev, const float *ret_dev, float clip_range, float clip_range_vf,
                   float ent_coef, float vf_coef, float *grad_dev, double *stats_dev, void *workspace_dev,
                   void *stream) {
    PpoParams p{};
    if (roboy_policy_layout(dim_obs, dim_action, p.off) != ROBOY_OK) return ROBOY_E_ARG;
    if (M == 0) return fail(ROBOY_E_ARG, "the minibatch is empty (M == 0)");
    if (!image_dev || !index_dev || !obs_dev || !actions_dev || !logp_dev || !values_dev || !ret_dev || !grad_dev ||
        !stats_dev || !workspace_dev)
        return fail(ROBOY_E_ARG, "NULL device pointer");
    if ((uintptr_t)image_dev & 15) return fail(ROBOY_E_ARG, "image must be 16-byte aligned");
    if ((uintptr_t)workspace_dev & 7) return fail(ROBOY_E_ARG, "workspace must be 8-byte aligned");
    p.P = p.off[ROBOY_POLICY_LAYOUT_FLOATS];
    // the bytes from workspace_dev to the end of the allocation that holds it (a pool allocator's block may be larger
    // than the caller's tensor: this catches what would run past the allocation)
    const uint64_t need = ppo_workspace_bytes(p.P, M);
    uint64_t room = 0;
    if (!allocation_room(workspace_dev, &room) || room < need)
        return fail(ROBOY_E_ARG, "the workspace holds %llu bytes; roboy_ppo_workspace_bytes asks for %llu",
                    (unsigned long long)room, (unsigned long long)need);
    p.J = dim_obs / 3;
    p.A = dim_action;
    p.M = M;
    p.n_rows = n_rows;
    p.image = image_dev;
    p.index = index_dev;
    p.obs = obs_dev;
    p.actions = actions_dev;
    p.logp = logp_dev;
    p.values = values_dev;
    p.ret = ret_dev;
    p.clip = clip_range;
    p.clip_vf = clip_range_vf;
    p.ent_coef = ent_coef;
    p.vf_coef = vf_coef;
    p.grad = grad_dev;
    p.stats = stats_dev;
    CUDA_TRY(launch_ppo_grad(p, workspace_dev, (cudaStream_t)stream));
    return ROBOY_OK;
}

int roboy_policy_geometry(roboy_env *env, int envs_per_thread, int *grid, int *block, int *smem_bytes, int *ept) {
    if (check_env(env)) return ROBOY_E_ARG;
    PolicyGeom geo;
    if (env->msj_shaped) {
        geo = policy_geometry(env->cfg.n_envs, env->sm_count, envs_per_thread);
    } else {
        if (envs_per_thread < 0 || envs_per_thread > 1)
            return fail(ROBOY_E_ARG, "the policy rollout of robots other than MSJ runs one env per thread (envs_per_thread 0 or 1)");
        uint32_t off[ROBOY_POLICY_LAYOUT_WORDS];
        if (roboy_policy_layout(env->D, env->A, off) != ROBOY_OK) return ROBOY_E_ARG;
        geo = generic_policy_geometry(env->spec.J, off[ROBOY_POLICY_LAYOUT_FLOATS], env->cfg.n_envs, env->sm_count);
    }
    if (grid) *grid = geo.grid;
    if (block) *block = geo.block;
    if (smem_bytes) *smem_bytes = geo.smem;
    if (ept) *ept = geo.envs_per_thread;
    return ROBOY_OK;
}

int roboy_enable_done_index(roboy_env *env, int enable) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    if (enable && !env->done_bits) {
        const uint64_t n_words = (env->cfg.n_envs + 31) / 32;
        const uint64_t n_tiles = (n_words + kDoneTileWords - 1) / kDoneTileWords;
        uint32_t *bits = nullptr, *tile_off = nullptr;
        unsigned int *ticket = nullptr;
        cudaError_t err = cudaMalloc((void **)&bits, sizeof(uint32_t) * n_words);
        if (err == cudaSuccess) err = cudaMalloc((void **)&tile_off, sizeof(uint32_t) * (n_tiles + 1));
        if (err == cudaSuccess) err = cudaMalloc((void **)&ticket, sizeof(unsigned int));
        if (err == cudaSuccess) err = cudaMemset(bits, 0, sizeof(uint32_t) * n_words);
        if (err == cudaSuccess) err = cudaMemset(ticket, 0, sizeof(unsigned int));
        if (err != cudaSuccess) {
            cudaFree(bits); cudaFree(tile_off); cudaFree(ticket);
            cudaGetLastError();
            return fail(ROBOY_E_ALLOC, "roboy_enable_done_index: %s", cudaGetErrorString(err));
        }
        env->done_bits = bits;
        env->done_tile_off = tile_off;
        env->done_ticket = ticket;
    } else if (!enable && env->done_bits) {
        CUDA_TRY(cudaDeviceSynchronize());
        cudaFree(env->done_bits); cudaFree(env->done_tile_off); cudaFree(env->done_ticket);
        env->done_bits = nullptr; env->done_tile_off = nullptr; env->done_ticket = nullptr;
    }
    return ROBOY_OK;
}

int roboy_done_indices(roboy_env *env, int32_t *idx_dev, uint64_t capacity, uint32_t *count_dev, float *terminal_rows_dev,
                       void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!env->done_bits) return fail(ROBOY_E_ARG, "roboy_enable_done_index(env, 1) first");
    if (!count_dev || (!idx_dev && capacity)) return fail(ROBOY_E_ARG, "NULL device pointer");
    if (terminal_rows_dev && !env->terminal_obs) return fail(ROBOY_E_ARG, "terminal rows requested but no terminal-obs buffer is set");
    DeviceGuard g(env->device);
    DoneIndexParams p{};
    p.bits = env->done_bits;
    p.n_words = (uint32_t)((env->cfg.n_envs + 31) / 32);
    p.n_envs = (uint32_t)env->cfg.n_envs;
    p.tile_off = env->done_tile_off;
    p.ticket = env->done_ticket;
    p.idx = idx_dev;
    p.capacity = capacity > 0xffffffffull ? 0xffffffffu : (uint32_t)capacity;
    p.count = count_dev;
    p.terminal_obs = env->terminal_obs;
    p.terminal_rows = terminal_rows_dev;
    p.obs_dim = env->D;
    CUDA_TRY(launch_done_index(p, (cudaStream_t)stream));
    env->launches += 2;
    return ROBOY_OK;
}

int roboy_launch_count(roboy_env *env, uint64_t *launches) {
    if (check_env(env) || !launches) return fail(ROBOY_E_ARG, "NULL argument");
    *launches = env->launches;
    return ROBOY_OK;
}

int roboy_robot_dims(roboy_env *env, int *dim_joint, int *dim_action, int *dim_obs, int *msj_kernels) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (dim_joint) *dim_joint = env->J;
    if (dim_action) *dim_action = env->A;
    if (dim_obs) *dim_obs = env->D;
    if (msj_kernels) *msj_kernels = env->msj_shaped ? 1 : 0;
    return ROBOY_OK;
}

int roboy_fast_division(roboy_env *env, int *proved) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!proved) return fail(ROBOY_E_ARG, "NULL argument");
    *proved = env->msj_shaped ? (env->fastdiv != kDivIeee ? 1 : 0) : env->spec.fastdiv;
    return ROBOY_OK;
}

int roboy_penalty_float32(roboy_env *env, int *on) {
    if (check_env(env)) return ROBOY_E_ARG;
    if (!on) return fail(ROBOY_E_ARG, "NULL argument");
    *on = env->spec.pen.on;
    return ROBOY_OK;
}

int roboy_null_step(roboy_env *env, void *stream) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    CUDA_TRY(launch_null_step(env->cfg.n_envs, env->cfg.joint_vel_penalty, env->cfg.bonus_for_goal, env->cfg.auto_reset,
                              env->fastdiv, env->sm_count, (cudaStream_t)stream));
    return ROBOY_OK;
}

int roboy_step_geometry(roboy_env *env, int *grid, int *block, int *smem_bytes) {
    if (check_env(env)) return ROBOY_E_ARG;
    DeviceGuard g(env->device);
    if (!env->msj_shaped) {
        int gr, bl, sm;
        generic_step_geometry(env->J, env->cfg.n_envs, env->sm_count, &gr, &bl, &sm);
        if (grid) *grid = gr;
        if (block) *block = bl;
        if (smem_bytes) *smem_bytes = sm;
        return ROBOY_OK;
    }
    const LaunchGeom geo = step_geometry(env->cfg.n_envs, env->cfg.joint_vel_penalty, env->cfg.bonus_for_goal,
                                         env->cfg.auto_reset, env->fastdiv, env->sm_count);
    if (grid) *grid = geo.grid;
    if (block) *block = geo.block;
    if (smem_bytes) *smem_bytes = geo.smem;
    return ROBOY_OK;
}

}  // extern "C"
