// sm_100a kernels of the PPO2 update: stable-baselines 2's clipped-surrogate loss over one minibatch of a rollout and
// its gradient with respect to every MlpPolicy parameter, in float32 FFMA, for every robot (J = 1..15 joints, A = 1..64
// tendons).  The semantics are stated in include/roboy_b200.h (roboy_ppo_grad).
//
// Three launches:
//   ppo_adv_stats_kernel    a fixed grid of kPpoAdvBlocks CTAs sums adv = ret - value and adv^2 (float64) and counts the
//                           indices outside [0, n_rows), one partial per CTA;
//   ppo_grad_kernel<J>      one CTA per slot (slots = min(tiles, kPpoMaxSlots), a function of M only).  Slot b works on
//                           the 64-sample tiles b, b + slots, ...; per tile it gathers the samples by index, runs both
//                           networks forward (h1, h2 kept in shared memory), forms the per-sample output deltas and
//                           back-propagates them through both tanh layers.  The gradient accumulator is the policy image's
//                           layout in shared memory; every entry has one owner thread, which adds the tile's sum to it, so
//                           no float value takes an atomic.  The slot's accumulator and its loss partials go to the
//                           workspace;
//   ppo_grad_reduce_kernel  sums the slots, in slot order, in float64, into the gradient image and the statistics.
// Nothing depends on the device, the SM count or the stream: the result is a function of the inputs, bit for bit.
//
// The backward pass reads the weights from the image as the forward pass does: the image stores W^T (row = input), and
// the delta of hidden unit j is a dot product over row j of W^T, so neither pass needs another copy of the weights.
//
// Accuracy: the gradient must stay within a few times float32 autograd's error of float64 autograd.  So the forward
// pass uses tanhf (within 2 ulp), not the rollouts' tanh_mufu: tanh_mufu's error (a few 1e-7) is
// systematic and does not average out of a minibatch mean, e.g. d b3 of the value net when the values fit the returns.
// The output layers add their bias after the 64-term sum, as a Linear layer does: a value net's bias of order
// r / (1 - gamma) would otherwise round every partial sum at its magnitude.
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/roboy_b200.h"
#include "policy_common.cuh"
#include "roboy_generic.cuh"
#include "roboy_policy.cuh"

namespace roboy {
namespace {

constexpr int kTs = kPpoTile;          // samples per tile
constexpr int kTsp = kTs + 4;          // row stride of the [rows][samples] tiles in shared memory (float4 along samples)
constexpr int kHid = ROBOY_POLICY_HIDDEN;

__host__ __device__ constexpr int d4_of(int D) { return (D + 3) & ~3; }

// Dynamic shared memory of ppo_grad_kernel: accumulator [P] | h1, h2 of the value net, h1, h2 of the policy net
// [4][64][kTsp] | observations [D4][kTsp] | z, then d mean [A8][kTsp] | d logp [kTs] | d value [kTs] | double [4 warps][4]
// + [4]
__host__ __device__ constexpr int ppo_smem_bytes(int D, int A8, uint32_t P) {
    return (int)sizeof(float) * ((int)P + (4 * kHid + d4_of(D) + A8) * kTsp + 2 * kTs) +
           (int)sizeof(double) * (4 * (kPpoThreads / 32) + 4);
}

__global__ void __launch_bounds__(kPpoAdvThreads) ppo_adv_stats_kernel(const __grid_constant__ PpoParams p) {
    double s1 = 0.0, s2 = 0.0, bad = 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.M; i += (uint64_t)gridDim.x * blockDim.x) {
        const int64_t idx = p.index[i];
        if (idx < 0 || (uint64_t)idx >= p.n_rows) {
            bad += 1.0;
            continue;
        }
        const double a = (double)__fsub_rn(p.ret[idx], p.values[idx]);   // SB2: advs = returns - values, in float32
        s1 += a;
        s2 = fma(a, a, s2);
    }
    __shared__ double red[kPpoAdvThreads / 32][3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s1 = warp_sum_d(s1);
    s2 = warp_sum_d(s2);
    bad = warp_sum_d(bad);
    if (lane == 0) {
        red[warp][0] = s1;
        red[warp][1] = s2;
        red[warp][2] = bad;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double v = 0.0;
        for (int w = 0; w < kPpoAdvThreads / 32; ++w) v += red[w][threadIdx.x];
        p.adv_part[blockIdx.x * 3 + threadIdx.x] = v;
    }
}

// acc[r][c] += sum over the tile's samples of a[r][s] * b[c][s], for the r < r_lim, c < c_lim of an R x C block (R, C
// multiples of 4); a and b are [rows][kTsp] in shared memory, acc[r * acc_rs + c].  A thread owns rows rb + i * R/4 and
// columns cb + j * C/4 (strided, so that the lanes' float4 reads of b fall in different banks).
__device__ __forceinline__ void acc_outer(const float *__restrict__ a, int R, int r_lim, const float *__restrict__ b, int C,
                                          int c_lim, float *__restrict__ acc, int acc_rs) {
    const int rq = R / 4, cq = C / 4;
    for (int blk = threadIdx.x; blk < rq * cq; blk += blockDim.x) {
        const int rb = blk / cq, cb = blk % cq;
        float c[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) c[i][j] = 0.0f;
#pragma unroll 2
        for (int s = 0; s < kTs; s += 4) {
            float4 av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = *reinterpret_cast<const float4 *>(a + (rb + i * rq) * kTsp + s);
#pragma unroll
            for (int j = 0; j < 4; ++j) bv[j] = *reinterpret_cast<const float4 *>(b + (cb + j * cq) * kTsp + s);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    c[i][j] = fmaf(av[i].x, bv[j].x, c[i][j]);
                    c[i][j] = fmaf(av[i].y, bv[j].y, c[i][j]);
                    c[i][j] = fmaf(av[i].z, bv[j].z, c[i][j]);
                    c[i][j] = fmaf(av[i].w, bv[j].w, c[i][j]);
                }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = rb + i * rq, cc = cb + j * cq;
                if (r < r_lim && cc < c_lim) acc[r * acc_rs + cc] += c[i][j];
            }
    }
}

// acc[r] += sum over the tile's samples of a[r][s], rows r < R, a thread per row
__device__ __forceinline__ void acc_rowsum(const float *__restrict__ a, int R, float *__restrict__ acc, int tid0, int nthreads) {
    for (int r = (int)threadIdx.x - tid0; r >= 0 && r < R; r += nthreads) {
        float v = 0.0f;
        for (int s = 0; s < kTs; ++s) v = __fadd_rn(v, a[r * kTsp + s]);
        acc[r] += v;
    }
}

// The tanh layer below an output delta: h[j][s] <- (sum_k WT[j * ldw + k] * d[k][s]) * (1 - h[j][s]^2), j < 64, k < K.
// WT is the image's W^T (row = input unit j), d is [K][kTsp] in shared memory; h turns from the layer's output into its
// pre-activation delta in place.  A thread owns rows jb + 16 i and the four samples 4 sb .. 4 sb + 3.
__device__ __forceinline__ void back_tanh(const float *__restrict__ WT, int ldw, int K, const float *__restrict__ d,
                                          float *__restrict__ h) {
    for (int blk = threadIdx.x; blk < 16 * (kTs / 4); blk += blockDim.x) {
        const int jb = blk / (kTs / 4), s = 4 * (blk % (kTs / 4));
        float c[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int e = 0; e < 4; ++e) c[i][e] = 0.0f;
#pragma unroll 2
        for (int k = 0; k < K; ++k) {
            const float4 dv = *reinterpret_cast<const float4 *>(d + k * kTsp + s);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float w = WT[(jb + 16 * i) * ldw + k];
                c[i][0] = fmaf(w, dv.x, c[i][0]);
                c[i][1] = fmaf(w, dv.y, c[i][1]);
                c[i][2] = fmaf(w, dv.z, c[i][2]);
                c[i][3] = fmaf(w, dv.w, c[i][3]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float4 *hp = reinterpret_cast<float4 *>(h + (jb + 16 * i) * kTsp + s);
            const float4 hv = *hp;
            *hp = make_float4(__fmul_rn(c[i][0], fmaf(-hv.x, hv.x, 1.0f)), __fmul_rn(c[i][1], fmaf(-hv.y, hv.y, 1.0f)),
                              __fmul_rn(c[i][2], fmaf(-hv.z, hv.z, 1.0f)), __fmul_rn(c[i][3], fmaf(-hv.w, hv.w, 1.0f)));
        }
    }
}

template <int J>
__global__ void __launch_bounds__(kPpoThreads, 1) ppo_grad_kernel(const __grid_constant__ PpoParams p) {
    constexpr int D = 3 * J, D4 = d4_of(D);
    const int A = p.A, A8 = (A + 7) & ~7;
    const uint32_t *off = p.off;
    extern __shared__ __align__(16) float smem[];
    float *acc = smem;
    float *hbuf = acc + p.P;                 // [4][64][kTsp]: value h1, value h2, policy h1, policy h2
    float *xs = hbuf + 4 * kHid * kTsp;      // [D4][kTsp]
    float *zs = xs + D4 * kTsp;              // [A8][kTsp]
    float *gs = zs + A8 * kTsp;              // [kTs] d loss / d logp_new
    float *dvs = gs + kTs;                   // [kTs] d loss / d value
    double *red = reinterpret_cast<double *>(dvs + kTs);   // [4 warps][4], then mean, std, 1 / M_valid
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (uint32_t i = tid; i < p.P; i += blockDim.x) acc[i] = 0.0f;
    for (int i = tid; i < (D4 - D) * kTsp; i += blockDim.x) xs[D * kTsp + i] = 0.0f;
    if (tid == 0) {
        double s1 = 0.0, s2 = 0.0, bad = 0.0;
        for (int b = 0; b < kPpoAdvBlocks; ++b) {
            s1 += p.adv_part[3 * b];
            s2 += p.adv_part[3 * b + 1];
            bad += p.adv_part[3 * b + 2];
        }
        const double mv = (double)p.M - bad;
        const double mean = mv > 0.0 ? s1 / mv : 0.0;
        red[16] = mean;
        red[17] = mv > 0.0 ? sqrt(fmax(s2 / mv - mean * mean, 0.0)) : 0.0;
        red[18] = mv > 0.0 ? 1.0 / mv : 0.0;
    }
    __syncthreads();
    const double adv_mean = red[16], adv_den = red[17] + 1e-8;
    const float inv_m = (float)red[18];

    const float *vf = p.image + off[ROBOY_POLICY_LAYOUT_VF];
    const float *pi = p.image + off[ROBOY_POLICY_LAYOUT_PI];
    const float *stdv = p.image + off[ROBOY_POLICY_LAYOUT_STD];
    const float lognorm = p.image[off[ROBOY_POLICY_LAYOUT_LOGNORM]];
    float *acc_vf = acc + off[ROBOY_POLICY_LAYOUT_VF], *acc_pi = acc + off[ROBOY_POLICY_LAYOUT_PI];
    const bool is_pi = tid >= kTs;
    const int s = tid & (kTs - 1);
    const float *net = is_pi ? pi : vf;
    float *h1 = hbuf + (is_pi ? 2 : 0) * kHid * kTsp, *h2 = h1 + kHid * kTsp;
    float *vh1 = hbuf, *vh2 = hbuf + kHid * kTsp, *ph1 = hbuf + 2 * kHid * kTsp, *ph2 = hbuf + 3 * kHid * kTsp;
    double st_pg = 0.0, st_vf = 0.0, st_kl = 0.0, st_clip = 0.0;
    const uint64_t n_tiles = (p.M + kTs - 1) / kTs;

    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // ---- gather: the sample's index, its observation into column s ----
        const uint64_t pos = tile * kTs + s;
        const int64_t idx = pos < p.M ? p.index[pos] : -1;
        const bool ok = idx >= 0 && (uint64_t)idx < p.n_rows;
        const size_t row = ok ? (size_t)idx : 0;
        if (!is_pi) {
#pragma unroll
            for (int k = 0; k < D; ++k) xs[k * kTsp + s] = ok ? p.obs[row * D + k] : 0.0f;
        }
        __syncthreads();

        // ---- forward: threads 0..63 the value net, 64..127 the policy net, one sample each ----
        {
            float2 a2[1][32];
            load_bias64<1>(net + off[ROBOY_POLICY_LAYOUT_B1], a2);
            dense64<1>(net + off[ROBOY_POLICY_LAYOUT_W1], xs + s, D, kTsp, 0, a2);
#pragma unroll
            for (int j2 = 0; j2 < 32; ++j2) {
                h1[(2 * j2) * kTsp + s] = tanhf(a2[0][j2].x);
                h1[(2 * j2 + 1) * kTsp + s] = tanhf(a2[0][j2].y);
            }
            load_bias64<1>(net + off[ROBOY_POLICY_LAYOUT_B2], a2);
            dense64<1>(net + off[ROBOY_POLICY_LAYOUT_W2], h1 + s, kHid, kTsp, 0, a2);
#pragma unroll
            for (int j2 = 0; j2 < 32; ++j2) {
                h2[(2 * j2) * kTsp + s] = tanhf(a2[0][j2].x);
                h2[(2 * j2 + 1) * kTsp + s] = tanhf(a2[0][j2].y);
            }
        }
        if (!is_pi) {
            // ---- value: vf_loss = 1/2 mean(max((v - R)^2, (v_clip - R)^2)) ----
            const float *w3 = vf + off[ROBOY_POLICY_LAYOUT_W3];
            float v = 0.0f;
            for (int j = 0; j < kHid; ++j) v = fmaf(h2[j * kTsp + s], w3[j * 8], v);
            v = __fadd_rn(v, vf[off[ROBOY_POLICY_LAYOUT_VF_B3]]);   // the bias last, as a Linear layer adds it
            float dv = 0.0f;
            if (ok) {
                const float v_old = p.values[row], R = p.ret[row];
                const float d1 = __fsub_rn(v, R), l1 = __fmul_rn(d1, d1);
                if (p.clip_vf >= 0.0f) {
                    const float e = p.clip_vf, dd = __fsub_rn(v, v_old);
                    const float d2 = __fsub_rn(__fadd_rn(v_old, fminf(fmaxf(dd, -e), e)), R), l2 = __fmul_rn(d2, d2);
                    const bool first = l1 >= l2;                // TF's maximum: the first argument at a tie
                    const bool inside = dd >= -e && dd <= e;    // clip_by_value passes the gradient inside the range
                    // as products (not selects), so that a NaN reaches the gradient where autograd's products carry it
                    dv = __fadd_rn(__fmul_rn(d1, first ? 1.0f : 0.0f), __fmul_rn(d2, (!first && inside) ? 1.0f : 0.0f));
                    st_vf += (double)(first ? l1 : l2);
                } else {
                    dv = d1;
                    st_vf += (double)l1;
                }
                dv = __fmul_rn(__fmul_rn(dv, p.vf_coef), inv_m);   // d (vf_coef / 2 mean(l)) / dv = vf_coef (v - .) / M
            }
            dvs[s] = dv;
        } else {
            // ---- policy: z = (a - mean) / std, logp_new, ratio, the clipped surrogate ----
            const float *w3 = pi + off[ROBOY_POLICY_LAYOUT_W3], *b3 = pi + off[ROBOY_POLICY_LAYOUT_PI_B3];
            float zz = 0.0f;
            for (int c = 0; c < A8 / 8; ++c) {
                float o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = 0.0f;
                for (int j = 0; j < kHid; ++j) {
                    const float t = h2[j * kTsp + s];
                    const float4 wa = reinterpret_cast<const float4 *>(w3 + j * A8 + 8 * c)[0];
                    const float4 wb = reinterpret_cast<const float4 *>(w3 + j * A8 + 8 * c)[1];
                    o[0] = fmaf(t, wa.x, o[0]); o[1] = fmaf(t, wa.y, o[1]); o[2] = fmaf(t, wa.z, o[2]); o[3] = fmaf(t, wa.w, o[3]);
                    o[4] = fmaf(t, wb.x, o[4]); o[5] = fmaf(t, wb.y, o[5]); o[6] = fmaf(t, wb.z, o[6]); o[7] = fmaf(t, wb.w, o[7]);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int k = 8 * c + i;
                    const float mean = __fadd_rn(o[i], b3[k]);
                    const float z = (ok && k < A) ? __fdiv_rn(__fsub_rn(p.actions[row * A + k], mean), stdv[k]) : 0.0f;
                    zs[k * kTsp + s] = z;
                    zz = fmaf(z, z, zz);
                }
            }
            float g = 0.0f;
            if (ok) {
                const float dl = __fsub_rn(fmaf(-0.5f, zz, lognorm), p.logp[row]);   // logp_new - logp_old
                const float ratio = expf(dl);
                const float adv = (float)(((double)__fsub_rn(p.ret[row], p.values[row]) - adv_mean) / adv_den);
                const float e = p.clip, lo = __fsub_rn(1.0f, e), hi = __fadd_rn(1.0f, e);
                const float pg1 = __fmul_rn(-adv, ratio), pg2 = __fmul_rn(-adv, fminf(fmaxf(ratio, lo), hi));
                const bool first = pg1 >= pg2;
                const bool inside = ratio >= lo && ratio <= hi;
                const float dratio = __fadd_rn(__fmul_rn(-adv, first ? 1.0f : 0.0f), __fmul_rn(-adv, (!first && inside) ? 1.0f : 0.0f));
                g = __fmul_rn(__fmul_rn(dratio, ratio), inv_m);    // d loss / d logp_new = d loss / d ratio * ratio
                st_pg += (double)(first ? pg1 : pg2);
                st_kl += (double)dl * (double)dl;
                st_clip += fabsf(__fsub_rn(ratio, 1.0f)) > e ? 1.0 : 0.0;
            }
            gs[s] = g;
        }
        __syncthreads();

        // ---- output deltas: d mean[k][s] = g z / std into zs; d log_std[k] += sum_s g (z^2 - 1); d b3 of the value net ----
        if (tid < A) {
            const float sd = stdv[tid];
            float dls = 0.0f;
            for (int j = 0; j < kTs; ++j) {
                const float z = zs[tid * kTsp + j], g = gs[j];
                dls = fmaf(g, fmaf(z, z, -1.0f), dls);
                zs[tid * kTsp + j] = __fdiv_rn(__fmul_rn(g, z), sd);
            }
            acc[off[ROBOY_POLICY_LAYOUT_STD] + tid] += dls;
        }
        if (tid == kPpoThreads - 1) {
            float v = 0.0f;
            for (int j = 0; j < kTs; ++j) v = __fadd_rn(v, dvs[j]);
            acc_vf[off[ROBOY_POLICY_LAYOUT_VF_B3]] += v;
        }
        __syncthreads();

        // ---- last layers: dW3, db3 ----
        acc_outer(ph2, kHid, kHid, zs, A8, A, acc_pi + off[ROBOY_POLICY_LAYOUT_W3], A8);
        acc_rowsum(zs, A, acc_pi + off[ROBOY_POLICY_LAYOUT_PI_B3], 0, kTs);
        if (tid >= kTs) {
            const int j = tid - kTs;
            float v = 0.0f;
            for (int k = 0; k < kTs; ++k) v = fmaf(vh2[j * kTsp + k], dvs[k], v);
            acc_vf[off[ROBOY_POLICY_LAYOUT_W3] + j * 8] += v;
        }
        __syncthreads();

        // ---- through tanh(h2): h2 <- d pre-activation of layer 2 ----
        back_tanh(pi + off[ROBOY_POLICY_LAYOUT_W3], A8, A8, zs, ph2);
        {
            const float *w3 = vf + off[ROBOY_POLICY_LAYOUT_W3];
            for (int i = tid; i < kHid * kTs; i += blockDim.x) {
                const int j = i / kTs, k = i % kTs;
                const float h = vh2[j * kTsp + k];
                vh2[j * kTsp + k] = __fmul_rn(__fmul_rn(w3[j * 8], dvs[k]), fmaf(-h, h, 1.0f));
            }
        }
        __syncthreads();

        // ---- layer 2: dW2 = h1 (x) d2, db2 ----
        acc_outer(vh1, kHid, kHid, vh2, kHid, kHid, acc_vf + off[ROBOY_POLICY_LAYOUT_W2], kHid);
        acc_outer(ph1, kHid, kHid, ph2, kHid, kHid, acc_pi + off[ROBOY_POLICY_LAYOUT_W2], kHid);
        acc_rowsum(vh2, kHid, acc_vf + off[ROBOY_POLICY_LAYOUT_B2], 0, kTs);
        acc_rowsum(ph2, kHid, acc_pi + off[ROBOY_POLICY_LAYOUT_B2], kTs, kTs);
        __syncthreads();

        // ---- through tanh(h1): h1 <- d pre-activation of layer 1 ----
        back_tanh(vf + off[ROBOY_POLICY_LAYOUT_W2], kHid, kHid, vh2, vh1);
        back_tanh(pi + off[ROBOY_POLICY_LAYOUT_W2], kHid, kHid, ph2, ph1);
        __syncthreads();

        // ---- layer 1: dW1 = x (x) d1, db1 ----
        acc_outer(xs, D4, D, vh1, kHid, kHid, acc_vf + off[ROBOY_POLICY_LAYOUT_W1], kHid);
        acc_outer(xs, D4, D, ph1, kHid, kHid, acc_pi + off[ROBOY_POLICY_LAYOUT_W1], kHid);
        acc_rowsum(vh1, kHid, acc_vf + off[ROBOY_POLICY_LAYOUT_B1], 0, kTs);
        acc_rowsum(ph1, kHid, acc_pi + off[ROBOY_POLICY_LAYOUT_B1], kTs, kTs);
        __syncthreads();
    }

    // ---- the slot's partials ----
    float *out = p.grad_part + (size_t)blockIdx.x * p.P;
    for (uint32_t i = tid; i < p.P; i += blockDim.x) out[i] = acc[i];
    const double st[4] = {warp_sum_d(st_pg), warp_sum_d(st_vf), warp_sum_d(st_kl), warp_sum_d(st_clip)};
    if (lane == 0)
        for (int k = 0; k < 4; ++k) red[warp * 4 + k] = st[k];
    __syncthreads();
    if (tid < 4) {
        double v = 0.0;
        for (int w = 0; w < kPpoThreads / 32; ++w) v += red[w * 4 + tid];
        p.stat_part[(size_t)blockIdx.x * 4 + tid] = v;
    }
}

__global__ void __launch_bounds__(256) ppo_grad_reduce_kernel(const __grid_constant__ PpoParams p, uint32_t slots) {
    const uint32_t std0 = p.off[ROBOY_POLICY_LAYOUT_STD];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < p.P; i += gridDim.x * blockDim.x) {
        double g = 0.0;
        for (uint32_t b = 0; b < slots; ++b) g += (double)p.grad_part[(size_t)b * p.P + i];
        if (i >= std0 && i < std0 + (uint32_t)p.A) g -= (double)p.ent_coef;   // d (-ent_coef entropy) / d log_std_k
        p.grad[i] = (float)g;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        double s1 = 0.0, s2 = 0.0, bad = 0.0, st[4] = {0.0, 0.0, 0.0, 0.0};
        for (int b = 0; b < kPpoAdvBlocks; ++b) {
            s1 += p.adv_part[3 * b];
            s2 += p.adv_part[3 * b + 1];
            bad += p.adv_part[3 * b + 2];
        }
        for (uint32_t b = 0; b < slots; ++b)
            for (int k = 0; k < 4; ++k) st[k] += p.stat_part[(size_t)b * 4 + k];
        const double mv = (double)p.M - bad, inv = mv > 0.0 ? 1.0 / mv : 0.0;
        const double mean = s1 * inv;
        const double pg = st[0] * inv, vfl = 0.5 * st[1] * inv;
        const double entropy = 0.5 * p.A - (double)p.image[p.off[ROBOY_POLICY_LAYOUT_LOGNORM]];   // sum(log_std) + A/2 log(2 pi e)
        double *o = p.stats;
        o[ROBOY_PPO_STAT_LOSS] = pg - (double)p.ent_coef * entropy + (double)p.vf_coef * vfl;
        o[ROBOY_PPO_STAT_PG_LOSS] = pg;
        o[ROBOY_PPO_STAT_VF_LOSS] = vfl;
        o[ROBOY_PPO_STAT_ENTROPY] = entropy;
        o[ROBOY_PPO_STAT_APPROXKL] = 0.5 * st[2] * inv;
        o[ROBOY_PPO_STAT_CLIPFRAC] = st[3] * inv;
        o[ROBOY_PPO_STAT_ADV_MEAN] = mean;
        o[ROBOY_PPO_STAT_ADV_STD] = mv > 0.0 ? sqrt(fmax(s2 * inv - mean * mean, 0.0)) : 0.0;
        o[ROBOY_PPO_STAT_BAD_INDICES] = bad;
    }
}

}  // namespace

uint32_t ppo_slots(uint64_t M) {
    const uint64_t tiles = (M + kTs - 1) / kTs;
    return (uint32_t)(tiles < (uint64_t)kPpoMaxSlots ? tiles : (uint64_t)kPpoMaxSlots);
}

uint64_t ppo_workspace_bytes(uint32_t P, uint64_t M) {
    const uint64_t slots = ppo_slots(M);
    return sizeof(double) * (3ull * kPpoAdvBlocks + 4ull * slots) + sizeof(float) * (uint64_t)P * slots;
}

cudaError_t launch_ppo_grad(PpoParams p, void *workspace, cudaStream_t stream) {
    const uint32_t slots = ppo_slots(p.M);
    p.adv_part = static_cast<double *>(workspace);
    p.stat_part = p.adv_part + 3 * kPpoAdvBlocks;
    p.grad_part = reinterpret_cast<float *>(p.stat_part + 4ull * slots);
    ppo_adv_stats_kernel<<<kPpoAdvBlocks, kPpoAdvThreads, 0, stream>>>(p);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    const int smem = ppo_smem_bytes(3 * p.J, (p.A + 7) & ~7, p.P);
    switch (p.J) {
#define ROBOY_PPO_CASE(JJ)                                                                                 \
        case JJ:                                                                                           \
            err = cudaFuncSetAttribute(ppo_grad_kernel<JJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); \
            if (err != cudaSuccess) return err;                                                            \
            ppo_grad_kernel<JJ><<<slots, kPpoThreads, smem, stream>>>(p);                                  \
            break;
        ROBOY_GENERIC_JOINT_COUNTS(ROBOY_PPO_CASE)
#undef ROBOY_PPO_CASE
        default: return cudaErrorInvalidValue;
    }
    err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    const uint32_t blocks = (p.P + 255) / 256;
    ppo_grad_reduce_kernel<<<blocks, 256, 0, stream>>>(p, slots);
    return cudaGetLastError();
}

}  // namespace roboy
