// ppo_kernels.cuh -- the CUDA-core kernels of the PPO minibatch update around the tcgen05 contractions (dn_umma.cuh):
// minibatch gather + BF16 plane split, Gaussian / value heads with the PPO losses and their gradients
// (sb3_ppo.py:222-282 spelled out by hand), deterministic reduction of all partial
// gradients into the flat bucket, gradient-norm clipping + Adam (sb3_ppo.py:291-294), FP32 -> BF16 plane refresh.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dn_philox.cuh"
#include "dn_umma.cuh"
#include "../../include/dnppo.h"

namespace dnppo {

constexpr int MAX_LAYERS = 4;       // hidden layers per network
constexpr int MAX_ACT = 8;
constexpr int XPAD = 64;            // observation width padded to one 64-element k-block
constexpr int HEAD_WARPS = 4;       // 128-thread blocks: ~160 registers per thread still leave 3 blocks per SM
constexpr int MAX_HEAD_COLS = 512;  // widest last hidden layer the head kernel keeps in registers (16 values per lane)

struct Ctrl {                       // device-resident control block of one update() call
    int stopped;                    // sticky: the KL early stop fired (sb3_ppo.py:283-287); later minibatches are no-ops
    int n_done;                     // minibatches whose statistics were accumulated (includes the one that fired the stop)
    int n_applied;                  // optimiser steps taken
    int pad;
    double stats[4];                // sums over minibatches of: policy-gradient loss, value loss, approx_kl, clip fraction
    float last_kl;
    float last_norm;
};

// ---------------------------------------------------------------------------------------------------------------
// gather: idx -> minibatch rows.  Observation rows become the padded BF16 planes the first layer reads through TMA;
// the per-sample scalars are copied; the advantage moments (mean / unbiased std, sb3_ppo.py:233-234) are reduced
// deterministically: one (sum, sum of squares) pair per block in double, summed in block order by the head kernel.
// ---------------------------------------------------------------------------------------------------------------
struct GatherArgs {
    const float* obs; const float* act; const float* logp; const float* val; const float* adv; const float* ret;
    const long long* idx;           // nullptr: identity
    int rows, obs_dim, act_dim;
    __nv_bfloat16* x_hi; __nv_bfloat16* x_lo;     // [rows_pad, XPAD]
    float* m_act; float* m_logp; float* m_val; float* m_adv; float* m_ret;
    double* adv_partial;            // [gridDim.x][2]
};

__global__ void __launch_bounds__(256) gather_kernel(const GatherArgs g) {
    const int t = blockIdx.x * 256 + threadIdx.x;
    const int row = t >> 3, chunk = t & 7;
    double s = 0.0, s2 = 0.0;
    if (row < g.rows) {
        const long long src = g.idx ? g.idx[row] : row;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = chunk * 8 + j;
            v[j] = (c < g.obs_dim) ? __ldg(g.obs + src * g.obs_dim + c) : 0.0f;
        }
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) dnmma::split_pair(v[2 * j], v[2 * j + 1], h[j], l[j]);
        reinterpret_cast<uint4*>(g.x_hi + static_cast<long long>(row) * XPAD)[chunk] = make_uint4(h[0], h[1], h[2], h[3]);
        if (g.x_lo) reinterpret_cast<uint4*>(g.x_lo + static_cast<long long>(row) * XPAD)[chunk] = make_uint4(l[0], l[1], l[2], l[3]);
        if (chunk == 0 && g.m_act) {
            for (int a = 0; a < g.act_dim; ++a) g.m_act[static_cast<long long>(row) * g.act_dim + a] = __ldg(g.act + src * g.act_dim + a);
            g.m_logp[row] = __ldg(g.logp + src);
            g.m_val[row] = __ldg(g.val + src);
            g.m_ret[row] = __ldg(g.ret + src);
            const float a = __ldg(g.adv + src);
            g.m_adv[row] = a;
            s = a; s2 = static_cast<double>(a) * a;
        }
    }
    if (g.adv_partial) {
        __shared__ double sh[2][8];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
        if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = s2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0.0, b = 0.0;
            for (int w = 0; w < 8; ++w) { a += sh[0][w]; b += sh[1][w]; }
            g.adv_partial[2 * blockIdx.x] = a;
            g.adv_partial[2 * blockIdx.x + 1] = b;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// heads + losses + their gradients.  One warp per sample; lane l owns columns {2l + 64 i, 2l + 64 i + 1}.
// ---------------------------------------------------------------------------------------------------------------
struct HeadArgs {
    int rows, act_dim, n_pi, n_vf;                     // widths of the last hidden layers
    int train;                                          // 0: inference only (mean / value out)
    const __nv_bfloat16* hp_hi; const __nv_bfloat16* hp_lo;   // last hidden activation of pi [rows, n_pi] (lo may be null)
    const __nv_bfloat16* hv_hi; const __nv_bfloat16* hv_lo;   // ... of vf
    const float* w_pi; const float* b_pi;               // [act_dim, n_pi], [act_dim]
    const float* w_vf; const float* b_vf;               // [1, n_vf], [1]
    const float* log_std;                               // [act_dim]
    // inference outputs
    float* out_mean; float* out_value;
    // training inputs
    const float* m_act; const float* m_logp; const float* m_val; const float* m_adv; const float* m_ret;
    const double* adv_partial; int adv_blocks;
    int normalize_adv;
    float clip_range, clip_range_vf, vf_coef;           // clip_range_vf < 0: no value clipping
    // training outputs
    __nv_bfloat16* dzp_hi; __nv_bfloat16* dzp_lo;       // gradient w.r.t. the pre-activation of pi's last hidden layer
    __nv_bfloat16* dzv_hi; __nv_bfloat16* dzv_lo;
    float* partial;                                     // [gridDim.x][head_partial_size]
    int partial_size;
    // sampling (dn_ppo_act, inference only): the SAMPLE instantiations write action / clipped action / log-prob
    float* out_action; float* out_clipped; float* out_logp;
    const long long* counter;                           // null: deterministic (action = mean, nothing drawn)
    unsigned long long seed; long long row_id_offset;
    float low, high;
};
// layout of one block's partial: dW_pi [act_dim * n_pi] | db_pi [act_dim] | dW_vf [n_vf] | db_vf [1] | dlog_std [act_dim]
//                                | dbh_pi [n_pi] | dbh_vf [n_vf]  (bias gradients of the LAST HIDDEN layers = column sums of dz)
//                                | stats [4] (pg loss, value loss, approx_kl, clip fraction; sums over the block's samples)
__host__ __device__ inline int head_partial_size(int act_dim, int n_pi, int n_vf) {
    return act_dim * n_pi + act_dim + n_vf + 1 + act_dim + n_pi + n_vf + 4;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Box-Muller on two Philox words: z0 = r cos(2 pi u2), z1 = r sin(2 pi u2), r = sqrt(-2 ln u1), u1 in (0, 1], u2 in [0, 1)
__device__ __forceinline__ void box_muller(uint32_t w1, uint32_t w2, float& z0, float& z1) {
    const float r = sqrtf(-2.0f * logf(dn::u01_open(w1)));
    float s, c;
    sincospif(2.0f * dn::u01(w2), &s, &c);
    z0 = r * c;
    z1 = r * s;
}

// the draw counter of a stochastic dn_ppo_act call advances after the head kernel has read it
__global__ void counter_advance_kernel(long long* counter) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *counter += 1;
}

// NP = column pairs per lane = (widest of the two last hidden layers) / 64: sizes the per-lane register arrays.
// SAMPLE: the dn_ppo_act instantiations (inference only, no training code: the Philox rounds cost the row loop no registers)
template <int ACT, int NP, bool SAMPLE>
__global__ void __launch_bounds__(HEAD_WARPS * 32) head_kernel(const HeadArgs g) {
    extern __shared__ float hsm[];
    float* s_wpi = hsm;                                   // [ACT][n_pi]
    float* s_wvf = s_wpi + ACT * g.n_pi;                  // [n_vf]
    float* s_red = s_wvf + g.n_vf;                        // [HEAD_WARPS][partial_size] (training)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < ACT * g.n_pi; i += blockDim.x) s_wpi[i] = g.w_pi[i];
    for (int i = threadIdx.x; i < g.n_vf; i += blockDim.x) s_wvf[i] = g.w_vf[i];
    __syncthreads();

    const int ip = g.n_pi / 64, iv = g.n_vf / 64;         // column pairs per lane
    float adv_mean = 0.0f, adv_rstd = 1.0f;
    if (!SAMPLE && g.train && g.normalize_adv) {
        // advantage moments: the gather blocks' (sum, sum of squares) pairs, added in a fixed order by the whole block
        __shared__ double s_adv[2][HEAD_WARPS * 32];
        double a = 0.0, b = 0.0;
        for (int i = threadIdx.x; i < g.adv_blocks; i += HEAD_WARPS * 32) { a += g.adv_partial[2 * i]; b += g.adv_partial[2 * i + 1]; }
        s_adv[0][threadIdx.x] = a; s_adv[1][threadIdx.x] = b;
        __syncthreads();
        for (int o = HEAD_WARPS * 16; o > 0; o >>= 1) {
            if (threadIdx.x < o) { s_adv[0][threadIdx.x] += s_adv[0][threadIdx.x + o]; s_adv[1][threadIdx.x] += s_adv[1][threadIdx.x + o]; }
            __syncthreads();
        }
        const double n = g.rows, mean = s_adv[0][0] / n;
        double var = (s_adv[1][0] - n * mean * mean) / (n - 1.0);   // torch.std: unbiased
        if (var < 0.0) var = 0.0;
        adv_mean = static_cast<float>(mean);
        adv_rstd = 1.0f / (static_cast<float>(sqrt(var)) + 1e-8f);
    }
    float sig2inv[ACT], lstd[ACT], bpi[ACT];
#pragma unroll
    for (int a = 0; a < ACT; ++a) { lstd[a] = g.log_std[a]; sig2inv[a] = expf(-2.0f * lstd[a]); bpi[a] = g.b_pi[a]; }
    const float bvf = g.b_vf[0];
    const float inv_rows = 1.0f / static_cast<float>(g.rows);

    // per-lane accumulators of the head weight gradients (training)
    float gw_pi[ACT][2 * NP], gw_vf[2 * NP], gbh_pi[2 * NP], gbh_vf[2 * NP];
    float gb_pi[ACT], gls[ACT], gb_vf = 0.0f, st_pg = 0.0f, st_v = 0.0f, st_kl = 0.0f, st_cf = 0.0f;
#pragma unroll
    for (int a = 0; a < ACT; ++a) {
        gb_pi[a] = 0.0f; gls[a] = 0.0f;
#pragma unroll
        for (int i = 0; i < 2 * NP; ++i) gw_pi[a][i] = 0.0f;
    }
#pragma unroll
    for (int i = 0; i < 2 * NP; ++i) { gw_vf[i] = 0.0f; gbh_pi[i] = 0.0f; gbh_vf[i] = 0.0f; }

    // raw BF16 words of a row (hi / lo planes of both networks); the NEXT row's are requested before the current row is
    // worked on, so a warp always has one row of loads in flight (the kernel is latency-bound otherwise: few warps, DRAM-cold rows)
    uint32_t rp_h[NP], rp_l[NP], rv_h[NP], rv_l[NP];
    auto fetch = [&](int row) {
        const long long op = static_cast<long long>(row) * g.n_pi, ov = static_cast<long long>(row) * g.n_vf;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            rp_h[i] = (i < ip) ? __ldg(reinterpret_cast<const uint32_t*>(g.hp_hi + op) + lane + 32 * i) : 0u;
            rp_l[i] = (i < ip && g.hp_lo) ? __ldg(reinterpret_cast<const uint32_t*>(g.hp_lo + op) + lane + 32 * i) : 0u;
            rv_h[i] = (i < iv) ? __ldg(reinterpret_cast<const uint32_t*>(g.hv_hi + ov) + lane + 32 * i) : 0u;
            rv_l[i] = (i < iv && g.hv_lo) ? __ldg(reinterpret_cast<const uint32_t*>(g.hv_lo + ov) + lane + 32 * i) : 0u;
        }
    };
    const int row_first = blockIdx.x * HEAD_WARPS + warp, row_step = gridDim.x * HEAD_WARPS;
    if (row_first < g.rows) fetch(row_first);
    for (int row = row_first; row < g.rows; row += row_step) {
        // ---- the two activation rows (hi + lo) ----
        float hp[2 * NP], hv[2 * NP];
        const long long op = static_cast<long long>(row) * g.n_pi, ov = static_cast<long long>(row) * g.n_vf;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            hp[2 * i] = dnmma::bf16lo_f(rp_h[i]) + dnmma::bf16lo_f(rp_l[i]);
            hp[2 * i + 1] = dnmma::bf16hi_f(rp_h[i]) + dnmma::bf16hi_f(rp_l[i]);
            hv[2 * i] = dnmma::bf16lo_f(rv_h[i]) + dnmma::bf16lo_f(rv_l[i]);
            hv[2 * i + 1] = dnmma::bf16hi_f(rv_h[i]) + dnmma::bf16hi_f(rv_l[i]);
        }
        if (row + row_step < g.rows) fetch(row + row_step);
        // ---- heads: mean[a] = W_pi[a] . hp + b, value = W_vf . hv + b ----
        float mean[ACT], value;
#pragma unroll
        for (int a = 0; a < ACT; ++a) {
            float acc = 0.0f;
#pragma unroll
            for (int i = 0; i < NP; ++i)
                if (i < ip) {
                    const float2 w = *reinterpret_cast<const float2*>(s_wpi + a * g.n_pi + 2 * lane + 64 * i);
                    acc = fmaf(w.x, hp[2 * i], acc);
                    acc = fmaf(w.y, hp[2 * i + 1], acc);
                }
            mean[a] = warp_sum(acc) + bpi[a];
        }
        {
            float acc = 0.0f;
#pragma unroll
            for (int i = 0; i < NP; ++i)
                if (i < iv) {
                    const float2 w = *reinterpret_cast<const float2*>(s_wvf + 2 * lane + 64 * i);
                    acc = fmaf(w.x, hv[2 * i], acc);
                    acc = fmaf(w.y, hv[2 * i + 1], acc);
                }
            value = warp_sum(acc) + bvf;
        }
        if (SAMPLE || !g.train) {
            if (lane == 0) {
                // dn_ppo_act: the mean is staged in the action output and turned into the action after the loop
                float* out = SAMPLE ? g.out_action : g.out_mean;
#pragma unroll
                for (int a = 0; a < ACT; ++a) out[static_cast<long long>(row) * ACT + a] = mean[a];
                g.out_value[row] = value;
            }
            continue;
        }
        // ---- losses (sb3_ppo.py:225-282) and their gradients w.r.t. mean, log_std, value ----
        float logp = 0.0f, diff[ACT];
#pragma unroll
        for (int a = 0; a < ACT; ++a) {
            diff[a] = g.m_act[static_cast<long long>(row) * ACT + a] - mean[a];
            logp += -0.5f * diff[a] * diff[a] * sig2inv[a] - lstd[a] - 0.918938533204672742f;      // 0.5 log(2 pi)
        }
        const float old_logp = g.m_logp[row], old_v = g.m_val[row], ret = g.m_ret[row];
        const float adv = (g.m_adv[row] - adv_mean) * adv_rstd;
        const float log_ratio = logp - old_logp;
        const float ratio = expf(log_ratio);
        const float lo = 1.0f - g.clip_range, hi = 1.0f + g.clip_range;
        const float pg1 = adv * ratio, pg2 = adv * fminf(fmaxf(ratio, lo), hi);
        const bool inside = (ratio >= lo) && (ratio <= hi);
        const bool flows = inside || (pg1 < pg2);          // gradient of min(pg1, pg2) w.r.t. ratio is adv where pg1 is (co-)selected
        const float dlogp = flows ? -adv * ratio * inv_rows : 0.0f;
        float v_pred = value;
        bool v_flows = true;
        if (g.clip_range_vf >= 0.0f) {
            const float dv = value - old_v;
            v_pred = old_v + fminf(fmaxf(dv, -g.clip_range_vf), g.clip_range_vf);
            v_flows = (dv >= -g.clip_range_vf) && (dv <= g.clip_range_vf);
        }
        const float verr = v_pred - ret;
        const float dvalue = v_flows ? g.vf_coef * 2.0f * verr * inv_rows : 0.0f;
        float dmean[ACT];
#pragma unroll
        for (int a = 0; a < ACT; ++a) {
            dmean[a] = dlogp * diff[a] * sig2inv[a];
            if (lane == 0) {
                gb_pi[a] += dmean[a];
                gls[a] += dlogp * (diff[a] * diff[a] * sig2inv[a] - 1.0f);
            }
        }
        if (lane == 0) {
            gb_vf += dvalue;
            st_pg += -fminf(pg1, pg2);
            st_v += verr * verr;
            st_kl += (ratio - 1.0f) - log_ratio;
            st_cf += (fabsf(ratio - 1.0f) > g.clip_range) ? 1.0f : 0.0f;
        }
        // ---- gradient w.r.t. the last hidden pre-activations, head weight gradients ----
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            if (i < ip) {
                float d0 = 0.0f, d1 = 0.0f;
#pragma unroll
                for (int a = 0; a < ACT; ++a) {
                    const float2 w = *reinterpret_cast<const float2*>(s_wpi + a * g.n_pi + 2 * lane + 64 * i);
                    d0 = fmaf(dmean[a], w.x, d0);
                    d1 = fmaf(dmean[a], w.y, d1);
                    gw_pi[a][2 * i] = fmaf(dmean[a], hp[2 * i], gw_pi[a][2 * i]);
                    gw_pi[a][2 * i + 1] = fmaf(dmean[a], hp[2 * i + 1], gw_pi[a][2 * i + 1]);
                }
                d0 *= fmaf(-hp[2 * i], hp[2 * i], 1.0f);
                d1 *= fmaf(-hp[2 * i + 1], hp[2 * i + 1], 1.0f);
                gbh_pi[2 * i] += d0; gbh_pi[2 * i + 1] += d1;
                uint32_t wh, wl;
                dnmma::split_pair(d0, d1, wh, wl);
                reinterpret_cast<uint32_t*>(g.dzp_hi + op)[lane + 32 * i] = wh;
                if (g.dzp_lo) reinterpret_cast<uint32_t*>(g.dzp_lo + op)[lane + 32 * i] = wl;
            }
            if (i < iv) {
                const float2 w = *reinterpret_cast<const float2*>(s_wvf + 2 * lane + 64 * i);
                float d0 = dvalue * w.x, d1 = dvalue * w.y;
                gw_vf[2 * i] = fmaf(dvalue, hv[2 * i], gw_vf[2 * i]);
                gw_vf[2 * i + 1] = fmaf(dvalue, hv[2 * i + 1], gw_vf[2 * i + 1]);
                d0 *= fmaf(-hv[2 * i], hv[2 * i], 1.0f);
                d1 *= fmaf(-hv[2 * i + 1], hv[2 * i + 1], 1.0f);
                gbh_vf[2 * i] += d0; gbh_vf[2 * i + 1] += d1;
                uint32_t wh, wl;
                dnmma::split_pair(d0, d1, wh, wl);
                reinterpret_cast<uint32_t*>(g.dzv_hi + ov)[lane + 32 * i] = wh;
                if (g.dzv_lo) reinterpret_cast<uint32_t*>(g.dzv_lo + ov)[lane + 32 * i] = wl;
            }
        }
    }
    if (SAMPLE || !g.train) {
        if (!SAMPLE) return;
        // ---- sampling (dn_ppo_act, draw layout in include/dnppo.h): this warp's rows, one per lane (lane 0's mean stores are
        // visible to the warp after __syncwarp) ----
        __syncwarp();
        const uint32_t draw = g.counter ? static_cast<uint32_t>(*g.counter) : 0u;
        for (int row = row_first + lane * row_step; row < g.rows; row += 32 * row_step) {
            const long long o = static_cast<long long>(row) * ACT;
            float z[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            if (g.counter) {
                const unsigned long long gid = static_cast<unsigned long long>(g.row_id_offset + row);
                const dn::U4 r = dn::philox4x32_10(dn::U4{draw, DN_PPO_ACT_TAG, static_cast<uint32_t>(gid), static_cast<uint32_t>(gid >> 32)},
                                                   static_cast<uint32_t>(g.seed), static_cast<uint32_t>(g.seed >> 32));
                box_muller(r.x, r.y, z[0], z[1]);
                if (ACT > 2) box_muller(r.z, r.w, z[2], z[3]);
            }
            float logp = 0.0f;
#pragma unroll
            for (int a = 0; a < ACT; ++a) {
                const float mean = g.out_action[o + a];
                const float act = g.counter ? fmaf(expf(lstd[a]), z[a], mean) : mean;
                const float diff = act - mean;
                logp += -0.5f * diff * diff * sig2inv[a] - lstd[a] - 0.918938533204672742f;      // the training branch's expression
                g.out_action[o + a] = act;
                if (g.out_clipped) g.out_clipped[o + a] = fminf(fmaxf(act, g.low), g.high);
            }
            g.out_logp[row] = logp;
        }
        return;
    }
    // ---- block reduction in warp order (deterministic), one partial vector per block ----
    const int P = g.partial_size;
    float* mine = s_red + warp * P;
    const int o_bpi = ACT * g.n_pi, o_wvf = o_bpi + ACT, o_bvf = o_wvf + g.n_vf, o_ls = o_bvf + 1, o_bhp = o_ls + ACT, o_bhv = o_bhp + g.n_pi,
              o_st = o_bhv + g.n_vf;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        if (i < ip) {
#pragma unroll
            for (int a = 0; a < ACT; ++a) {
                mine[a * g.n_pi + 2 * lane + 64 * i] = gw_pi[a][2 * i];
                mine[a * g.n_pi + 2 * lane + 64 * i + 1] = gw_pi[a][2 * i + 1];
            }
            mine[o_bhp + 2 * lane + 64 * i] = gbh_pi[2 * i];
            mine[o_bhp + 2 * lane + 64 * i + 1] = gbh_pi[2 * i + 1];
        }
        if (i < iv) {
            mine[o_wvf + 2 * lane + 64 * i] = gw_vf[2 * i];
            mine[o_wvf + 2 * lane + 64 * i + 1] = gw_vf[2 * i + 1];
            mine[o_bhv + 2 * lane + 64 * i] = gbh_vf[2 * i];
            mine[o_bhv + 2 * lane + 64 * i + 1] = gbh_vf[2 * i + 1];
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < ACT; ++a) { mine[o_bpi + a] = gb_pi[a]; mine[o_ls + a] = gls[a]; }
        mine[o_bvf] = gb_vf;
        mine[o_st] = st_pg; mine[o_st + 1] = st_v; mine[o_st + 2] = st_kl; mine[o_st + 3] = st_cf;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        float acc = 0.0f;
#pragma unroll
        for (int w = 0; w < HEAD_WARPS; ++w) acc += s_red[w * P + i];
        g.partial[static_cast<long long>(blockIdx.x) * P + i] = acc;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// deterministic reduction of every partial gradient into the flat bucket (+ statistics and the KL flag)
// ---------------------------------------------------------------------------------------------------------------
struct Seg {                 // dst[dst_off + r * cols + c] = sum_s src[s * slice_stride + r * ld + c]
    const float* src;
    long long slice_stride, dst_off;
    int n_slices, rows, cols, ld;
    int first_block, n_blocks;
    int deep;                // 1: few elements, many slices (head / bias partials): 32 elements per block, the slices split over its warps
};
constexpr int REDUCE_PER_BLOCK = 1024;       // wide segments: 4 elements per thread, every thread walks all slices
constexpr int REDUCE_DEEP_PER_BLOCK = 32;    // deep segments: lane = element, warp w takes slices w, w + 8, ...
constexpr int REDUCE_DEEP_MIN_SLICES = 48;

struct ReduceArgs {
    const Seg* segs; int n_segs;
    const int* seg_of_block;
    float* grads; long long n_params;
    // statistics / KL flag (last block)
    const float* head_partial; int head_blocks, head_psize, head_stats_off;
    float ent_coef; int act_dim; long long log_std_off;
    float kl_limit;            // 1.5 * target_kl, < 0: no early stop
    int rows;
    Ctrl* ctrl;
};

// Every sum below is evaluated in an order fixed by the launch geometry alone: gradients are bit-reproducible run to run.
__global__ void __launch_bounds__(256) reduce_kernel(const ReduceArgs g) {
    if (blockIdx.x == gridDim.x - 1) {
        // statistics of this minibatch: the head blocks' sums, strided over the threads, then a fixed-order tree
        __shared__ double sh[4][256];
        double a[4] = {0, 0, 0, 0};
        for (int b = threadIdx.x; b < g.head_blocks; b += 256)
            for (int k = 0; k < 4; ++k) a[k] += g.head_partial[static_cast<long long>(b) * g.head_psize + g.head_stats_off + k];
        for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] = a[k];
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o)
                for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            const double inv = 1.0 / g.rows;
            const float kl = static_cast<float>(sh[2][0] * inv);
            const bool was_stopped = g.ctrl->stopped != 0;
            if (!was_stopped) {
                for (int k = 0; k < 4; ++k) g.ctrl->stats[k] += sh[k][0] * inv;
                g.ctrl->n_done += 1;
                g.ctrl->last_kl = kl;
            }
            // this rank's early-stop vote rides in the extra element of the bucket (summed by the all-reduce)
            g.grads[g.n_params] = (g.kl_limit >= 0.0f && kl > g.kl_limit) ? 1.0f : 0.0f;
        }
        return;
    }
    const Seg s = g.segs[g.seg_of_block[blockIdx.x]];
    const long long count = static_cast<long long>(s.rows) * s.cols;
    if (s.deep) {
        __shared__ float part[8][REDUCE_DEEP_PER_BLOCK];
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const long long i = static_cast<long long>(blockIdx.x - s.first_block) * REDUCE_DEEP_PER_BLOCK + lane;
        float acc = 0.0f;
        if (i < count) {
            const int r = static_cast<int>(i / s.cols), c = static_cast<int>(i % s.cols);
            const float* p = s.src + static_cast<long long>(r) * s.ld + c;
            int sl = warp;
            for (; sl + 56 < s.n_slices; sl += 64) {         // 8 loads in flight, added in slice order
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldg(p + (sl + 8 * u) * s.slice_stride);
#pragma unroll
                for (int u = 0; u < 8; ++u) acc += v[u];
            }
            for (; sl < s.n_slices; sl += 8) acc += __ldg(p + sl * s.slice_stride);
        }
        part[warp][lane] = acc;
        __syncthreads();
        if (warp == 0 && i < count) {
            float t = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; ++w) t += part[w][lane];
            if (s.dst_off == g.log_std_off) t -= g.ent_coef;      // entropy bonus, see below
            g.grads[s.dst_off + i] = t;
        }
        return;
    }
    const long long base = static_cast<long long>(blockIdx.x - s.first_block) * REDUCE_PER_BLOCK;
#pragma unroll
    for (int k = 0; k < REDUCE_PER_BLOCK / 256; ++k) {
        const long long i = base + k * 256 + threadIdx.x;
        if (i < count) {
            const int r = static_cast<int>(i / s.cols), c = static_cast<int>(i % s.cols);
            const float* p = s.src + static_cast<long long>(r) * s.ld + c;
            float acc = 0.0f;
            int sl = 0;
            for (; sl + 8 <= s.n_slices; sl += 8) {          // 8 loads in flight, added in slice order (deterministic)
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldg(p + (sl + u) * s.slice_stride);
#pragma unroll
                for (int u = 0; u < 8; ++u) acc += v[u];
            }
            for (; sl < s.n_slices; ++sl) acc += __ldg(p + sl * s.slice_stride);
            // entropy bonus: ent_loss = -sum_a(0.5 + 0.5 log 2 pi + log_std_a) -> d/dlog_std_a = -ent_coef
            if (s.dst_off == g.log_std_off) acc -= g.ent_coef;
            g.grads[s.dst_off + i] = acc;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// clip_grad_norm_ + Adam (torch.optim.Adam arithmetic), then the BF16 planes of the weights
// ---------------------------------------------------------------------------------------------------------------
constexpr int NORM_BLOCKS = 64;

__global__ void __launch_bounds__(256) norm_kernel(const float* __restrict__ grads, long long n, double* __restrict__ partial) {
    double acc = 0.0;
    for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<long long>(NORM_BLOCKS) * 256) {
        const double v = grads[i];
        acc += v * v;
    }
    __shared__ double sh[256];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}

struct AdamArgs {
    float* params; float* grads; float* exp_avg; float* exp_avg_sq; float* step;   // step: FP32 scalar (torch's capturable Adam keeps it so)
    long long n;
    const double* norm_partial;
    float lr, beta1, beta2, eps, max_grad_norm, inv_world;
    Ctrl* ctrl;
};

__global__ void __launch_bounds__(256) adam_kernel(const AdamArgs g) {
    __shared__ float s_scale;
    __shared__ int s_stop;
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < NORM_BLOCKS; ++i) t += g.norm_partial[i];
        const float norm = static_cast<float>(sqrt(t)) * g.inv_world;               // norm of the averaged gradient
        const float coef = fminf(g.max_grad_norm / (norm + 1e-6f), 1.0f);           // clip_grad_norm_
        s_scale = coef * g.inv_world;
        s_stop = (g.ctrl->stopped != 0) || (g.grads[g.n] > 0.5f);
    }
    __syncthreads();
    if (s_stop) return;
    const float scale = s_scale;
    const float t = *g.step + 1.0f;
    const float bc1 = 1.0f - powf(g.beta1, t), bc2 = 1.0f - powf(g.beta2, t);
    const float step_size = g.lr / bc1, rsq_bc2 = rsqrtf(bc2);
    for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < g.n; i += static_cast<long long>(gridDim.x) * 256) {
        const float gr = g.grads[i] * scale;
        const float m = g.exp_avg[i] + (1.0f - g.beta1) * (gr - g.exp_avg[i]);      // lerp, as torch's _single_tensor_adam
        const float v = g.beta2 * g.exp_avg_sq[i] + (1.0f - g.beta2) * gr * gr;
        g.exp_avg[i] = m;
        g.exp_avg_sq[i] = v;
        const float denom = sqrtf(v) * rsq_bc2 + g.eps;
        g.params[i] -= step_size * (m / denom);
    }
}

// commits the decision of this optimiser step (runs after adam_kernel, before anything reads ctrl again)
__global__ void ctrl_commit_kernel(Ctrl* ctrl, const float* grads, long long n, float* step, const double* norm_partial, float inv_world,
                                   volatile int* host_mirror /* pinned, mapped: [0] stopped, [1] n_done, [2] n_applied */) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const bool stop = (ctrl->stopped != 0) || (grads[n] > 0.5f);
        if (!stop) {
            *step += 1.0f;
            ctrl->n_applied += 1;
            double t = 0.0;
            for (int i = 0; i < NORM_BLOCKS; ++i) t += norm_partial[i];
            ctrl->last_norm = static_cast<float>(sqrt(t)) * inv_world;
        }
        ctrl->stopped = stop ? 1 : 0;
        if (host_mirror) {
            host_mirror[0] = ctrl->stopped; host_mirror[1] = ctrl->n_done; host_mirror[2] = ctrl->n_applied;
            __threadfence_system();
        }
    }
}

// FP32 weights -> BF16 hi / lo planes [2][rows][ld] (columns >= cols are zero padding)
struct PlaneSeg {
    long long param_off; int rows, cols, ld;
    __nv_bfloat16* planes;
    int first_block, n_blocks;
};
__global__ void __launch_bounds__(256) planes_kernel(const PlaneSeg* __restrict__ segs, const int* __restrict__ seg_of_block,
                                                     const float* __restrict__ params, int write_lo) {
    const PlaneSeg s = segs[seg_of_block[blockIdx.x]];
    const long long count = static_cast<long long>(s.rows) * s.ld;
    const long long i = (static_cast<long long>(blockIdx.x - s.first_block) * 256 + threadIdx.x) * 2;     // two columns per thread
    if (i >= count) return;
    const int r = static_cast<int>(i / s.ld), c = static_cast<int>(i % s.ld);
    const float v0 = (c < s.cols) ? params[s.param_off + static_cast<long long>(r) * s.cols + c] : 0.0f;
    const float v1 = (c + 1 < s.cols) ? params[s.param_off + static_cast<long long>(r) * s.cols + c + 1] : 0.0f;
    uint32_t wh, wl;
    dnmma::split_pair(v0, v1, wh, wl);
    reinterpret_cast<uint32_t*>(s.planes)[i / 2] = wh;
    if (write_lo) reinterpret_cast<uint32_t*>(s.planes + count)[i / 2] = wl;
}

}  // namespace dnppo
