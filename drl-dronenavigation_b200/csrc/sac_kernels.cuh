// sac_kernels.cuh -- the CUDA-core kernels of dn_sac_act (include/dnsac.h) after the actor's latent layers, which run on the
// tcgen05 contraction with the ReLU epilogue (dn_umma.cuh, K_FWD_RELU): the mu / log_std heads and the squashed-Gaussian
// sampler of SB3's sac.policies.Actor, and the uniform draws SB3 takes before learning_starts.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dn_philox.cuh"
#include "ppo_kernels.cuh"
#include "../../include/dnsac.h"

namespace dnsac {

using dnppo::HEAD_WARPS;

struct SacHeadArgs {
    int rows, n;                                        // rows of this call, width of the last hidden layer
    int mode;                                           // DN_SAC_SAMPLE | DN_SAC_DETERMINISTIC
    const __nv_bfloat16* h_hi; const __nv_bfloat16* h_lo;   // last hidden activation [rows, n] (lo may be null)
    const float* w_mu; const float* b_mu;               // [act_dim, n], [act_dim]
    const float* w_ls; const float* b_ls;
    float* mu; float* log_std;                          // [rows, act_dim]: the heads (log_std clamped), kept for inspection
    float* action; float* log_prob;                     // [rows, act_dim], [rows] (log_prob nullable)
    const long long* counter;                           // DN_SAC_SAMPLE: the device draw counter
    unsigned long long seed; long long row_id_offset;
};

__device__ __forceinline__ dn::U4 sac_words(uint32_t draw, unsigned long long seed, long long row_id_offset, int row) {
    const unsigned long long gid = static_cast<unsigned long long>(row_id_offset + row);
    return dn::philox4x32_10(dn::U4{draw, DN_SAC_ACT_TAG, static_cast<uint32_t>(gid), static_cast<uint32_t>(gid >> 32)},
                             static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
}

// One warp per row; lane l owns columns {2l + 64 i, 2l + 64 i + 1}.  NP = column pairs per lane (n / 64).  After the warp sums
// every lane holds mu and log_std; all lanes evaluate the row's draw and lane 0 stores it.
template <int ACT, int NP>
__global__ void __launch_bounds__(HEAD_WARPS * 32) sac_head_kernel(const SacHeadArgs g) {
    extern __shared__ float ssm[];                      // [2 ACT][n]: W_mu rows, then W_log_std rows
    for (int i = threadIdx.x; i < 2 * ACT * g.n; i += blockDim.x) ssm[i] = (i < ACT * g.n) ? g.w_mu[i] : g.w_ls[i - ACT * g.n];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ip = g.n / 64;
    float bmu[ACT], bls[ACT];
#pragma unroll
    for (int a = 0; a < ACT; ++a) { bmu[a] = g.b_mu[a]; bls[a] = g.b_ls[a]; }
    const bool sample = g.mode == DN_SAC_SAMPLE;
    const uint32_t draw = sample ? static_cast<uint32_t>(*g.counter) : 0u;
    for (int row = blockIdx.x * HEAD_WARPS + warp; row < g.rows; row += gridDim.x * HEAD_WARPS) {
        const long long o = static_cast<long long>(row) * g.n;
        float h[2 * NP];
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            const uint32_t wh = (i < ip) ? __ldg(reinterpret_cast<const uint32_t*>(g.h_hi + o) + lane + 32 * i) : 0u;
            const uint32_t wl = (i < ip && g.h_lo) ? __ldg(reinterpret_cast<const uint32_t*>(g.h_lo + o) + lane + 32 * i) : 0u;
            h[2 * i] = dnmma::bf16lo_f(wh) + dnmma::bf16lo_f(wl);
            h[2 * i + 1] = dnmma::bf16hi_f(wh) + dnmma::bf16hi_f(wl);
        }
        float mu[ACT], ls[ACT];
#pragma unroll
        for (int a = 0; a < ACT; ++a) {
            float am = 0.0f, al = 0.0f;
#pragma unroll
            for (int i = 0; i < NP; ++i)
                if (i < ip) {
                    const float2 wm = *reinterpret_cast<const float2*>(ssm + a * g.n + 2 * lane + 64 * i);
                    const float2 wls = *reinterpret_cast<const float2*>(ssm + (ACT + a) * g.n + 2 * lane + 64 * i);
                    am = fmaf(wm.x, h[2 * i], am); am = fmaf(wm.y, h[2 * i + 1], am);
                    al = fmaf(wls.x, h[2 * i], al); al = fmaf(wls.y, h[2 * i + 1], al);
                }
            mu[a] = dnppo::warp_sum(am) + bmu[a];
            ls[a] = fminf(fmaxf(dnppo::warp_sum(al) + bls[a], -20.0f), 2.0f);      // LOG_STD_MIN, LOG_STD_MAX
        }
        float z[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if (sample) {
            const dn::U4 r = sac_words(draw, g.seed, g.row_id_offset, row);
            dnppo::box_muller(r.x, r.y, z[0], z[1]);
            if (ACT > 2) dnppo::box_muller(r.z, r.w, z[2], z[3]);
        }
        // Normal(mu, std).log_prob(g) = -0.5 eps^2 - log_std - 0.5 log(2 pi); minus log(1 - tanh(g)^2 + 1e-6).  libm tanhf: the
        // MUFU tanh's 3e-7 absolute error is large against 1 - a^2 near saturation.
        float act[ACT], gauss = 0.0f, squash = 0.0f;
#pragma unroll
        for (int a = 0; a < ACT; ++a) {
            const float pre = sample ? fmaf(expf(ls[a]), z[a], mu[a]) : mu[a];
            act[a] = tanhf(pre);
            gauss += -0.5f * z[a] * z[a] - ls[a] - 0.918938533204672742f;
            squash += logf(1.0f - act[a] * act[a] + 1e-6f);
        }
        if (lane == 0) {
#pragma unroll
            for (int a = 0; a < ACT; ++a) {
                g.action[static_cast<long long>(row) * ACT + a] = act[a];
                g.mu[static_cast<long long>(row) * ACT + a] = mu[a];
                g.log_std[static_cast<long long>(row) * ACT + a] = ls[a];
            }
            if (g.log_prob) g.log_prob[row] = gauss - squash;
        }
    }
}

// SB3's action_space.sample() for Box(-1, 1): a = 2 u01(word a) - 1, exact in FP32; log_prob = log density of U[-1, 1)^A
__global__ void __launch_bounds__(256) sac_uniform_kernel(int rows, int act_dim, const long long* counter, unsigned long long seed,
                                                          long long row_id_offset, float* action, float* log_prob) {
    const int row = blockIdx.x * 256 + threadIdx.x;
    if (row >= rows) return;
    const dn::U4 r = sac_words(static_cast<uint32_t>(*counter), seed, row_id_offset, row);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    for (int a = 0; a < act_dim; ++a) action[static_cast<long long>(row) * act_dim + a] = 2.0f * dn::u01(w[a]) - 1.0f;
    if (log_prob) log_prob[row] = -0.693147180559945309f * static_cast<float>(act_dim);
}

}  // namespace dnsac
