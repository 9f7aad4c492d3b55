/*
 * dnsac.h -- C ABI of the SAC actor of libdronenav.so (B200, sm_100a): SB3's sac.policies.Actor (latent ReLU MLP, then
 * mu and log_std heads, tanh-squashed diagonal Gaussian) with on-device sampling, for collection and deployment of a
 * trained SAC policy without torch.  The latent layers run on the tcgen05 contraction of the PPO update (dnppo.h) with a
 * ReLU epilogue; the heads and the sampler are one CUDA-core kernel.
 *
 * Conventions are those of dronenav.h / dnppo.h: 0 / negative DN_E* codes, dn_last_error(), caller-owned DEVICE buffers,
 * everything enqueued on the caller's stream, CUDA-graph capturable, no host synchronisation, no CPU fallback.
 */
#ifndef DNSAC_H_
#define DNSAC_H_

#include <stdint.h>

#include "dnppo.h"   /* DN_MLP_BF16X3, DN_MLP_BF16 */

#ifdef __cplusplus
extern "C" {
#endif

#define DN_SAC_MAX_LAYERS 4

typedef struct dn_sac_actor dn_sac_actor;

/* The parameters live in ONE flat FP32 vector owned by the caller (torch Parameters are views into it): latent layer l is
 * [hidden[l], in_l] row-major at w_off[l] (in_0 = obs_dim), its bias at b_off[l]; then mu [act_dim, hidden[n_hidden-1]] and
 * its bias, then log_std (a Linear layer, as in SB3) and its bias.  Accepted shapes: 1..4 hidden layers, widths multiples of
 * 128 between 128 and 512, 1 <= obs_dim <= 64, 1 <= act_dim <= 4, max_rows a positive multiple of 128; every tensor inside
 * [0, n_params).  dn_sac_actor_create checks all of this before it touches a device. */
typedef struct dn_sac_actor_config {
    int32_t abi_version;           /* = DN_ABI_VERSION */
    int32_t obs_dim, act_dim;
    int32_t max_rows;              /* largest row count of a dn_sac_act call */
    int32_t n_hidden;              /* latent layers (1..DN_SAC_MAX_LAYERS) */
    int32_t hidden[DN_SAC_MAX_LAYERS];
    int32_t precision;             /* DN_MLP_BF16X3 | DN_MLP_BF16 */
    int64_t w_off[DN_SAC_MAX_LAYERS], b_off[DN_SAC_MAX_LAYERS];
    int64_t mu_w_off, mu_b_off, log_std_w_off, log_std_b_off;
    int64_t n_params;
} dn_sac_actor_config;

int dn_sac_actor_create(const dn_sac_actor_config* cfg, int device, const float* params, dn_sac_actor** out);
int dn_sac_actor_destroy(dn_sac_actor* h);
/* Refresh the BF16 planes of the latent weights from the flat FP32 vector (after an optimiser step or a checkpoint load).
 * The heads read the FP32 vector directly. */
int dn_sac_actor_sync_weights(dn_sac_actor* h, void* stream);

/* Actor.forward of SB3 (sac/policies.py), per row:
 *   h        = ReLU MLP(obs)                                   (tcgen05, FP32-faithful BF16x3 planes by default)
 *   mu       = W_mu h + b_mu,   log_std = clamp(W_ls h + b_ls, -20, 2)
 *   DN_SAC_SAMPLE:        g = fmaf(exp(log_std), eps, mu),  action = tanh(g)
 *                         log_prob = sum_a (-0.5 eps_a^2 - log_std_a - 0.5 log(2 pi)) - sum_a log(1 - action_a^2 + 1e-6)
 *   DN_SAC_DETERMINISTIC: action = tanh(mu), log_prob = the same expression with eps = 0; nothing is drawn
 *   DN_SAC_UNIFORM:       action_a = 2 u01(word a) - 1 (SB3's action_space.sample() for Box(-1, 1) before learning_starts,
 *                         exact in FP32), log_prob = -act_dim log 2; the network is not evaluated
 * In FP32: expf, libm tanhf and logf.
 *
 * Draw layout (bit-exact, restated in numpy by tests/sac_act_reference.py).  Row r of a call with counter value c takes ONE
 * Philox4x32-10 block (dn_philox.cuh, the generator of the random spawn and of dn_ppo_act):
 *   key     = (seed lo, seed hi)
 *   counter = (c mod 2^32, DN_SAC_ACT_TAG, g lo, g hi),   g = row_id_offset + r   (global row id: shard-invariant)
 *   -> words (x, y, z, w).  The spawn draws use 0 and 1 in the second counter word and dn_ppo_act DN_PPO_ACT_TAG, so the
 *   three streams never meet.
 * DN_SAC_SAMPLE: Box-Muller on two pairs (x, y) and (z, w), 24-bit uniforms u01(v) = (v >> 8) 2^-24 in [0, 1),
 * u01_open(v) = ((v >> 8) + 1) 2^-24 in (0, 1]:
 *   r  = sqrt(-2 ln u01_open(x)),  eps[0] = r cos(2 pi u01(y)),  eps[1] = r sin(2 pi u01(y))
 *   r' = sqrt(-2 ln u01_open(z)),  eps[2] = r' cos(2 pi u01(w)), eps[3] = r' sin(2 pi u01(w))
 * act_dim a uses eps[0..a).  |eps| <= sqrt(48 ln 2) ~= 5.77.  In FP32: logf, sqrtf and sincospif.
 * DN_SAC_UNIFORM: action component a takes word a of (x, y, z, w).
 *
 * `counter` is a DEVICE int64: a DN_SAC_SAMPLE or DN_SAC_UNIFORM call reads *counter when its kernel runs and adds 1 after
 * it (stream-ordered), so a captured CUDA graph replays draw after draw without host involvement; a DN_SAC_DETERMINISTIC
 * call leaves it untouched.  `seed` is the same on every rank and `row_id_offset` is the shard's env_id_offset
 * (dn_config): the env with global id g then draws the same noise on any split. */
#define DN_SAC_ACT_TAG 0x53414341u   /* "SACA": second counter word of the SAC actor's draws */
#define DN_SAC_SAMPLE        0
#define DN_SAC_DETERMINISTIC 1
#define DN_SAC_UNIFORM       2
typedef struct dn_sac_sample {
    uint64_t seed;                 /* Philox key */
    int64_t  row_id_offset;        /* global id of row 0 (>= 0) */
    int64_t* counter;              /* device; drawing calls draw at *counter, then *counter += 1.  May be NULL when deterministic */
    int32_t  mode;                 /* DN_SAC_SAMPLE | DN_SAC_DETERMINISTIC | DN_SAC_UNIFORM */
    int32_t  reserved0;
} dn_sac_sample;
/* obs [rows, obs_dim]; action [rows, act_dim]; log_prob [rows] (nullable); 1 <= rows <= max_rows.  Capturable, no host
 * synchronisation; the arguments are checked before the handle is read. */
int dn_sac_act(dn_sac_actor* h, const float* obs, int32_t rows, const dn_sac_sample* s, float* action, float* log_prob, void* stream);
/* Test hook: device pointer / element count of an internal buffer: "x", "h1".."h4", "w1".."w4" (BF16 planes, lo plane at
 * + elems / 2), "mu", "log_std" (FP32 [max_rows, act_dim], written by the last non-uniform dn_sac_act). */
int dn_sac_actor_buffer(dn_sac_actor* h, const char* name, void** ptr, int64_t* elems);

#ifdef __cplusplus
}
#endif
#endif
