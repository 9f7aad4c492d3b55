/*
 * dnppo.h -- C ABI of the PPO minibatch update of libdronenav.so (B200, sm_100a).
 *
 * Replaces, for the policy the reference trains (Sol/Model/PBDroneSimulator.py:251-258: separate pi / vf MLPs
 * [512, 512, 256] with Tanh, SB3 ActorCriticPolicy, diagonal Gaussian head), the body of the minibatch loop of
 *   PPO.train                               Sol/Model/Algorithms/sb3_ppo.py:190-316
 * i.e. evaluate_actions (:222), advantage normalisation (:233-234), clipped surrogate (:237-243), clipped value
 * loss (:251-262), entropy bonus (:265-271), approx-KL (:279-282), backward (:291), clip_grad_norm_ (:293) and the Adam step
 * (:294), as hand-written kernels: TMA + tcgen05.mma (BF16 planes, FP32 accumulation in TMEM) for the three
 * contractions of every layer, CUDA-core kernels for the heads / losses / reductions / Adam.
 *
 * Conventions are those of dronenav.h: 0 / negative DN_E* codes, dn_last_error(), caller-owned DEVICE buffers,
 * everything enqueued on the caller's stream, CUDA-graph capturable, no host synchronisation, no CPU fallback.
 */
#ifndef DNPPO_H_
#define DNPPO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* arithmetic of the contractions */
#define DN_MLP_BF16X3  0   /* FP32-faithful: x = hi + lo BF16 planes, A B ~= Ah Bh + Ah Bl + Al Bh (default) */
#define DN_MLP_BF16    1   /* plain BF16 inputs, FP32 accumulation (labelled option) */

/* Numerics-test hook: one contraction of the update on caller-owned planes.  A "planes" buffer holds the hi plane
 * followed by the lo plane (BF16, row-major); with passes = 1 only the hi plane is read / written.
 *   kind 0 (forward)   out[M,N] planes = act(A[M,K] B[N,K]^T + bias[N])          act: 1 tanh, 0 identity
 *   kind 1 (dgrad)     out[M,N] planes = (A[M,K] B[K,N]) * (1 - H[M,N]^2)
 *   kind 2 (wgrad)     partial[slices][M][N] f32 = A[rows_s, M]^T B[rows_s, N]    rows = K, split into `slices`
 * M, N, K: multiples of 128 / 64 / 64 (kind 2: K a multiple of 64 * slices). */
int dn_mlp_gemm(int kind, int passes, int M, int N, int K, int slices, const void* a_planes, const void* b_planes,
                const float* bias, int act, const void* h_planes, void* out_planes, float* partial, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * The update handle
 * ---------------------------------------------------------------------------------------------------------- */
#define DN_PPO_MAX_LAYERS 4

typedef struct dn_ppo dn_ppo;

/* Hyper-parameters = PPO(...) kwargs of PBDroneSimulator.setup_agent (PBDroneSimulator.py:251-286) + SB3 defaults.
 * The parameters live in ONE flat FP32 vector owned by the caller (torch Parameters are views into it); weight l of a
 * network is [out_l, in_l] row-major at *_w_off[l], its bias at *_b_off[l]; index n_hidden is the output head
 * (action_net [act_dim, h_last] / value_net [1, h_last]). */
typedef struct dn_ppo_config {
    int32_t abi_version;           /* = DN_ABI_VERSION */
    int32_t obs_dim, act_dim;      /* 13 (12 without the distance entry) / 4 */
    int32_t max_rows;              /* rows of the workspaces: >= the largest minibatch and dn_ppo_forward batch */
    int32_t n_pi, n_vf;            /* hidden layers of the policy / value network (1..DN_PPO_MAX_LAYERS) */
    int32_t pi_hidden[DN_PPO_MAX_LAYERS], vf_hidden[DN_PPO_MAX_LAYERS];   /* widths: multiples of 128, 128..512 */
    int32_t precision;             /* DN_MLP_BF16X3 | DN_MLP_BF16 */
    int32_t normalize_advantage;   /* sb3_ppo.py:233-234 */
    int32_t world_size;            /* ranks whose gradients the caller sums into the bucket between grad and apply */
    int32_t reserved0;
    float clip_range;              /* :237-243 */
    float clip_range_vf;           /* :251-259; < 0 = None */
    float ent_coef, vf_coef;       /* :273 */
    float max_grad_norm;           /* :293 */
    float target_kl;               /* :283-287 (stop when approx_kl > 1.5 target_kl); < 0 = None */
    float learning_rate, beta1, beta2, adam_eps;
    int64_t pi_w_off[DN_PPO_MAX_LAYERS + 1], pi_b_off[DN_PPO_MAX_LAYERS + 1];
    int64_t vf_w_off[DN_PPO_MAX_LAYERS + 1], vf_b_off[DN_PPO_MAX_LAYERS + 1];
    int64_t log_std_off, n_params;
} dn_ppo_config;

/* The rollout the minibatch indices point into (RolloutBuffer.get, sb3_ppo.py:213): flat [rows, ...] FP32, device. */
typedef struct dn_ppo_rollout {
    const float* obs;              /* [rows, obs_dim] */
    const float* actions;          /* [rows, act_dim] */
    const float* old_log_prob;     /* [rows] */
    const float* old_values;       /* [rows] */
    const float* advantages;       /* [rows] */
    const float* returns;          /* [rows] */
} dn_ppo_rollout;

/* Logger values of PPO.train (sb3_ppo.py:296-316), means over the minibatches run since dn_ppo_begin_update. */
typedef struct dn_ppo_stats {
    double policy_gradient_loss, value_loss, approx_kl, clip_fraction;
    int32_t minibatches;           /* minibatches whose losses were evaluated (includes the one that fired the stop) */
    int32_t optimizer_steps;
    int32_t early_stop;
    float last_approx_kl, last_grad_norm;
} dn_ppo_stats;

/* `params`, `exp_avg`, `exp_avg_sq`: [n_params]; `grads`: [n_params + 1] (the extra element carries this rank's
 * early-stop vote through the caller's all-reduce); `step`: one FP32 scalar (torch's capturable Adam step). */
int dn_ppo_create(const dn_ppo_config* cfg, int device, float* params, float* grads, float* exp_avg, float* exp_avg_sq, float* step,
                  dn_ppo** out);
int dn_ppo_destroy(dn_ppo* h);
/* Refresh the BF16 planes from the FP32 parameters (after the caller changed them: checkpoint load, init). */
int dn_ppo_sync_weights(dn_ppo* h, void* stream);
/* Start of PPO.train: clears the early-stop state and the statistics. */
int dn_ppo_begin_update(dn_ppo* h, void* stream);
/* One minibatch, first half (sb3_ppo.py:213-291): gather rows idx[0..mb_rows) of the rollout, evaluate_actions, the
 * losses, backward.  Leaves the gradient of the loss in grads[0..n_params) and the early-stop vote in grads[n_params].
 * mb_rows: multiple of 128, <= max_rows.  idx: int64 device pointer. */
int dn_ppo_minibatch_grad(dn_ppo* h, const dn_ppo_rollout* r, const int64_t* idx, int32_t mb_rows, void* stream);
/* Second half (sb3_ppo.py:283-294): if any rank voted to stop, this and every later call until dn_ppo_begin_update is a
 * no-op; otherwise grads / world_size -> clip_grad_norm_ -> Adam -> refreshed BF16 planes. */
int dn_ppo_minibatch_apply(dn_ppo* h, void* stream);
/* Data-parallel update (one process per GPU, every rank with its own handle and its own shard of the rollout): the sum over
 * the ranks of the flat gradient bucket (n_params + 1 floats -- the last one carries the rank's KL early-stop vote), in place,
 * between dn_ppo_minibatch_grad and dn_ppo_minibatch_apply (which divides by cfg.world_size).  The exchange runs over NVLink
 * peer memory: dn_ppo_comm_create allocates this rank's exchange region and returns its CUDA IPC handle (64 bytes); the caller
 * gathers the handles of all ranks with whatever it has (torch.distributed, MPI, a file) and passes them, rank-major, to
 * dn_ppo_comm_connect.  dn_ppo_allreduce is then ONE kernel of three phases (publish, reduce-scatter + push, collect) that waits
 * for the peers through flags in the mapped regions: capturable in a CUDA graph, bit-identical results on every rank (every
 * element is summed once, in rank order, by its owner).  Every rank must call it the same number of times; a wait that is not answered
 * within about a minute traps (CUDA error on the host) instead of hanging the GPU.  Single node only (CUDA IPC); the Python layer falls
 * back to ncclAllReduce elsewhere.  What it replaces: nothing in the reference (its PPO is single-process, sb3_ppo.py:288-294). */
#define DN_PPO_COMM_HANDLE_BYTES 64
int dn_ppo_comm_create(dn_ppo* h, int32_t rank, int32_t world, unsigned char* handle_out);
int dn_ppo_comm_connect(dn_ppo* h, const unsigned char* handles);
int dn_ppo_allreduce(dn_ppo* h, void* stream);

/* Statistics so far; synchronises `stream`. */
int dn_ppo_get_stats(dn_ppo* h, dn_ppo_stats* out, void* stream);
/* Non-blocking look at the early-stop state as of the last completed dn_ppo_minibatch_apply (pinned mirror). */
int dn_ppo_poll(dn_ppo* h, int32_t* early_stop, int32_t* minibatches, int32_t* optimizer_steps);
/* ActorCriticPolicy.forward without sampling: mean [rows, act_dim] and value [rows] for obs [rows, obs_dim] with the
 * same kernels and arithmetic as the update (rollout collection, evaluation).  rows <= max_rows. */
int dn_ppo_forward(dn_ppo* h, const float* obs, int32_t rows, float* mean, float* value, void* stream);

/* ActorCriticPolicy.forward with sampling (rollout collection): dn_ppo_forward's kernels and arithmetic for mean and value,
 * then, per row, in the same kernel:
 *   action[a]          = fmaf(exp(log_std[a]), z[a], mean[a])         (deterministic: action = mean, nothing is drawn)
 *   log_prob           = sum_a -0.5 diff_a^2 exp(-2 log_std[a]) - log_std[a] - 0.5 log(2 pi),   diff = action - mean
 *                        (the expression of the gradient half, which therefore recomputes the same old_log_prob)
 *   clipped_action[a]  = min(max(action[a], low), high)                 (SB3 clips to the Box before env.step)
 *
 * Draw layout (bit-exact, restated in numpy by tests/ppo_act_reference.py).  Row r of a call with counter value c takes ONE
 * Philox4x32-10 block (dn_philox.cuh, the generator of the random spawn):
 *   key     = (seed lo, seed hi)
 *   counter = (c mod 2^32, DN_PPO_ACT_TAG, g lo, g hi),   g = row_id_offset + r   (global row id: shard-invariant)
 *   -> words (x, y, z, w).  The spawn draws use 0 and 1 in the second counter word, so the two streams never meet.
 * Box-Muller on two pairs (x, y) and (z, w), 24-bit uniforms u01(v) = (v >> 8) 2^-24 in [0, 1),
 * u01_open(v) = ((v >> 8) + 1) 2^-24 in (0, 1]:
 *   r  = sqrt(-2 ln u01_open(x)),  z[0] = r cos(2 pi u01(y)),  z[1] = r sin(2 pi u01(y))
 *   r' = sqrt(-2 ln u01_open(z)),  z[2] = r' cos(2 pi u01(w)), z[3] = r' sin(2 pi u01(w))
 * act_dim 1 uses z[0], act_dim 3 z[0..2], act_dim 4 z[0..3].  The smallest u01_open is 2^-24, so |z| <= sqrt(48 ln 2) ~= 5.77:
 * the tails beyond 5.77 sigma (probability ~8e-9 per component) are never drawn.  In FP32: logf, sqrtf and sincospif.
 *
 * `counter` is a DEVICE int64: a stochastic call reads *counter when its kernel runs and adds 1 after it (stream-ordered), so
 * a captured CUDA graph replays draw after draw without host involvement.  `seed` is the same on every rank and
 * `row_id_offset` is the shard's env_id_offset (dn_config): the env with global id g then draws the same noise on any split. */
#define DN_PPO_ACT_TAG 0x50504F41u   /* "PPOA": second counter word of the sampler's draws */
typedef struct dn_ppo_sample {
    uint64_t seed;                 /* Philox key */
    int64_t  row_id_offset;        /* global id of row 0 (>= 0) */
    int64_t* counter;              /* device; this call draws at *counter, then *counter += 1.  May be NULL when deterministic */
    int32_t  deterministic;        /* 1: action = mean, no draw, counter untouched; 0: sample */
    float    low, high;            /* Box bounds of clipped_action, low <= high */
} dn_ppo_sample;
/* obs [rows, obs_dim]; action, clipped_action (nullable) [rows, act_dim]; log_prob, value [rows]; rows <= max_rows.
 * Capturable, no host synchronisation; the arguments are checked before the handle is read. */
int dn_ppo_act(dn_ppo* h, const float* obs, int32_t rows, const dn_ppo_sample* s, float* action, float* clipped_action,
               float* log_prob, float* value, void* stream);
/* Test hook: device pointer / element count of an internal buffer: "x", "pi.h1".."pi.h4", "pi.dz1".., "pi.w1".. (BF16
 * planes, lo plane at + elems / 2), and the same with "vf.". */
int dn_ppo_buffer(dn_ppo* h, const char* name, void** ptr, int64_t* elems);

#ifdef __cplusplus
}
#endif
#endif
