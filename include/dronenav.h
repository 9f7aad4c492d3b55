/*
 * dronenav.h -- C ABI of libdronenav.so, the B200 (sm_100a) batched drone-navigation
 * environment.
 *
 * The reference (eRGiBi/DRL-DroneNavigation) is pure Python and has no FFI of its own;
 * its boundary for this path is the Python object protocol of
 *   - PBDroneEnv.reset / PBDroneEnv.step   (Sol/Model/Environments/PBDroneEnv.py:609-665, 171-199)
 *   - BaseAviary.step                      (Sol/PyBullet/BaseAviary.py:324-453)
 *   - SB3 SubprocVecEnv + Monitor + NormalizeObservation built by
 *     PBDroneSimulator.make_env            (Sol/Model/PBDroneSimulator.py:136-204, 653-681)
 * Each entry point below names the reference interface it replaces.  The Python side
 * (drl-dronenavigation_b200/vec_env.py, env.py) binds these with ctypes; the binding a
 * reference maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - return 0 on success, a negative DN_E* code on failure; dn_last_error() returns a
 *     thread-local message for the last failure on the calling thread;
 *   - every I/O buffer is CALLER-OWNED DEVICE memory (plain pointers, no torch types)
 *     and must stay alive until the work enqueued on `stream` has completed;
 *   - all work is enqueued on the caller's stream (pass the raw cudaStream_t as void*;
 *     NULL = legacy default stream); no hidden synchronisation, no host allocation on
 *     the step path, CUDA-graph capturable;
 *   - one handle per device shard; a handle is not thread-safe; handles are independent;
 *   - there is NO CPU fallback: without a CUDA device dn_create fails with DN_ECUDA.
 *
 * Launch behaviour
 *   - dn_step / dn_step_many launch small grids (at most half the SMs) with programmatic stream serialization
 *     (PDL): the grid may be scheduled
 *     while the previous kernel of the stream is still running, but it executes griddepcontrol.wait before
 *     its first global memory access, so stream-order semantics of all buffers are unchanged.
 */
#ifndef DRONENAV_H_
#define DRONENAV_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DN_ABI_VERSION 4

/* error codes */
#define DN_OK        0
#define DN_EINVAL   -1   /* bad argument / config */
#define DN_ECUDA    -2   /* CUDA runtime error (message has the cudaError string) */
#define DN_ENOMEM   -3

/* ActionType (Sol/PyBullet/enums.py:36-43).  THRUST is what PBDroneEnv runs; the others are the
 * BaseSingleAgentAviary._preprocessAction branches (BaseSingleAgentAviary.py:153-225) that PBDroneEnv overrides. */
#define DN_ACT_THRUST     0   /* PBDroneEnv._preprocessAction, PBDroneEnv.py:872-895 */
#define DN_ACT_RPM        1   /* BaseSingleAgentAviary.py:176-179 */
#define DN_ACT_ONE_D_RPM  2   /* BaseSingleAgentAviary.py:211-212 (uses action[:,0]) */
#define DN_ACT_PID        3   /* :180-194: action[:,0:3] = destination; _calculateNextStep (BaseAviary.py:1255-1297)
                                 + DSLPIDControl.computeControl (Sol/PyBullet/DSLPIDControl.py:82-261) fused into the step */
#define DN_ACT_VEL        4   /* :195-210: action = (direction xyz, speed fraction); PID velocity tracking, current yaw held */
#define DN_ACT_ONE_D_PID  5   /* :213-223: target = current position + 0.1 * (0, 0, action[:,0]) */

/* DroneModel (Sol/PyBullet/enums.py:3-8): airframe constants of Sol/resources/{safegym/cf2x,cf2p,racer}.urdf and the
 * torque-mix branch of BaseAviary._dynamics (BaseAviary.py:927-935).  The reference itself can only construct CF2X
 * (BaseAviary.py:99 opens Sol/resources/safegym/<model>.urdf and the other two URDFs lack the pwm attributes its
 * parser reads, :1157-1160), so THRUST actions need CF2X; CF2P / RACE take the RPM types, CF2P also the PID types
 * (with the CF2X mixer, as BaseSingleAgentAviary.py:72-73 constructs it). */
#define DN_MODEL_CF2X     0
#define DN_MODEL_CF2P     1
#define DN_MODEL_RACE     2

/* physics flags.  0 == Physics.DYN (BaseAviary.py:899-973).  The add-ons restate the
 * PYB_* formulas inside the DYN integrator (documented extension, SURVEY.md a7). */
#define DN_PHYS_DYN            0
#define DN_PHYS_DRAG           1   /* BaseAviary._drag, BaseAviary.py:838-865 */
#define DN_PHYS_GROUND_EFFECT  2   /* BaseAviary._groundEffect, BaseAviary.py:798-834 */
#define DN_PHYS_GROUND_CONTACT 4   /* analytic substitute for p.getContactPoints(), PBDroneEnv.py:699 */

/* reward functions (reward_id) */
#define DN_REWARD_DEFAULT   0   /* PBDroneEnv._computeReward, PBDroneEnv.py:475-571 */
#define DN_REWARD_DUMMY     1   /* dummy_env.py:446-550 */
#define DN_REWARD_THRUSTENV 2   /* ThrustEnv.py:368-513 */
#define DN_REWARD_HER       3   /* HerPBDroneEnv.py:314-398 (first element of its tuple) */
#define DN_REWARD_REACHING  4   /* dummy_env.py:617-643 == Rewarder.py:8-40 reaching-progress (arXiv 2310.10943) */
#define DN_REWARD_PROGRESS  5   /* PBDroneEnv reward with the projection progress of Rewarder.py:43-62 (arXiv 2103.08624) x 2000
                                   in place of the distance difference (the reference only calls it from commented-out
                                   code, ThrustEnv.py:416-421; p_t / p_t-1 = position after / before the step) */
#define DN_REWARD_HOVER     6   /* upstream HoverAviary.py:65-76 */
#define DN_REWARD_FLYTHRUGATE 7 /* FlyThruGateAviary.py:100-112 */
#define DN_REWARD_BOOTSTRAPPED 8 /* Rewarder.BootstrappedImiVisionRewardCalculator (Rewarder.py:66-104, arXiv 2403.12203) */
#define DN_REWARD_CHAMP     9   /* Rewarder.ChampRewardCalculator (Rewarder.py:107-150, Nature 2023).  Both are formula classes the
                                   reference never calls ("yet unused"); here they are fed from PBDroneEnv's waypoint machine:
                                   (prev_dis, dis) = the stale distance pair of the default reward, delta_cam = angle between the
                                   forward vector and the direction to the current target, a_t / a_t-1 = this step's action /
                                   _last_action, omega_t = rpy_rates, passed = target captured this step, crashed = collision */
#define DN_NUM_REWARDS      10

/* spawn modes for (auto-)reset.  0 is the reference behaviour (PBDroneEnv.py:609-665). */
#define DN_SPAWN_FIXED      0   /* INIT_XYZS / INIT_RPYS, deterministic */
#define DN_SPAWN_LINE       1   /* Philox: within 0.1 m of a random target-pair line (PBDroneEnv.py:622-629,
                                   position_generator.py:121-152); commented out in the reference, offered as an option */
#define DN_SPAWN_MIDPOINT   2   /* Philox: midpoint of a random track segment, target order rolled to start behind it
                                   (PBDroneEnv.py:641-648, commented out in the reference, offered as an option) */

/* done byte written by dn_step */
#define DN_DONE_TERMINATED  1
#define DN_DONE_TRUNCATED   2

typedef struct dn_env dn_env;

/* Constructor arguments: PBDroneEnv.__init__ kwargs (PBDroneEnv.py:41-65) restricted to the
 * ones that reach the hot path, plus the shard description.  Geometry is double so the
 * host-side derived tables are computed in the reference's precision before being
 * rounded to FP32 for the kernel. */
typedef struct dn_config {
    int32_t  abi_version;        /* = DN_ABI_VERSION */
    int32_t  num_envs;           /* N, environments owned by this handle */
    int64_t  env_id_offset;      /* global id of local env 0 (Philox subsequence = global env id) */
    uint64_t seed;
    int32_t  pyb_freq;           /* PBDroneEnv.py:49 */
    int32_t  ctrl_freq;          /* PBDroneEnv.py:50 ; substeps S = pyb_freq / ctrl_freq */
    int32_t  act_type;           /* DN_ACT_* */
    int32_t  normalize_actions;  /* PBDroneEnv.py:63,173-176 (rescale_action) */
    int32_t  physics;            /* DN_PHYS_* flags */
    int32_t  reward_id;          /* DN_REWARD_* */
    int32_t  include_distance;   /* PBDroneEnv.py:62 -> obs dim 13 (else 12) */
    int32_t  cylinder;           /* PBDroneEnv.py:59 */
    int32_t  circle;             /* PBDroneEnv.py:60 */
    int32_t  max_steps;          /* PBDroneEnv.py:43,79 */
    int32_t  spawn_mode;         /* DN_SPAWN_* */
    int32_t  normalize_obs;      /* fuse normalize.NormalizeObservation (normalize.py:50-97), per env */
    double   threshold;          /* PBDroneEnv.py:43,77 */
    double   discount;           /* PBDroneEnv.py:43,78 */
    double   aviary_dim[6];      /* x_low,y_low,z_low,x_high,y_high,z_high (PBDroneEnv.py:83) */
    double   init_xyz[3];        /* INIT_XYZS[0] (BaseAviary.py:248-257) */
    double   init_rpy[3];        /* INIT_RPYS[0] (BaseAviary.py:258-263) */
    int32_t  num_targets;        /* T */
    int32_t  normalize_reward;   /* fuse normalize.NormalizeReward (normalize.py:100-147; args.norm_rew, PBDroneSimulator.py:193) */
    double   clip_reward;        /* > 0: clip the reward to +-this before normalisation (args.clip_rew, PBDroneSimulator.py:191-192: 10) */
    double   reward_gamma;       /* NormalizeReward gamma; 0 = its default 0.99 */
    const double* targets;       /* HOST pointer, [T,3] row-major (copied by dn_create) */
    int32_t  drone_model;        /* DN_MODEL_* (BaseAviary.__init__ drone_model, BaseAviary.py:30,76) */
    int32_t  reserved0;          /* = 0 */
} dn_config;

/* Buffers of one dn_step call.  Device pointers, caller-owned.  Nullable where noted. */
typedef struct dn_step_io {
    const float* actions;        /* [N,4] f32 (ONE_D_RPM / ONE_D_PID read column 0, PID columns 0..2) */
    float*       obs;            /* [N,obs_dim] f32 : obs of the step, or the reset obs if done */
    float*       reward;         /* [N] f32                                                     */
    uint8_t*     done;           /* [N] u8 : DN_DONE_TERMINATED | DN_DONE_TRUNCATED             */
    float*       terminal_obs;   /* [N,obs_dim] f32, rows written only where done; nullable     */
    int32_t*     found_targets;  /* [N] i32 info["found_targets"] (PBDroneEnv.py:434-442); nullable */
    float*       episode_return; /* [N] f32 Monitor info["episode"]["r"], written where done; nullable */
    int32_t*     episode_length; /* [N] i32 Monitor info["episode"]["l"], written where done; nullable */
} dn_step_io;

/* Row-major per-field view used to upload / download the full per-env state (parity tests
 * upload the oracle's state; checkpointing downloads it).  Device pointers, any may be NULL. */
typedef struct dn_state_view {
    float*    pos;            /* [N,3]  BaseAviary.pos                                   */
    float*    quat;           /* [N,4]  BaseAviary.quat, (x,y,z,w)                        */
    float*    vel;            /* [N,3]  BaseAviary.vel                                   */
    float*    rpy_rates;      /* [N,3]  BaseAviary.rpy_rates (body rates, BaseAviary.py:958) */
    float*    ang_v;          /* [N,3]  BaseAviary.ang_v (world, BaseAviary.py:952-956)   */
    float*    prev_vel;       /* [N,3]  PBDroneEnv.prev_vel                              */
    float*    prev_ang_v;     /* [N,3]  PBDroneEnv.prev_ang_v                            */
    float*    dist;           /* [N]    PBDroneEnv._distance_to_target                   */
    float*    prev_dist;      /* [N]    PBDroneEnv._prev_distance_to_target              */
    int32_t*  target_idx;     /* [N]    PBDroneEnv._current_target_index                 */
    int32_t*  steps;          /* [N]    PBDroneEnv._steps                                */
    uint8_t*  just_found;     /* [N]    PBDroneEnv.just_found                            */
    float*    ep_return;      /* [N]    Monitor running return                           */
    int32_t*  ep_length;      /* [N]    Monitor running length                           */
    uint32_t* episode_count;  /* [N]    episodes finished so far (Philox counter)        */
    float*    last_rpm_sum;   /* [N]    sum(last_clipped_action) (drag only, BaseAviary.py:429,442) */
    double*   obs_rms;        /* [N,2*obs_dim+1] FP64 mean | var | count, the dtype of the reference's RunningMeanStd
                                 (normalize.py:10-47); only if normalize_obs */
    float*    aux;            /* [N,4] _current_position.xyz | last travel with DN_REWARD_REACHING (with a random spawn mode
                                 _last_position.xyz | last travel); PBDroneEnv._last_action with
                                 DN_REWARD_BOOTSTRAPPED / DN_REWARD_CHAMP; absent otherwise */
    float*    rew_rms;        /* [N,4] returns | mean | var | count (normalize.py:100-147); only if normalize_reward */
    float*    spawn;          /* [N,4] INIT_XYZS[0] of the current episode | target roll; only with a random spawn mode */
    float*    pid;            /* [N,9] DSLPIDControl.integral_pos_e | integral_rpy_e | last_rpy (DSLPIDControl.py:66-80);
                                 only with the PID action types.  Like the reference's controller object it survives
                                 episode resets (BaseSingleAgentAviary never calls ctrl.reset()) */
} dn_state_view;

/* Aggregated Monitor statistics since the last clear (SB3 Monitor / ep_info_buffer). */
typedef struct dn_stats {
    double   return_sum;      /* sum of finished-episode returns   */
    uint64_t length_sum;      /* sum of finished-episode lengths   */
    uint64_t episodes;        /* finished episodes                 */
    uint64_t successes;       /* episodes that ended with _is_done (all targets reached) */
    uint64_t found_targets;   /* sum of found_targets at episode end */
    uint64_t crashes;         /* episodes ended by the -10 branch  */
    uint64_t truncations;     /* episodes ended by max_steps only  */
} dn_stats;

int         dn_abi_version(void);
const char* dn_last_error(void);

/* PBDroneEnv.__init__ + BaseAviary.__init__ for N environments on `device`
 * (PBDroneEnv.py:41-169, BaseAviary.py:27-272).  Allocates the persistent SoA state. */
int dn_create(const dn_config* cfg, int device, dn_env** out);
int dn_destroy(dn_env* env);

int dn_num_envs(const dn_env* env);
int dn_obs_dim(const dn_env* env);
/* kernels launched by this handle since creation (bench.py's gpu_launches) */
int64_t dn_launch_count(const dn_env* env);

/* PBDroneEnv.reset (PBDroneEnv.py:609-665 over BaseAviary.py:276-320) for every env, or
 * for the envs with mask[i] != 0.  Writes the reset observation rows (unmasked rows are
 * left untouched).  mask and obs_out may be NULL. */
int dn_reset(dn_env* env, const uint8_t* mask, float* obs_out, void* stream);

/* One control step of every env = PBDroneEnv.step (PBDroneEnv.py:171-199) including the
 * SubprocVecEnv worker's auto-reset and Monitor bookkeeping.  ONE kernel launch. */
int dn_step(dn_env* env, const dn_step_io* io, void* stream);

/* `num_steps` consecutive control steps in ONE launch with state held in registers:
 * step t reads actions[t] ([num_steps,N,4]).  Per-step outputs are [num_steps,...]-shaped
 * when `per_step_outputs` != 0, otherwise only the last step's outputs are written
 * ([N,...]).  Used for open-loop rollouts / the step-only throughput benchmark. */
int dn_step_many(dn_env* env, const dn_step_io* io, int num_steps, int per_step_outputs, void* stream);

/* dn_step with HOST buffers (caller-owned; same shapes as dn_step_io).  Returns when the results are in
 * the host buffers.  Pinned, device-mapped buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory)
 * are read and written by the fused kernel directly over PCIe (zero copy: one launch, whose last CTA
 * announces completion through a pinned word the call polls); pageable buffers are staged (H2D actions ->
 * kernel -> D2H outputs).  This is the call an out-of-process / numpy caller such as SB3's VecEnv.step_wait
 * makes; staging buffers and the stream belong to the handle. */
int dn_step_host(dn_env* env, const dn_step_io* host_io);

/* The host-buffer call on handle-owned buffers, moved by DMA: the HANDLE owns one pinned host slab laid out
 *   actions | obs | reward | found_targets | done | [episode_return | episode_length | terminal_obs]
 * and a device slab of the same layout.  dn_host_buffers fills `out` with HOST pointers into that slab (write actions
 * there, read results there: no copy on either side); `with_episode_info` = 0 leaves the three bracketed outputs NULL.
 * A dn_step_host / dn_step_host_async call that is given exactly these pointers replays ONE captured CUDA graph:
 * one H2D DMA of the actions, the fused kernel, one D2H DMA of the contiguous outputs (whose last word is the completion
 * flag the host waits on) -- instead of a kernel that reads and writes host memory over PCIe word by word plus a poll of the
 * stream.  dn_step_host_async returns as soon as the graph is launched, dn_step_host_wait when the results are in the slab
 * (SB3 VecEnv.step_async / step_wait).  Any other pointer set takes the paths described above; dn_step_host_async accepts only
 * the zero-copy one.  Until dn_step_host_wait has returned, every other call on the handle fails with DN_EINVAL. */
int dn_host_buffers(dn_env* env, int with_episode_info, dn_step_io* out);
int dn_step_host_async(dn_env* env, const dn_step_io* host_io);
int dn_step_host_wait(dn_env* env);

/* Resident step server for the zero-copy form of dn_step_host (pinned, device-mapped caller buffers).  A host step through a
 * kernel launch costs ~13 us on a B200 before a byte has moved (launch, scheduling, completion hand-off).  With idle_us > 0 the
 * step kernel (the dn_step_many variant) stays RESIDENT on the GPU instead: dn_step_host writes the step's actions pointer and a
 * sequence number to a doorbell word in pinned memory and polls the completion word; no launch per step.  The kernel leaves by
 * itself after `idle_us` microseconds without a command (so a device-wide synchronise elsewhere in the process waits at most
 * that long) and the next dn_step_host launches it again; every other call on the handle stops it first.  All CTAs of the
 * resident grid must fit on the device at once: DN_EINVAL above 4 CTAs (256 environments) per SM.  idle_us = 0 switches the
 * server off (the default).  What SB3's SubprocVecEnv workers are to the reference -- processes that stay alive between
 * steps and wait on a pipe (Sol/Model/PBDroneSimulator.py:171-200) -- this is to the GPU path.
 * dn_host_server_stats: how many residencies (kernel launches) and steps the server has run. */
int dn_host_server(dn_env* env, int idle_us);
int dn_host_server_stats(dn_env* env, int64_t* residencies, int64_t* steps);

/* The action map alone, elementwise over `n` action components (device pointers):
 * PBDroneEnv._preprocessAction(rescale_action(a)) (PBDroneEnv.py:872-895,949-971) or the RPM map
 * (BaseSingleAgentAviary.py:176-179), whichever the handle was created with.  Bit-identical to
 * the reference's float32 numpy arithmetic; used by the parity tests and by callers that log RPMs.
 * DN_EINVAL for the PID action types (their RPMs depend on the drone and controller state). */
int dn_action_to_rpm(dn_env* env, const float* actions, float* rpm_out, int64_t n, void* stream);

int dn_get_state(dn_env* env, const dn_state_view* view, void* stream);
int dn_set_state(dn_env* env, const dn_state_view* view, void* stream);

/* Copies the aggregated statistics to host (synchronises `stream`); clears them if `clear`. */
int dn_episode_stats(dn_env* env, dn_stats* host_out, int clear, void* stream);

/* Generalised advantage estimation over a device-resident rollout, the recursion of SB3's
 * RolloutBuffer.compute_returns_and_advantage that Sol/Model/Algorithms/sb3_ppo.py:190-316 consumes
 * (advantages, returns).  Layout [T, N] row-major; `done[t, n] != 0` means the episode of env n ended
 * with step t (so values[t+1, n] belongs to a new episode); `last_values[n]` is V(obs after step T-1).
 * One thread per env walks its T steps backwards (coalesced across envs).  Runs on the current device. */
int dn_gae(const float* rewards, const float* values, const uint8_t* done, const float* last_values,
           float gamma, float gae_lambda, float* advantages_out, float* returns_out,
           int32_t num_steps, int32_t num_envs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DRONENAV_H_ */
