// dronenav.cu -- fused control-step kernel for sm_100a + the C ABI of include/dronenav.h.
//
// One launch of step_kernel = PBDroneEnv.step for every environment of the shard:
//   rescale_action -> _preprocessAction -> S x (_dynamics + _integrateQ) -> Euler ->
//   _computeObs -> _computeReward (waypoint state machine) -> _computeTerminated ->
//   _computeTruncated -> _update_state_post_step -> Monitor bookkeeping ->
//   SubprocVecEnv auto-reset [-> NormalizeObservation]
// (Sol/Model/Environments/PBDroneEnv.py:171-223,296-398,434-607,609-665,678-786,872-971;
//  Sol/PyBullet/BaseAviary.py:324-453,899-973; Sol/Model/Environments/normalize.py:10-97).
//
// Data movement per env-step: 1 x LDG.128 action, 7 x LDG.128 + 7 x STG.128 state planes,
// reward / done / found_targets scalars, and the [BLOCK, obs_dim] observation tile which
// is staged in shared memory and written with ONE 1-D TMA bulk store
// (cp.async.bulk.global.shared::cta) per CTA.  No tensor cores: the step is a streaming
// map, HBM-bound at S = 1 and issue/HBM balanced at S = 8.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <new>
#include <cstdlib>
#include <algorithm>

#include "../../include/dronenav.h"
#include "dn_params.h"
#include "dn_device.cuh"
#include "dn_host.h"

namespace dn {

// 64 threads per CTA, 16 CTAs per SM: same occupancy as 128 x 8, but mid-size grids balance better over the 148 SMs
// (65 536 envs: 1024 CTAs = 6.9 per SM instead of 512 = 3.5; measured 7.93 -> 7.68 us, 4096 envs 4.20 -> 4.08 us)
#ifndef DN_BLOCK
#define DN_BLOCK 64
#endif
constexpr int kBlock = DN_BLOCK;
constexpr int kCtasPerSm = 1024 / kBlock;   // resident CTAs per SM at 64 registers per thread

// ---------------------------------------------------------------------------
// small PTX wrappers (TMA 1-D bulk store of the observation tile)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_g2s_commit(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t saddr = static_cast<uint32_t>(__cvta_generic_to_shared(ssrc));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(saddr), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// resident step server: polling loads (host doorbell / device command word), the step's actions straight from host memory (the
// same host addresses are read again in later steps of the SAME kernel: never through the non-coherent path), timer for the idle bound
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ float4 ld_volatile_f4(const float4* p) {
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// The next command of the resident step server, the same for every thread of every CTA.  0 in the pointer field = leave.
// Every wait is bounded: the leader leaves after `srv_idle_us` without a command (and publishes that), the others after the
// leader says so -- or, as a last resort, after a spin cap (a kernel that cannot hear its leader must not stay forever).
__device__ __forceinline__ unsigned long long srv_next_command(const StepIO& io, unsigned long long last, unsigned long long* s_cmd, int tid) {
    if (tid == 0) {
        unsigned long long w = last;
        if (blockIdx.x == 0) {
            const unsigned long long t0 = globaltimer_ns(), idle_ns = 1000ull * io.srv_idle_us;
            unsigned int spins = 0;
            for (;;) {
                w = ld_volatile_u64(io.srv_doorbell);
                if ((w >> 48) != (last >> 48)) break;
                ++spins;
                if (((spins & 15u) == 0u && globaltimer_ns() - t0 > idle_ns) || spins > (1u << 24)) { w = last & ~kSrvPtrMask; break; }
            }
            st_release_gpu_u64(io.srv_cmd, w);
        } else {
            unsigned int spins = 0;
            for (;;) {
                w = ld_acquire_gpu_u64(io.srv_cmd);
                if (w != last) break;
                if (++spins > (1u << 26)) { w = last & ~kSrvPtrMask; break; }
            }
        }
        *s_cmd = w;
    }
    __syncthreads();
    return *s_cmd;
}

// fire-and-forget L2 prefetch: raises the number of DRAM requests in flight without holding registers
__device__ __forceinline__ void prefetch_l2(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
}

// ---------------------------------------------------------------------------
// the fused step kernel
// ---------------------------------------------------------------------------
// Monitor statistics without contended atomics: every CTA owns one BlockStats slot, its warps add
// their finished episodes to it, and dn_episode_stats reduces the slots.  (A first version used one
// atomicAdd per warp per counter on 7 GLOBAL addresses; with ~12 % of the envs finishing per step
// that serialised in L2 and doubled the step time at 4 Mi envs.)
// eps|suc and cra|tru are packed 16:16.  A lane adds at most one episode per step, and the multi-step kernel flushes and
// clears its accumulator every kStatsFlushSteps steps, so every half stays below 2^15: the low halves never carry into the
// high ones and the arithmetic shift of a high half never sees a sign bit, whatever num_steps is.
struct BlockAcc { float ret; int len, fnd, eps_suc, cra_tru; };
constexpr int kStatsFlushSteps = 32767;

__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }

// ---- Monitor statistics: warp shuffle -> this CTA's slot.  Only the (up to 4) warps of one CTA ever
// touch a slot, so these reductions do not contend; integer sums are exact and the float returns are
// added as doubles (exact for any realistic count), so the totals do not depend on arrival order.
// (per-lane counts are < 2^15 between flushes, so a warp's packed 16:16 sums need the two halves summed apart)
__device__ __forceinline__ void flush_stats(const Params& P, const BlockAcc& acc, const int tid) {
    const int eps_w = warp_sum(acc.eps_suc & 0xffff);
    if (eps_w != 0) {                              // warp-uniform
        float ret = acc.ret;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) ret += __shfl_xor_sync(0xffffffffu, ret, d);
        const int len = warp_sum(acc.len), fnd = warp_sum(acc.fnd), suc = warp_sum(acc.eps_suc >> 16);
        const int cra = warp_sum(acc.cra_tru & 0xffff), tru = warp_sum(acc.cra_tru >> 16);
        if ((tid & 31) == 0) {
            BlockStats* b = &P.block_stats[blockIdx.x];
            atomicAdd(&b->return_sum, static_cast<double>(ret));
            atomicAdd(&b->length_sum, static_cast<unsigned long long>(len));
            atomicAdd(&b->episodes, static_cast<unsigned long long>(eps_w));
            atomicAdd(&b->found_targets, static_cast<unsigned long long>(fnd));
            if (suc) atomicAdd(&b->successes, static_cast<unsigned long long>(suc));
            if (cra) atomicAdd(&b->crashes, static_cast<unsigned long long>(cra));
            if (tru) atomicAdd(&b->truncations, static_cast<unsigned long long>(tru));
        }
    }
}

// MULTI = false: exactly one control step per launch (dn_step): no step loop, no per-thread
// statistics carried across steps, <= 64 registers (1024 resident threads / SM).  MULTI = true: dn_step_many.
template <int PHYS, bool NORM, bool MULTI, bool FULL>
__global__ void __launch_bounds__(kBlock, (MULTI || NORM) ? (kCtasPerSm * 3) / 4 : kCtasPerSm)
step_kernel(const __grid_constant__ Params P, const __grid_constant__ StepIO io, int num_steps_arg, int per_step_arg) {
    __shared__ __align__(128) float tile[kBlock * kMaxObs];
    // bookkeeping planes 4..6 of this CTA's environments, staged by cp.async at kernel entry and consumed after the
    // last substep: the copy is in flight during the whole physics loop without holding registers, and the epilogue
    // starts with a shared-memory read instead of an L2 / HBM round trip (single-step kernel only)
    __shared__ __align__(16) float4 aux_stage[MULTI ? 1 : 3 * kBlock];
    const int num_steps = MULTI ? num_steps_arg : 1;
    const int per_step = MULTI ? per_step_arg : 1;
    // programmatic dependent launch (see launch_step): let the next kernel of the stream be scheduled now, and do not
    // touch global memory before the previous kernel has completed.  Both are no-ops for a normal launch.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int tid = threadIdx.x;
    const int base = blockIdx.x * kBlock;
    const int i = base + tid;
    const bool active = i < P.n;
    if (io.pdl_prefetch && active) {
        // While the previous kernel of the stream is still running: start this thread's lines towards L2.  L2 is the
        // coherence point, so a line prefetched early is still the one the previous kernel's stores update; for a
        // handle whose state is cold (another handle ran in between) this overlaps the HBM fetch with that kernel.
        prefetch_l2(io.actions + i);
#pragma unroll
        for (int p = 0; p < kPlanes; ++p) prefetch_l2(&P.s[p][i]);
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int D = P.obs_dim;
    float* const obs_row = tile + tid * D;

    EnvState s;
    float last_rpm_sum = 0.0f;
    if (active) {
        load_core(P, i, s);
        if (PHYS & 1) last_rpm_sum = P.last_rpm_sum[i];
        // The bookkeeping planes are consumed ~1000 instructions from now.
        if (MULTI) {
            prefetch_l2(&P.s[4][i]); prefetch_l2(&P.s[5][i]); prefetch_l2(&P.s[6][i]);
        } else {
#pragma unroll
            for (int p = 0; p < 3; ++p) {
                const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(&aux_stage[p * kBlock + tid]));
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(&P.s[4 + p][i]) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        // Software pipelining across CTAs: the CTA that will run on this SM slot one "GPU-full of CTAs"
        // later finds its physics planes and actions already in L2 (the kernel is otherwise limited by
        // the DRAM latency exposed at the top of each thread, not by bandwidth or issue slots).
        const long long j = static_cast<long long>(i) + static_cast<long long>(P.prefetch_ctas) * kBlock;
        if (j < P.n) {
            prefetch_l2(&P.s[0][j]); prefetch_l2(&P.s[1][j]); prefetch_l2(&P.s[2][j]); prefetch_l2(&P.s[3][j]);
            prefetch_l2(io.actions + j);
        }
    }
    BlockAcc acc = {0.f, 0, 0, 0, 0};            // this thread's finished episodes over the launch
    __shared__ unsigned long long srv_cmd_s;
    const bool srv = MULTI && io.srv_doorbell != nullptr;      // resident step server: one host command per loop iteration
    unsigned long long srv_word = io.srv_word0;

    for (int t = 0; t < num_steps; ++t) {
        if (MULTI && srv) {
            srv_word = srv_next_command(io, srv_word, &srv_cmd_s, tid);
            if ((srv_word & kSrvPtrMask) == 0ull) break;             // quit / idle: every CTA leaves after the same step
        }
        const bool write_out = per_step || (t == num_steps - 1) || srv;
        const size_t o = (per_step ? static_cast<size_t>(t) * P.n : 0) + i;      // output element index of this env
        if (active) {
            const float4 act = (MULTI && srv) ? ld_volatile_f4(reinterpret_cast<const float4*>(srv_word & kSrvPtrMask) + i)
                                              : __ldg(io.actions + static_cast<size_t>(t) * P.n + i);
            const StepResult r = env_step<PHYS, FULL>(P, i, s, act, last_rpm_sum, obs_row,   // obs_row: obs of the step (terminal obs if finished)
                                                MULTI ? nullptr : &aux_stage[tid], kBlock);
            float* term_out = (write_out && r.finished && io.terminal_obs) ? io.terminal_obs + o * D : nullptr;
            if (!MULTI) {
                // single-step kernel: the state is final here; storing it now frees its registers for the
                // wrapper code below (the multi-step variant keeps the physics planes in registers across steps)
                store_state(P, i, s);
                if (PHYS & 1) P.last_rpm_sum[i] = last_rpm_sum;
            }
            if (NORM) {
                // NormalizeObservation sits inside Monitor and the worker's auto-reset
                // (PBDroneSimulator.py:181): the terminal observation updates the running
                // statistics in .step, the reset observation again in .reset (normalize.py:74-92).
                // All 2 x obs_dim statistics are fetched first (independent loads in flight together; a
                // load -> update -> store loop per entry serialised 13 L2 round trips: 9 us for a 12-env launch).
                // The statistics are FP64 (the reference's dtype); they are fetched four entries at a time so that the
                // independent loads are in flight together without holding all 2 x obs_dim doubles in registers.
                const size_t N = P.n;
                double* cnt_p = P.obs_rms + static_cast<size_t>(2 * D) * N + i;
                const double cnt = *cnt_p;
#pragma unroll
                for (int k0 = 0; k0 < kMaxObs; k0 += 4) {
                    double m[4], v[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int k = k0 + j;
                        if (k < D) {
                            m[j] = P.obs_rms[static_cast<size_t>(k) * N + i];
                            v[j] = P.obs_rms[static_cast<size_t>(D + k) * N + i];
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int k = k0 + j;
                        if (k < D) {
                            const float tn = rms_update_normalize(obs_row[k], m[j], v[j], cnt);
                            float ob = tn;
                            if (r.finished) {
                                if (term_out) term_out[k] = tn;
                                const float raw = (k < 3) ? r.spawn_obs[k] : ((k < 12) ? P.init_obs[k] : r.reset_obs_dist);
                                ob = rms_update_normalize(raw, m[j], v[j], cnt + 1.0);
                            }
                            obs_row[k] = ob;
                            P.obs_rms[static_cast<size_t>(k) * N + i] = m[j];
                            P.obs_rms[static_cast<size_t>(D + k) * N + i] = v[j];
                        }
                    }
                }
                *cnt_p = cnt + (r.finished ? 2.0 : 1.0);
            } else if (r.finished) {
                if (term_out) {
#pragma unroll
                    for (int k = 0; k < 12; ++k) term_out[k] = obs_row[k];
                    if (D == 13) term_out[12] = obs_row[12];
                }
#pragma unroll
                for (int k = 3; k < 12; ++k) obs_row[k] = P.init_obs[k];
                obs_row[0] = r.spawn_obs[0]; obs_row[1] = r.spawn_obs[1]; obs_row[2] = r.spawn_obs[2];
                if (D == 13) obs_row[12] = r.reset_obs_dist;
            }
            if (write_out) {
                io.reward[o] = r.reward;
                io.done[o] = r.done;
                if (io.found_targets) io.found_targets[o] = r.found;
                if (r.finished) {
                    if (io.episode_return) io.episode_return[o] = r.ep_ret;
                    if (io.episode_length) io.episode_length[o] = r.ep_len;
                }
            }
            if (r.finished) {
                acc.ret += r.ep_ret; acc.len += r.ep_len; acc.fnd += r.found;
                acc.eps_suc += 1 + (r.success ? 0x10000 : 0);
                acc.cra_tru += (r.crash ? 1 : 0) + ((r.done == DN_DONE_TRUNCATED) ? 0x10000 : 0);
            }
            // MULTI: stored every step -- the next step's epilogue re-reads the bookkeeping planes and, on a crash, the
            // entry position from memory; the physics planes stay in registers across steps
            if (MULTI) {
                store_state(P, i, s);
                if ((PHYS & 1) && t == num_steps - 1) P.last_rpm_sum[i] = last_rpm_sum;
            }
        }
        // ---- observation rows: shared memory -> one TMA bulk store PER WARP (32 rows are contiguous both in
        // shared and in global memory, 32 * obs_dim * 4 bytes is a multiple of 16): no CTA-wide barrier.
        if (write_out) {
            const int wbase = base + (tid & ~31);                        // first env of this warp
            const int n_here = min(32, P.n - wbase);                     // <= 0 for warps past the end
            if (n_here > 0) {
                float* gdst = io.obs + ((per_step ? static_cast<size_t>(t) * P.n : 0) + wbase) * D;
                const float* wsrc = tile + (tid & ~31) * D;
                const uint32_t bytes = static_cast<uint32_t>(n_here) * D * 4u;
                const bool bulk_ok = ((reinterpret_cast<uintptr_t>(gdst) & 15u) == 0) && ((bytes & 15u) == 0);
                if (bulk_ok) {
                    fence_proxy_async_smem();
                    __syncwarp();
                    if ((tid & 31) == 0) {
                        bulk_store_g2s_commit(gdst, wsrc, bytes);
                        if (MULTI && t + 1 < num_steps) bulk_store_wait_read();   // rows are rewritten by the next step
                    }
                    if (MULTI && t + 1 < num_steps) __syncwarp();
                } else {
                    __syncwarp();
                    for (int j = (tid & 31); j < n_here * D; j += 32) gdst[j] = wsrc[j];
                    if (MULTI && t + 1 < num_steps) __syncwarp();
                }
            }
        }
        if (MULTI && !srv && (t + 1) % kStatsFlushSteps == 0) {
            // t is the same for every thread, so the warp collectives of flush_stats stay convergent
            flush_stats(P, acc, tid);
            acc = BlockAcc{0.f, 0, 0, 0, 0};
        }
        if (MULTI && srv) {
            // the step is complete for the host when every CTA's stores (bulk stores of the observation rows included) are
            // visible system-wide: count this CTA done; the last one writes the step's sequence number to the pinned word
            flush_stats(P, acc, tid);
            acc = BlockAcc{0.f, 0, 0, 0, 0};
            if ((tid & 31) == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                __threadfence_system();          // one fence per CTA: cumulative over the stores the barrier ordered before it
                const unsigned int prev = atomicAdd(io.done_counter, 1u);
                if (prev == gridDim.x - 1) {
                    *io.done_counter = 0u;
                    __threadfence_system();
                    *reinterpret_cast<volatile unsigned int*>(io.host_flag) = static_cast<unsigned int>(srv_word >> 48);
                }
            }
        }
    }
    if (MULTI && srv) return;
    flush_stats(P, acc, tid);
    if (io.host_flag != nullptr) {
        // Host call on mapped host buffers: completion is announced through host memory.  Every thread's stores (the bulk
        // stores of the observation rows included) are made visible system-wide, the CTA counts itself done, and the last
        // CTA writes the step's sequence number to the pinned word the host is polling -- no stream query, no interrupt.
        if ((tid & 31) == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            __threadfence_system();              // one fence per CTA: cumulative over the stores the barrier ordered before it
            const unsigned int prev = atomicAdd(io.done_counter, 1u);
            if (prev == gridDim.x - 1) {
                *io.done_counter = 0u;
                __threadfence_system();
                *reinterpret_cast<volatile unsigned int*>(io.host_flag) = io.seq;
            }
        }
        return;
    }
    if ((tid & 31) == 0) bulk_store_wait_read();   // shared memory must outlive the bulk read
}

// reduces the per-CTA slots into one Stats record (dn_episode_stats); optionally clears the slots
__global__ void stats_reduce_kernel(BlockStats* slots, int n_slots, Stats* out, int clear) {
    __shared__ double s_ret[256];
    __shared__ unsigned long long s_cnt[6][256];
    double ret = 0.0;
    unsigned long long c[6] = {0, 0, 0, 0, 0, 0};
    for (int k = threadIdx.x; k < n_slots; k += blockDim.x) {
        const BlockStats b = slots[k];
        ret += b.return_sum;
        c[0] += b.length_sum; c[1] += b.episodes; c[2] += b.successes; c[3] += b.found_targets; c[4] += b.crashes; c[5] += b.truncations;
        if (clear) slots[k] = BlockStats{0.0, 0, 0, 0, 0, 0, 0};
    }
    s_ret[threadIdx.x] = ret;
    for (int q = 0; q < 6; ++q) s_cnt[q][threadIdx.x] = c[q];
    __syncthreads();
    for (int d = blockDim.x / 2; d > 0; d >>= 1) {
        if (threadIdx.x < d) {
            s_ret[threadIdx.x] += s_ret[threadIdx.x + d];
            for (int q = 0; q < 6; ++q) s_cnt[q][threadIdx.x] += s_cnt[q][threadIdx.x + d];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out->return_sum = s_ret[0]; out->length_sum = s_cnt[0][0]; out->episodes = s_cnt[1][0]; out->successes = s_cnt[2][0];
        out->found_targets = s_cnt[3][0]; out->crashes = s_cnt[4][0]; out->truncations = s_cnt[5][0];
    }
}

// ---------------------------------------------------------------------------
// construction-time state, explicit reset, state (un)packing
// ---------------------------------------------------------------------------
__global__ void init_kernel(const __grid_constant__ Params P, float d0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n) return;
    EnvState s;
    s.px = P.init_pos[0]; s.py = P.init_pos[1]; s.pz = P.init_pos[2]; s.dist = d0;
    s.qx = P.init_quat[0]; s.qy = P.init_quat[1]; s.qz = P.init_quat[2]; s.qw = P.init_quat[3];
    s.vx = s.vy = s.vz = 0.f; s.prev_dist = d0;
    s.wx = s.wy = s.wz = 0.f; s.ep_ret = 0.f;
    s.ax = s.ay = s.az = 0.f; s.bits = 0u;
    s.pvx = s.pvy = s.pvz = 0.f; s.ep_len = 0;
    s.pax = s.pay = s.paz = 0.f; s.ep_count = 0u;
    store_state(P, i, s);
    if (P.last_rpm_sum) P.last_rpm_sum[i] = 0.f;
    if (P.spawn) P.spawn[i] = make_float4(P.init_pos[0], P.init_pos[1], P.init_pos[2], 0.f);
    if (P.aux) P.aux[i] = (P.rw.mode == RW_LITERATURE) ? make_float4(0.f, 0.f, 0.f, 0.f)      // _last_action = 0 (PBDroneEnv.py:131)
                                                        : make_float4(P.init_pos[0], P.init_pos[1], P.init_pos[2], 0.f);   // _last_position = _current_position = INIT_XYZS[0]
    if (P.rew_rms) P.rew_rms[i] = make_float4(0.f, 0.f, 1.f, 1e-4f);                       // returns 0; RunningMeanStd(): mean 0, var 1, count 1e-4
    if (P.pid[0]) { P.pid[0][i] = P.pid[1][i] = P.pid[2][i] = make_float4(0.f, 0.f, 0.f, 0.f); }   // DSLPIDControl.reset (DSLPIDControl.py:66-80)
    if (P.obs_rms) {
        const size_t N = P.n; const int D = P.obs_dim;
        for (int k = 0; k < D; ++k) { P.obs_rms[k * N + i] = 0.0; P.obs_rms[(D + k) * N + i] = 1.0; }
        P.obs_rms[2 * D * N + i] = 1e-4;                    // RunningMeanStd(epsilon=1e-4), normalize.py:13-17
    }
}

// PBDroneEnv.reset called explicitly (VecEnv.reset / evaluate_policy), PBDroneEnv.py:609-665
template <bool NORM>
__global__ void reset_kernel(const __grid_constant__ Params P, const uint8_t* mask, float* obs_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n) return;
    if (mask && !mask[i]) return;
    EnvState s;
    load_state(P, i, s);
    const int steps = static_cast<int>(s.bits & kStepsMask);
    const float stale_dist = s.dist;
    float D0 = s.dist;
    if (steps != 0) {                           // _current_position == pos of the last post-step
        const float4 t0 = target_at(P, 0);
        const float dx = s.px - t0.x, dy = s.py - t0.y, dz = s.pz - t0.z;
        D0 = sqrtf(dx * dx + dy * dy + dz * dz);
    }
    s.px = P.init_pos[0]; s.py = P.init_pos[1]; s.pz = P.init_pos[2];
    if (P.spawn_mode != DN_SPAWN_FIXED) {       // see env_step; the Philox counter advances on explicit resets too
        s.ep_count += 1u;
        int roll = 0;
        if (P.spawn_mode == DN_SPAWN_LINE) spawn_line(P, i, s.ep_count, s.px, s.py, s.pz);
        else spawn_midpoint(P, i, s.ep_count, s.px, s.py, s.pz, roll);
        P.spawn[i] = make_float4(s.px, s.py, s.pz, static_cast<float>(roll));
        if (P.aux && P.rw.mode == RW_REACHING) reaching_travel_after_spawn(P, i, s.px, s.py, s.pz);
        const float4 t0 = target_at(P, roll);
        const float dx = s.px - t0.x, dy = s.py - t0.y, dz = s.pz - t0.z;
        D0 = sqrtf(dx * dx + dy * dy + dz * dz);
    }
    s.qx = P.init_quat[0]; s.qy = P.init_quat[1]; s.qz = P.init_quat[2]; s.qw = P.init_quat[3];
    s.vx = s.vy = s.vz = 0.f; s.wx = s.wy = s.wz = 0.f; s.ax = s.ay = s.az = 0.f;
    s.pvx = s.pvy = s.pvz = 0.f; s.pax = s.pay = s.paz = 0.f;
    s.dist = D0; s.prev_dist = D0; s.bits = 0u;
    s.ep_ret = 0.f; s.ep_len = 0;               // Monitor.reset
    store_state(P, i, s);
    if (P.last_rpm_sum) P.last_rpm_sum[i] = 0.f;
    const int D = P.obs_dim;
    float o[kMaxObs];
#pragma unroll
    for (int k = 0; k < 12; ++k) o[k] = P.init_obs[k];
    if (P.spawn_mode != DN_SPAWN_FIXED) { o[0] = s.px * P.inv_x_high; o[1] = s.py * P.inv_y_high; o[2] = s.pz * P.inv_z_high; }
    o[12] = stale_dist * P.inv_max_target_dist;
    if (NORM) {
        const size_t N = P.n;
        double* cnt_p = P.obs_rms + static_cast<size_t>(2 * D) * N + i;
        const double cnt = *cnt_p;
        for (int k = 0; k < D; ++k) {
            double* mp = P.obs_rms + static_cast<size_t>(k) * N + i;
            double* vp = P.obs_rms + static_cast<size_t>(D + k) * N + i;
            double m = *mp, v = *vp;
            o[k] = rms_update_normalize(o[k], m, v, cnt);
            *mp = m; *vp = v;
        }
        *cnt_p = cnt + 1.0;
    }
    if (obs_out) for (int k = 0; k < D; ++k) obs_out[static_cast<size_t>(i) * D + k] = o[k];
}

__global__ void action_map_kernel(const __grid_constant__ Params P, const float* __restrict__ a, float* __restrict__ out, long long n) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = action_to_rpm(P, a[i]);
}

__global__ void gae_kernel(const float* __restrict__ rew, const float* __restrict__ val, const uint8_t* __restrict__ done,
                           const float* __restrict__ last_val, float gamma, float lam, float* __restrict__ adv,
                           float* __restrict__ ret, int T, int N) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float next_v = last_val[n], gae = 0.0f;
    for (int t = T - 1; t >= 0; --t) {
        const size_t k = static_cast<size_t>(t) * N + n;
        const float nnt = done[k] ? 0.0f : 1.0f;
        const float v = val[k];
        const float delta = rew[k] + gamma * next_v * nnt - v;
        gae = delta + gamma * lam * nnt * gae;
        adv[k] = gae;
        ret[k] = gae + v;
        next_v = v;
    }
}

struct StateView {   // device mirror of dn_state_view
    float *pos, *quat, *vel, *rpy_rates, *ang_v, *prev_vel, *prev_ang_v, *dist, *prev_dist;
    int32_t *target_idx, *steps; uint8_t* just_found; float* ep_return; int32_t* ep_length;
    uint32_t* episode_count; float* last_rpm_sum; double* obs_rms; float* aux; float* rew_rms; float* spawn; float* pid;
};

template <bool SET>
__global__ void state_xfer_kernel(const __grid_constant__ Params P, const __grid_constant__ StateView V) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n) return;
    EnvState s;
    load_state(P, i, s);
    int idx = static_cast<int>(s.bits >> kIdxShift);
    int steps = static_cast<int>(s.bits & kStepsMask);
    int jf = (s.bits & kJustFoundBit) ? 1 : 0;
#define DN_V3(ptr, a, b, c) if (V.ptr) { if (SET) { a = V.ptr[3*i]; b = V.ptr[3*i+1]; c = V.ptr[3*i+2]; } else { V.ptr[3*i] = a; V.ptr[3*i+1] = b; V.ptr[3*i+2] = c; } }
#define DN_V1(ptr, a, T) if (V.ptr) { if (SET) { a = static_cast<decltype(a)>(V.ptr[i]); } else { V.ptr[i] = static_cast<T>(a); } }
    DN_V3(pos, s.px, s.py, s.pz)
    if (V.quat) {
        if (SET) { s.qx = V.quat[4*i]; s.qy = V.quat[4*i+1]; s.qz = V.quat[4*i+2]; s.qw = V.quat[4*i+3]; }
        else { V.quat[4*i] = s.qx; V.quat[4*i+1] = s.qy; V.quat[4*i+2] = s.qz; V.quat[4*i+3] = s.qw; }
    }
    DN_V3(vel, s.vx, s.vy, s.vz)
    DN_V3(rpy_rates, s.wx, s.wy, s.wz)
    DN_V3(ang_v, s.ax, s.ay, s.az)
    DN_V3(prev_vel, s.pvx, s.pvy, s.pvz)
    DN_V3(prev_ang_v, s.pax, s.pay, s.paz)
    DN_V1(dist, s.dist, float)
    DN_V1(prev_dist, s.prev_dist, float)
    DN_V1(target_idx, idx, int32_t)
    DN_V1(steps, steps, int32_t)
    DN_V1(just_found, jf, uint8_t)
    DN_V1(ep_return, s.ep_ret, float)
    DN_V1(ep_length, s.ep_len, int32_t)
    DN_V1(episode_count, s.ep_count, uint32_t)
#undef DN_V3
#undef DN_V1
    if (V.last_rpm_sum && P.last_rpm_sum) {
        if (SET) P.last_rpm_sum[i] = V.last_rpm_sum[i]; else V.last_rpm_sum[i] = P.last_rpm_sum[i];
    }
    if (V.aux && P.aux) {
        float4* g = reinterpret_cast<float4*>(V.aux);
        if (SET) P.aux[i] = g[i]; else g[i] = P.aux[i];
    }
    if (V.spawn && P.spawn) {
        float4* g = reinterpret_cast<float4*>(V.spawn);
        if (SET) P.spawn[i] = g[i]; else g[i] = P.spawn[i];
    }
    if (V.pid && P.pid[0]) {                                  // [N,9] integral_pos_e | integral_rpy_e | last_rpy
        float* g = V.pid + 9 * static_cast<size_t>(i);
        for (int k = 0; k < 3; ++k) {
            if (SET) P.pid[k][i] = make_float4(g[3 * k], g[3 * k + 1], g[3 * k + 2], 0.f);
            else { const float4 v = P.pid[k][i]; g[3 * k] = v.x; g[3 * k + 1] = v.y; g[3 * k + 2] = v.z; }
        }
    }
    if (V.rew_rms && P.rew_rms) {
        float4* g = reinterpret_cast<float4*>(V.rew_rms);
        if (SET) P.rew_rms[i] = g[i]; else g[i] = P.rew_rms[i];
    }
    if (V.obs_rms && P.obs_rms) {
        const int W = 2 * P.obs_dim + 1; const size_t N = P.n;
        for (int k = 0; k < W; ++k) {
            if (SET) P.obs_rms[k * N + i] = V.obs_rms[static_cast<size_t>(i) * W + k];
            else V.obs_rms[static_cast<size_t>(i) * W + k] = P.obs_rms[k * N + i];
        }
    }
    if (SET) {
        // resetBasePositionAndOrientation -> read-back returns a unit quaternion.  One that is already unit to FP32 precision
        // (every quaternion dn_get_state returns) is kept bit for bit, so that a get / set round trip clones the state exactly.
        const float q2 = s.qx * s.qx + s.qy * s.qy + s.qz * s.qz + s.qw * s.qw;
        if (V.quat && fabsf(q2 - 1.0f) > 4e-6f) {
            const float inv = rsqrtf(q2);
            s.qx *= inv; s.qy *= inv; s.qz *= inv; s.qw *= inv;
        }
        s.bits = (static_cast<uint32_t>(idx) << kIdxShift) | (jf ? kJustFoundBit : 0u) | (static_cast<uint32_t>(steps) & kStepsMask);
        store_state(P, i, s);
    }
}

}  // namespace dn

// ===========================================================================
// host side: the C ABI
// ===========================================================================
using dn::Params;

// Every step_kernel instantiation, [physics & 3][MULTI] for one (normalize_obs, full) pair; dn_create keeps the two a handle
// launches.
using StepKernel = void (*)(dn::Params, dn::StepIO, int, int);
template <bool NORM, bool FULL>
const StepKernel kStepKernels[4][2] = {
    {dn::step_kernel<0, NORM, false, FULL>, dn::step_kernel<0, NORM, true, FULL>},
    {dn::step_kernel<1, NORM, false, FULL>, dn::step_kernel<1, NORM, true, FULL>},
    {dn::step_kernel<2, NORM, false, FULL>, dn::step_kernel<2, NORM, true, FULL>},
    {dn::step_kernel<3, NORM, false, FULL>, dn::step_kernel<3, NORM, true, FULL>}};

// Byte offsets of the host-call buffers, each at 256-byte alignment:
//   actions | obs | reward | found_targets | done | [episode_return | episode_length | terminal_obs] | completion word
// Everything after the actions is one contiguous range [obs, word + 4): the slab moves its outputs with a single D2H copy.
struct IoLayout { size_t act, obs, rew, fnd, done, epr, epl, term, word, bytes; bool episode; };

static IoLayout io_layout(size_t N, size_t D, bool episode) {
    IoLayout L = {};
    L.episode = episode;
    auto take = [&L](size_t b) { const size_t at = L.bytes; L.bytes += (b + 255) & ~static_cast<size_t>(255); return at; };
    L.act = take(N * 16); L.obs = take(N * D * 4); L.rew = take(N * 4); L.fnd = take(N * 4); L.done = take(N);
    if (episode) { L.epr = take(N * 4); L.epl = take(N * 4); L.term = take(N * D * 4); }
    L.word = take(4);
    return L;
}

static dn_step_io io_at(const IoLayout& L, char* b) {
    dn_step_io io;
    io.actions = reinterpret_cast<const float*>(b + L.act); io.obs = reinterpret_cast<float*>(b + L.obs);
    io.reward = reinterpret_cast<float*>(b + L.rew); io.found_targets = reinterpret_cast<int32_t*>(b + L.fnd);
    io.done = reinterpret_cast<uint8_t*>(b + L.done);
    io.episode_return = L.episode ? reinterpret_cast<float*>(b + L.epr) : nullptr;
    io.episode_length = L.episode ? reinterpret_cast<int32_t*>(b + L.epl) : nullptr;
    io.terminal_obs = L.episode ? reinterpret_cast<float*>(b + L.term) : nullptr;
    return io;
}

enum class InFlight { None, Slab, ZeroCopy };   // which dn_step_host_async step dn_step_host_wait has to wait for

struct dn_env {
    Params P;
    int device;
    int normalize_obs;
    StepKernel step_one, step_many;   // this handle's step_kernel: one step per launch (MULTI = false) | dn_step_many
    void* state_mem;
    float4* d_targets;
    float4* d_segs;
    dn::Stats* d_stats;          // one reduced record (output of stats_reduce_kernel)
    dn::BlockStats* d_block_stats; // one slot per CTA of the step grid
    int n_slots;
    int64_t launches;
    int sms;                // multiprocessor count of the device
    float d0;
    // host-buffer calls (allocated on first use)
    cudaStream_t host_stream;
    void* stage;            // device staging of the pageable path: IoLayout with the episode outputs
    dn_step_io host_seen;   // last host io whose pointers were classified
    dn_step_io host_mapped; // device aliases of those pointers when all of them are pinned + mapped (UVA)
    int host_direct;        // 1: the kernel reads / writes the caller's pinned buffers directly (zero copy)
    const void* ptr_cache_h[32]; void* ptr_cache_d[32]; int ptr_cache_n; unsigned ptr_cache_next;   // pinned + mapped pointers seen so far
    InFlight in_flight;     // the dn_step_host_async step that has not been waited for
    // dn_host_buffers: handle-owned pinned slab + device slab, stepped by replaying one captured graph
    char* slab_h; char* slab_d;
    IoLayout slab;
    dn_step_io slab_io_h, slab_io_d;
    cudaGraphExec_t slab_exec;
    // zero-copy host call: completion word in pinned host memory, written by the last CTA of the step kernel
    unsigned int* zc_flag_h; unsigned int* zc_flag_d; unsigned int* zc_counter; unsigned int zc_seq;
    // resident step server (dn_host_server): a dn_step_many kernel that stays on the GPU and takes one host command per step
    int srv_idle_us;        // > 0: dn_step_host on pinned + mapped buffers goes through the server
    int srv_alive;          // a server kernel has been launched on srv_stream and has not been seen to finish
    cudaStream_t srv_stream;
    unsigned long long* srv_doorbell_h; unsigned long long* srv_doorbell_d;   // pinned + mapped
    unsigned long long* srv_word_h;     // pinned staging word for the initial value of srv_cmd
    unsigned long long* srv_cmd;        // device
    unsigned int srv_seq;   // sequence number of the last command (16 bits, never 0)
    dn_step_io srv_io;      // mapped output pointers the running server writes
    long long srv_residencies, srv_steps;
};

static thread_local std::string g_err;

static int fail(int code, const std::string& msg) { g_err = msg; return code; }

int dn_internal_fail(int code, const std::string& msg) { return fail(code, msg); }   // other translation units (ppo_update.cu)

#define DN_CUDA(expr)                                                                    \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            return fail(DN_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));   \
    } while (0)

namespace {
struct DeviceGuard {   // switches the calling thread to the handle's device only when it is on another one
    int prev = -1; bool ok = false, switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        if (prev == dev) { ok = true; return; }
        if (cudaSetDevice(dev) == cudaSuccess) { ok = true; switched = true; }
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
}  // namespace

extern "C" {

// Every call that touches the handle's state goes through here first.  It refuses while a dn_step_host_async step has not been
// waited for (that step still runs on the handle's stream against the same state), then stops the resident step server if one
// is running -- unless `stop_server` is false (dn_step_host on the server path).
static int quiesce(dn_env* env, const char* who, bool stop_server = true) {
    if (env->in_flight != InFlight::None)
        return fail(DN_EINVAL, std::string(who) + ": a dn_step_host_async step has not been waited for (dn_step_host_wait)");
    if (!stop_server || !env->srv_alive) return DN_OK;
    DeviceGuard guard(env->device);
    env->srv_seq = (env->srv_seq % 0xFFFFu) + 1u;
    *reinterpret_cast<volatile unsigned long long*>(env->srv_doorbell_h) = static_cast<unsigned long long>(env->srv_seq) << 48;   // pointer 0: quit
    env->srv_alive = 0;
    DN_CUDA(cudaStreamSynchronize(env->srv_stream));
    return DN_OK;
}

int dn_abi_version(void) { return DN_ABI_VERSION; }
const char* dn_last_error(void) { return g_err.c_str(); }

int dn_create(const dn_config* cfg, int device, dn_env** out) {
    if (!cfg || !out) return fail(DN_EINVAL, "dn_create: null argument");
    *out = nullptr;
    if (cfg->abi_version != DN_ABI_VERSION) return fail(DN_EINVAL, "dn_create: abi_version mismatch");
    if (cfg->num_envs <= 0) return fail(DN_EINVAL, "dn_create: num_envs must be > 0");
    if (cfg->pyb_freq <= 0 || cfg->ctrl_freq <= 0 || cfg->pyb_freq % cfg->ctrl_freq != 0)
        return fail(DN_EINVAL, "dn_create: pyb_freq is not divisible by ctrl_freq");   // BaseAviary.py:81-82
    if (cfg->num_targets <= 0 || cfg->num_targets >= 2047 || !cfg->targets)
        return fail(DN_EINVAL, "dn_create: need 1..2046 targets");
    if (cfg->act_type < 0 || cfg->act_type > DN_ACT_ONE_D_PID) return fail(DN_EINVAL, "dn_create: unsupported act_type");
    const dn::host::Airframe* frame = dn::host::airframe(cfg->drone_model);
    if (!frame) return fail(DN_EINVAL, "dn_create: unknown drone_model");
    if (cfg->act_type == DN_ACT_THRUST && !frame->has_pwm)     // BaseAviary._parse_urdf_parameters, BaseAviary.py:1157-1160
        return fail(DN_EINVAL, "dn_create: the THRUST action map needs the pwm2rpm attributes, which only cf2x.urdf has");
    if (cfg->act_type >= DN_ACT_PID && cfg->drone_model == DN_MODEL_RACE)   // BaseSingleAgentAviary.py:72-75
        return fail(DN_EINVAL, "dn_create: no controller is available for DroneModel.RACE");
    if (cfg->physics & ~7) return fail(DN_EINVAL, "dn_create: unknown physics flags");
    if (cfg->spawn_mode < DN_SPAWN_FIXED || cfg->spawn_mode > DN_SPAWN_MIDPOINT) return fail(DN_EINVAL, "dn_create: unknown spawn_mode");
    if (cfg->spawn_mode != DN_SPAWN_FIXED && cfg->num_targets < 2) return fail(DN_EINVAL, "dn_create: random spawn needs >= 2 targets");
    if (cfg->max_steps < 0 || cfg->max_steps > (int)dn::kStepsMask - 1) return fail(DN_EINVAL, "dn_create: max_steps out of range");
    dn::RewardParams rw;
    if (!dn::host::reward_table(cfg->reward_id, cfg->discount, rw)) return fail(DN_EINVAL, "dn_create: reward_id not implemented");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DN_ECUDA, "dn_create: no CUDA device (libdronenav has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(DN_EINVAL, "dn_create: bad device index");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(DN_ECUDA, "dn_create: cudaSetDevice failed");

    dn_env* e = new (std::nothrow) dn_env();
    if (!e) return fail(DN_ENOMEM, "dn_create: out of host memory");
    std::memset(e, 0, sizeof(*e));
    e->device = device;
    e->normalize_obs = cfg->normalize_obs ? 1 : 0;
    Params& P = e->P;
    const int N = cfg->num_envs, T = cfg->num_targets;
    std::vector<float4> h_t, h_s;
    dn::host::fill_params(*cfg, rw, P, h_t, h_s, e->d0);
    {   // FULL kernels when any optional feature is on (random spawn, another reward family, reward wrappers, PID actions)
        const bool full = cfg->spawn_mode != DN_SPAWN_FIXED || rw.mode != dn::RW_WAYPOINT || rw.proj_w != 0.0f ||
                          cfg->normalize_reward || cfg->clip_reward > 0.0 || cfg->act_type >= DN_ACT_PID;
        const StepKernel (&ks)[4][2] = e->normalize_obs ? (full ? kStepKernels<true, true> : kStepKernels<true, false>)
                                                        : (full ? kStepKernels<false, true> : kStepKernels<false, false>);
        e->step_one = ks[P.physics & 3][0];
        e->step_many = ks[P.physics & 3][1];
    }

    auto cleanup = [&](int code, const std::string& msg) {
        if (e->state_mem) cudaFree(e->state_mem);
        if (e->d_targets) cudaFree(e->d_targets);
        if (e->d_segs) cudaFree(e->d_segs);
        if (e->d_stats) cudaFree(e->d_stats);
        if (e->d_block_stats) cudaFree(e->d_block_stats);
        delete e;
        return fail(code, msg);
    };
    // persistent state: 7 float4 planes (+ optional drag / obs-RMS planes), one allocation
    const size_t plane = ((static_cast<size_t>(N) * sizeof(float4) + 255) / 256) * 256;
    const size_t fplane = ((static_cast<size_t>(N) * sizeof(float) + 255) / 256) * 256;
    size_t bytes = dn::kPlanes * plane;
    const bool drag = (cfg->physics & DN_PHYS_DRAG) != 0;
    if (drag) bytes += fplane;
    const size_t rms_floats = e->normalize_obs ? static_cast<size_t>(2 * P.obs_dim + 1) * N : 0;
    bytes += ((rms_floats * sizeof(double) + 255) / 256) * 256;
    const bool need_aux = (rw.mode == dn::RW_REACHING || rw.mode == dn::RW_LITERATURE), need_rew_rms = (cfg->normalize_reward != 0);
    const bool need_spawn = (cfg->spawn_mode != DN_SPAWN_FIXED), need_pid = (cfg->act_type >= DN_ACT_PID);
    if (need_pid) bytes += 3 * plane;
    if (need_aux) bytes += plane;
    if (need_rew_rms) bytes += plane;
    if (need_spawn) bytes += plane;
    cudaError_t ce = cudaMalloc(&e->state_mem, bytes);
    if (ce != cudaSuccess) return cleanup(DN_ENOMEM, std::string("dn_create: cudaMalloc state: ") + cudaGetErrorString(ce));
    char* p = static_cast<char*>(e->state_mem);
    for (int k = 0; k < dn::kPlanes; ++k) { P.s[k] = reinterpret_cast<float4*>(p); p += plane; }
    if (drag) { P.last_rpm_sum = reinterpret_cast<float*>(p); p += fplane; }
    if (rms_floats) { P.obs_rms = reinterpret_cast<double*>(p); p += ((rms_floats * sizeof(double) + 255) / 256) * 256; }
    if (need_aux) { P.aux = reinterpret_cast<float4*>(p); p += plane; }
    if (need_rew_rms) { P.rew_rms = reinterpret_cast<float4*>(p); p += plane; }
    if (need_spawn) { P.spawn = reinterpret_cast<float4*>(p); p += plane; }
    if (need_pid) { for (int k = 0; k < 3; ++k) { P.pid[k] = reinterpret_cast<float4*>(p); p += plane; } }
    if ((ce = cudaMalloc(&e->d_targets, T * sizeof(float4))) != cudaSuccess ||
        (ce = cudaMalloc(&e->d_segs, 2 * T * sizeof(float4))) != cudaSuccess ||
        (ce = cudaMalloc(&e->d_stats, sizeof(dn::Stats))) != cudaSuccess ||
        (ce = cudaMalloc(&e->d_block_stats, sizeof(dn::BlockStats) * ((N + dn::kBlock - 1) / dn::kBlock))) != cudaSuccess)
        return cleanup(DN_ENOMEM, std::string("dn_create: cudaMalloc tables: ") + cudaGetErrorString(ce));
    if ((ce = cudaMemcpy(e->d_targets, h_t.data(), T * sizeof(float4), cudaMemcpyHostToDevice)) != cudaSuccess ||
        (ce = cudaMemcpy(e->d_segs, h_s.data(), 2 * T * sizeof(float4), cudaMemcpyHostToDevice)) != cudaSuccess ||
        (ce = cudaMemset(e->d_stats, 0, sizeof(dn::Stats))) != cudaSuccess ||
        (ce = cudaMemset(e->d_block_stats, 0, sizeof(dn::BlockStats) * ((N + dn::kBlock - 1) / dn::kBlock))) != cudaSuccess)
        return cleanup(DN_ECUDA, std::string("dn_create: table upload: ") + cudaGetErrorString(ce));
    e->n_slots = (N + dn::kBlock - 1) / dn::kBlock;
    {
        cudaDeviceProp prop;
        int sms = 148;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) sms = prop.multiProcessorCount;
        P.prefetch_ctas = sms * dn::kCtasPerSm;  // 1024 resident threads per SM at 64 registers
        e->sms = sms;
    }
    P.targets = e->d_targets; P.segs = e->d_segs; P.block_stats = e->d_block_stats;

    dn::init_kernel<<<(N + 255) / 256, 256>>>(P, e->d0);
    ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) return cleanup(DN_ECUDA, std::string("dn_create: init_kernel: ") + cudaGetErrorString(ce));
    e->launches = 1;
    *out = e;
    return DN_OK;
}

int dn_destroy(dn_env* env) {
    if (!env) return DN_OK;
    DeviceGuard guard(env->device);
    if (env->in_flight != InFlight::None) cudaStreamSynchronize(env->host_stream);
    env->in_flight = InFlight::None;
    quiesce(env, "dn_destroy");
    if (env->srv_stream) cudaStreamDestroy(env->srv_stream);
    if (env->srv_doorbell_h) cudaFreeHost(env->srv_doorbell_h);
    if (env->srv_cmd) cudaFree(env->srv_cmd);
    cudaFree(env->state_mem); cudaFree(env->d_targets); cudaFree(env->d_segs); cudaFree(env->d_stats);
    cudaFree(env->d_block_stats);
    if (env->stage) cudaFree(env->stage);
    if (env->zc_flag_h) cudaFreeHost(env->zc_flag_h);
    if (env->zc_counter) cudaFree(env->zc_counter);
    if (env->slab_exec) cudaGraphExecDestroy(env->slab_exec);
    if (env->slab_h) cudaFreeHost(env->slab_h);
    if (env->slab_d) cudaFree(env->slab_d);
    if (env->host_stream) cudaStreamDestroy(env->host_stream);
    delete env;
    return DN_OK;
}

int dn_num_envs(const dn_env* env) { return env ? env->P.n : fail(DN_EINVAL, "null handle"); }
int dn_obs_dim(const dn_env* env) { return env ? env->P.obs_dim : fail(DN_EINVAL, "null handle"); }
int64_t dn_launch_count(const dn_env* env) { return env ? env->launches : 0; }

int dn_reset(dn_env* env, const uint8_t* mask, float* obs_out, void* stream) {
    if (!env) return fail(DN_EINVAL, "dn_reset: null handle");
    { const int rq = quiesce(env, "dn_reset"); if (rq != DN_OK) return rq; }
    DeviceGuard guard(env->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int N = env->P.n;
    if (env->normalize_obs) dn::reset_kernel<true><<<(N + 255) / 256, 256, 0, st>>>(env->P, mask, obs_out);
    else dn::reset_kernel<false><<<(N + 255) / 256, 256, 0, st>>>(env->P, mask, obs_out);
    DN_CUDA(cudaGetLastError());
    env->launches += 1;
    return DN_OK;
}

// The argument checks of the step calls and the dn_step_io -> dn::StepIO conversion; the completion word and the server
// fields are left empty for the caller to fill in.
static int step_io(const dn_env* env, const dn_step_io* io, int num_steps, dn::StepIO& k) {
    if (!env || !io) return fail(DN_EINVAL, "dn_step: null argument");
    if (!io->actions || !io->obs || !io->reward || !io->done) return fail(DN_EINVAL, "dn_step: actions/obs/reward/done are required");
    if (num_steps <= 0) return fail(DN_EINVAL, "dn_step_many: num_steps must be > 0");
    if (reinterpret_cast<uintptr_t>(io->actions) & 15u) return fail(DN_EINVAL, "dn_step: actions must be 16-byte aligned");
    k = dn::StepIO{};
    k.actions = reinterpret_cast<const float4*>(io->actions);
    k.obs = io->obs; k.reward = io->reward; k.done = io->done; k.terminal_obs = io->terminal_obs;
    k.found_targets = io->found_targets; k.episode_return = io->episode_return; k.episode_length = io->episode_length;
    return DN_OK;
}

// One launch of the handle's step kernel: the single-step one for num_steps == 1, the dn_step_many one otherwise.  `pdl`: the
// caller allows a programmatic dependent launch (not inside the slab graph, whose predecessor is a copy node, nor for the server).
static int launch_step(dn_env* env, dn::StepIO k, int num_steps, int per_step, cudaStream_t st, bool pdl) {
    DeviceGuard guard(env->device);
    const int N = env->P.n;
    const dim3 grid((N + dn::kBlock - 1) / dn::kBlock), block(dn::kBlock);
    // Programmatic dependent launch: the step kernel may be scheduled while the previous kernel of the stream is still
    // running (its CTAs trigger at entry); it then waits (griddepcontrol.wait, before its first global access) until that
    // kernel has completed and flushed.  Back-to-back steps -- plain or replayed from a CUDA graph -- thereby hide
    // the launch / CTA-scheduling latency, which is a third of a 4096-env step.
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = 0; lc.stream = st;
    // Only for grids of at most half the SMs: a dependent grid is made resident while its predecessor still runs, so
    // two consecutive small grids each get SMs of their own.  With mid-size grids (0.3 - 1 wave) the early-resident
    // CTAs of the next step pile up on the SMs that had free slots, and the step then runs unbalanced (measured:
    // 65 536 envs 7.7 -> 9.8 us, 16 384 envs with drag / ground effect 7.4 -> 9.1 us per replayed step).
    lc.attrs = attr; lc.numAttrs = (pdl && static_cast<int>(grid.x) * 2 <= env->sms) ? 1 : 0;
    k.pdl_prefetch = static_cast<int>(lc.numAttrs);
    const cudaError_t lerr = num_steps == 1 ? cudaLaunchKernelEx(&lc, env->step_one, env->P, k, 1, 1)
                                            : cudaLaunchKernelEx(&lc, env->step_many, env->P, k, num_steps, per_step);
    DN_CUDA(lerr);
    DN_CUDA(cudaGetLastError());
    env->launches += 1;
    return DN_OK;
}

int dn_step(dn_env* env, const dn_step_io* io, void* stream) {
    dn::StepIO k;
    int rc = step_io(env, io, 1, k);
    if (rc == DN_OK) rc = quiesce(env, "dn_step");
    return rc != DN_OK ? rc : launch_step(env, k, 1, 1, static_cast<cudaStream_t>(stream), true);
}

int dn_step_many(dn_env* env, const dn_step_io* io, int num_steps, int per_step_outputs, void* stream) {
    dn::StepIO k;
    int rc = step_io(env, io, num_steps, k);
    if (rc == DN_OK) rc = quiesce(env, "dn_step_many");
    return rc != DN_OK ? rc : launch_step(env, k, num_steps, per_step_outputs ? 1 : 0, static_cast<cudaStream_t>(stream), true);
}

// Zero-copy classification: if every buffer is pinned host memory mapped into the device address space (torch /
// cudaHostAlloc / cudaHostRegister), the fused kernel reads the actions and writes its outputs over PCIe itself -- one
// launch per step, no staging copies.  The classification is cached on the pointer set.
static int host_classify(dn_env* env, const dn_step_io* h) {
    if (std::memcmp(&env->host_seen, h, sizeof(*h)) == 0) return DN_OK;
    env->host_seen = *h;
    env->host_direct = 1;
    const void* src[8] = {h->actions, h->obs, h->reward, h->done, h->terminal_obs, h->found_targets, h->episode_return, h->episode_length};
    void* dst[8] = {nullptr};
    for (int k = 0; k < 8 && env->host_direct; ++k) {
        if (!src[k]) continue;
        // callers rotate a few action buffers over fixed output buffers: remember what each pointer turned out to be
        // (cudaPointerGetAttributes costs about a microsecond per pointer)
        int hit = -1;
        for (int c = 0; c < env->ptr_cache_n; ++c) if (env->ptr_cache_h[c] == src[k]) { hit = c; break; }
        if (hit >= 0) { dst[k] = env->ptr_cache_d[hit]; continue; }
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, src[k]) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
            cudaGetLastError();
            env->host_direct = 0;
        } else {
            dst[k] = at.devicePointer;
            const int slot = env->ptr_cache_n < 32 ? env->ptr_cache_n++ : (env->ptr_cache_next++ & 31);
            env->ptr_cache_h[slot] = src[k]; env->ptr_cache_d[slot] = at.devicePointer;
        }
    }
    if (env->host_direct && (reinterpret_cast<uintptr_t>(dst[0]) & 15u)) env->host_direct = 0;
    env->host_mapped.actions = static_cast<const float*>(dst[0]); env->host_mapped.obs = static_cast<float*>(dst[1]);
    env->host_mapped.reward = static_cast<float*>(dst[2]); env->host_mapped.done = static_cast<uint8_t*>(dst[3]);
    env->host_mapped.terminal_obs = static_cast<float*>(dst[4]); env->host_mapped.found_targets = static_cast<int32_t*>(dst[5]);
    env->host_mapped.episode_return = static_cast<float*>(dst[6]); env->host_mapped.episode_length = static_cast<int32_t*>(dst[7]);
    return DN_OK;
}

// The completion word of the zero-copy call and of the resident server: a pinned, device-mapped word that the last CTA of
// the step kernel writes after a system-scope fence, and the device counter through which the CTAs find the last one.
static int ensure_completion_word(dn_env* env) {
    if (env->zc_flag_h) return DN_OK;
    void* hp = nullptr; void* dp = nullptr;
    DN_CUDA(cudaHostAlloc(&hp, 64, cudaHostAllocMapped));
    DN_CUDA(cudaHostGetDevicePointer(&dp, hp, 0));
    std::memset(hp, 0, 64);
    env->zc_flag_h = static_cast<unsigned int*>(hp); env->zc_flag_d = static_cast<unsigned int*>(dp);
    DN_CUDA(cudaMalloc(reinterpret_cast<void**>(&env->zc_counter), 64));
    DN_CUDA(cudaMemset(env->zc_counter, 0, 64));
    return DN_OK;
}

// One launch of the step kernel on the mapped host buffers; the kernel announces completion through the completion word.
static int zero_copy_launch(dn_env* env) {
    dn::StepIO k;
    int rc = ensure_completion_word(env);
    if (rc == DN_OK) rc = step_io(env, &env->host_mapped, 1, k);
    if (rc != DN_OK) return rc;
    env->zc_seq += 1; if (env->zc_seq == 0u) env->zc_seq = 1u;
    // the word is shared with the resident server (its own sequence numbers): never start a wait on a stale equal value
    if (*reinterpret_cast<volatile unsigned int*>(env->zc_flag_h) == env->zc_seq) *reinterpret_cast<volatile unsigned int*>(env->zc_flag_h) = 0u;
    k.done_counter = env->zc_counter; k.host_flag = env->zc_flag_d; k.seq = env->zc_seq;
    return launch_step(env, k, 1, 1, env->host_stream, true);
}

// Spins until the pinned completion word holds `want`.  Every 2^16 spins it looks at the stream, so that a failed launch, or a
// step that finished without writing the word, ends in an error instead of an endless spin.
static int wait_word(dn_env* env, const volatile uint32_t* word, uint32_t want, cudaStream_t st, const char* who, const char* message) {
    for (uint32_t spins = 0; *word != want;) {
        if ((++spins & 0xFFFFu) != 0u) continue;
        DeviceGuard guard(env->device);
        const cudaError_t e = cudaStreamQuery(st);
        if (e != cudaErrorNotReady && *word != want)
            return fail(DN_ECUDA, std::string(who) + ": " + (e == cudaSuccess ? message : cudaGetErrorString(e)));
    }
    return DN_OK;
}

static int zero_copy_wait(dn_env* env) {
    return wait_word(env, env->zc_flag_h, env->zc_seq, env->host_stream, "dn_step_host", "the step finished without writing the completion word");
}

// ---------------------------------------------------------------------------------------------------------------------------
// Resident step server.  A host step through a kernel LAUNCH costs 13 us before any byte has moved (launch, scheduling,
// completion hand-off: tools/e2e_breakdown.py).  With dn_host_server(env, idle_us) the step kernel (the dn_step_many variant:
// state in registers, stored every step) stays resident instead: the host writes the step's actions, rings a doorbell word in
// pinned memory and polls the completion word; the kernel leaves by itself after `idle_us` without a command and is launched
// again by the next dn_step_host.  Every other call that touches the handle's state stops the server first (quiesce).
// ---------------------------------------------------------------------------------------------------------------------------
static int srv_start(dn_env* env, unsigned int seq_done) {
    if (!env->srv_stream) {
        DN_CUDA(cudaStreamCreateWithFlags(&env->srv_stream, cudaStreamNonBlocking));
        void* hp = nullptr; void* dp = nullptr;
        DN_CUDA(cudaHostAlloc(&hp, 128, cudaHostAllocMapped));
        DN_CUDA(cudaHostGetDevicePointer(&dp, hp, 0));
        std::memset(hp, 0, 128);
        env->srv_doorbell_h = static_cast<unsigned long long*>(hp); env->srv_doorbell_d = static_cast<unsigned long long*>(dp);
        env->srv_word_h = env->srv_doorbell_h + 8;
        DN_CUDA(cudaMalloc(reinterpret_cast<void**>(&env->srv_cmd), 64));
    }
    // the command word the kernel starts from: "step seq_done has been run" (any non-zero pointer field)
    *env->srv_word_h = (static_cast<unsigned long long>(seq_done) << 48) | 1ull;
    DN_CUDA(cudaMemcpyAsync(env->srv_cmd, env->srv_word_h, 8, cudaMemcpyHostToDevice, env->srv_stream));
    dn_step_io io = env->srv_io;
    io.actions = reinterpret_cast<const float*>(env->srv_doorbell_d);   // placeholder (16-byte aligned); the commands carry the real pointer
    dn::StepIO k;
    int rc = step_io(env, &io, 0x7fffffff, k);
    if (rc != DN_OK) return rc;
    k.done_counter = env->zc_counter; k.host_flag = env->zc_flag_d;
    k.srv_doorbell = env->srv_doorbell_d; k.srv_cmd = env->srv_cmd; k.srv_word0 = *env->srv_word_h;
    k.srv_idle_us = static_cast<unsigned int>(env->srv_idle_us);
    rc = launch_step(env, k, 0x7fffffff, 0, env->srv_stream, false);
    if (rc != DN_OK) return rc;
    env->srv_alive = 1;
    env->srv_residencies += 1;
    return DN_OK;
}

// one step through the server; env->host_mapped holds the mapped pointers of this call
static int srv_step(dn_env* env) {
    const dn_step_io& m = env->host_mapped;
    if (reinterpret_cast<uintptr_t>(m.actions) >> 48) return fail(DN_EINVAL, "dn_step_host: device pointer does not fit the doorbell word");
    dn_step_io outs = m; outs.actions = nullptr;
    if (env->srv_alive && std::memcmp(&outs, &env->srv_io, sizeof(outs)) != 0) {      // other output buffers: new residency
        const int rq = quiesce(env, "dn_step_host");
        if (rq != DN_OK) return rq;
    }
    const int rw = ensure_completion_word(env);
    if (rw != DN_OK) return rw;
    const unsigned int prev = env->srv_seq;
    const unsigned int seq = (prev % 0xFFFFu) + 1u;
    if (!env->srv_alive) {
        env->srv_io = outs;
        *reinterpret_cast<volatile unsigned int*>(env->zc_flag_h) = 0u;
        const int rs = srv_start(env, prev);
        if (rs != DN_OK) return rs;
    }
    env->srv_seq = seq;
    volatile unsigned int* flag = env->zc_flag_h;
    *reinterpret_cast<volatile unsigned long long*>(env->srv_doorbell_h) =
        (static_cast<unsigned long long>(seq) << 48) | static_cast<unsigned long long>(reinterpret_cast<uintptr_t>(m.actions));
    uint32_t spins = 0, restarts = 0;
    while (*flag != seq) {
        if ((++spins & 0x3FFFu) == 0u) {
            // the server may have left (idle) just before the doorbell rang: its stream is then idle -- start another residency,
            // which finds the pending command at once.  An error on the stream must surface, not spin.
            const cudaError_t e = cudaStreamQuery(env->srv_stream);
            if (e == cudaErrorNotReady) continue;
            if (*flag == seq) break;
            env->srv_alive = 0;
            if (e != cudaSuccess) return fail(DN_ECUDA, std::string("dn_step_host (server): ") + cudaGetErrorString(e));
            if (++restarts > 8u) return fail(DN_ECUDA, "dn_step_host (server): the resident kernel keeps leaving without running the step");
            const int rs = srv_start(env, prev);
            if (rs != DN_OK) return rs;
        }
    }
    env->srv_steps += 1;          // (no launch: dn_launch_count counts the residencies)
    return DN_OK;
}

int dn_host_server(dn_env* env, int idle_us) {
    if (!env) return fail(DN_EINVAL, "dn_host_server: null handle");
    if (idle_us < 0 || idle_us > 1000000) return fail(DN_EINVAL, "dn_host_server: idle_us must be in [0, 1000000]");
    const int rq = quiesce(env, "dn_host_server");
    if (rq != DN_OK) return rq;
    // every CTA of the resident grid must fit on the device at once (they wait for each other's commands)
    const int grid = (env->P.n + dn::kBlock - 1) / dn::kBlock;
    if (idle_us > 0 && grid > 4 * env->sms) return fail(DN_EINVAL, "dn_host_server: more environments than a resident grid can hold (4 CTAs per SM)");
    env->srv_idle_us = idle_us;
    return DN_OK;
}

int dn_host_server_stats(dn_env* env, int64_t* residencies, int64_t* steps) {
    if (!env) return fail(DN_EINVAL, "dn_host_server_stats: null handle");
    if (residencies) *residencies = env->srv_residencies;
    if (steps) *steps = env->srv_steps;
    return DN_OK;
}

static int ensure_host_stream(dn_env* env) {
    if (!env->host_stream) DN_CUDA(cudaStreamCreateWithFlags(&env->host_stream, cudaStreamNonBlocking));
    return DN_OK;
}

int dn_host_buffers(dn_env* env, int with_episode_info, dn_step_io* out) {
    if (!env || !out) return fail(DN_EINVAL, "dn_host_buffers: null argument");
    { const int rq = quiesce(env, "dn_host_buffers"); if (rq != DN_OK) return rq; }
    DeviceGuard guard(env->device);
    { const int rs = ensure_host_stream(env); if (rs != DN_OK) return rs; }
    if (env->slab_h && env->slab.episode != (with_episode_info != 0)) {
        if (env->slab_exec) { cudaGraphExecDestroy(env->slab_exec); env->slab_exec = nullptr; }
        cudaFreeHost(env->slab_h); cudaFree(env->slab_d);
        env->slab_h = env->slab_d = nullptr;
    }
    if (!env->slab_h) {
        const IoLayout L = io_layout(env->P.n, env->P.obs_dim, with_episode_info != 0);
        void* hp = nullptr; void* dp = nullptr;
        DN_CUDA(cudaHostAlloc(&hp, L.bytes, cudaHostAllocDefault));
        cudaError_t ce = cudaMalloc(&dp, L.bytes);
        if (ce != cudaSuccess) { cudaFreeHost(hp); return fail(DN_ENOMEM, std::string("dn_host_buffers: cudaMalloc: ") + cudaGetErrorString(ce)); }
        std::memset(hp, 0, L.bytes);
        DN_CUDA(cudaMemset(dp, 0, L.bytes));
        const uint32_t one = 1;                        // the completion word: constant 1 on the device, cleared on the host before a launch
        DN_CUDA(cudaMemcpy(static_cast<char*>(dp) + L.word, &one, 4, cudaMemcpyHostToDevice));
        env->slab_h = static_cast<char*>(hp); env->slab_d = static_cast<char*>(dp);
        env->slab = L;
        env->slab_io_h = io_at(L, env->slab_h);
        env->slab_io_d = io_at(L, env->slab_d);
    }
    *out = env->slab_io_h;
    return DN_OK;
}

int dn_step_host_async(dn_env* env, const dn_step_io* h) {
    if (!env || !h) return fail(DN_EINVAL, "dn_step_host_async: null argument");
    { const int rq = quiesce(env, "dn_step_host_async"); if (rq != DN_OK) return rq; }
    DeviceGuard guard(env->device);
    if (!env->slab_h || std::memcmp(h, &env->slab_io_h, sizeof(*h)) != 0) {
        // caller-owned buffers: only the zero-copy form (pinned + mapped) can be left in flight
        if (!h->actions || !h->obs || !h->reward || !h->done) return fail(DN_EINVAL, "dn_step_host_async: actions/obs/reward/done are required");
        int rc = ensure_host_stream(env);
        if (rc == DN_OK) rc = host_classify(env, h);
        if (rc != DN_OK) return rc;
        if (!env->host_direct)
            return fail(DN_EINVAL, "dn_step_host_async: needs pinned, device-mapped host buffers or the buffers dn_host_buffers returned");
        rc = zero_copy_launch(env);
        if (rc != DN_OK) return rc;
        env->in_flight = InFlight::ZeroCopy;
        return DN_OK;
    }
    cudaStream_t st = env->host_stream;
    if (!env->slab_exec) {
        // capture once: H2D(actions) -> fused step kernel -> D2H(outputs + completion word)
        dn::StepIO k;
        int rc = step_io(env, &env->slab_io_d, 1, k);
        if (rc != DN_OK) return rc;
        cudaGraph_t graph = nullptr;
        DN_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        cudaError_t ce = cudaMemcpyAsync(env->slab_d, env->slab_h, static_cast<size_t>(env->P.n) * 16, cudaMemcpyHostToDevice, st);
        rc = (ce == cudaSuccess) ? launch_step(env, k, 1, 1, st, false) : DN_ECUDA;
        if (ce == cudaSuccess && rc == DN_OK)
            ce = cudaMemcpyAsync(env->slab_h + env->slab.obs, env->slab_d + env->slab.obs, env->slab.word + 4 - env->slab.obs, cudaMemcpyDeviceToHost, st);
        cudaError_t ce2 = cudaStreamEndCapture(st, &graph);
        if (rc != DN_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess || ce2 != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            return fail(DN_ECUDA, std::string("dn_step_host_async: graph capture: ") + cudaGetErrorString(ce != cudaSuccess ? ce : ce2));
        }
        ce = cudaGraphInstantiate(&env->slab_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { env->slab_exec = nullptr; return fail(DN_ECUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce)); }
        env->launches -= 1;                            // the captured launch is counted per replay below
    }
    *reinterpret_cast<volatile uint32_t*>(env->slab_h + env->slab.word) = 0u;
    DN_CUDA(cudaGraphLaunch(env->slab_exec, st));
    env->in_flight = InFlight::Slab;
    env->launches += 1;
    return DN_OK;
}

int dn_step_host_wait(dn_env* env) {
    if (!env) return fail(DN_EINVAL, "dn_step_host_wait: null handle");
    const InFlight f = env->in_flight;
    env->in_flight = InFlight::None;
    if (f == InFlight::ZeroCopy) return zero_copy_wait(env);
    if (f == InFlight::Slab)                           // the graph's D2H copy writes the device's constant 1 to the word last
        return wait_word(env, reinterpret_cast<volatile uint32_t*>(env->slab_h + env->slab.word), 1u, env->host_stream,
                         "dn_step_host_wait", "the graph finished without setting the completion word");
    return DN_OK;
}

int dn_step_host(dn_env* env, const dn_step_io* h) {
    if (!env || !h) return fail(DN_EINVAL, "dn_step_host: null argument");
    if (!h->actions || !h->obs || !h->reward || !h->done) return fail(DN_EINVAL, "dn_step_host: actions/obs/reward/done are required");
    if (env->slab_h && std::memcmp(h, &env->slab_io_h, sizeof(*h)) == 0) {     // the handle's own slab: graph replay
        const int rc = dn_step_host_async(env, h);
        return rc != DN_OK ? rc : dn_step_host_wait(env);
    }
    DeviceGuard guard(env->device);
    int rc = ensure_host_stream(env);
    if (rc == DN_OK) rc = host_classify(env, h);
    const bool server = env->host_direct && env->srv_idle_us > 0;
    if (rc == DN_OK) rc = quiesce(env, "dn_step_host", !server);
    if (rc != DN_OK) return rc;
    if (server) return srv_step(env);
    if (env->host_direct) {
        rc = zero_copy_launch(env);
        return rc != DN_OK ? rc : zero_copy_wait(env);
    }
    const size_t N = env->P.n, D = env->P.obs_dim;
    const IoLayout L = io_layout(N, D, true);
    if (!env->stage) DN_CUDA(cudaMalloc(&env->stage, L.bytes));
    char* d = static_cast<char*>(env->stage);
    cudaStream_t st = env->host_stream;
    DN_CUDA(cudaMemcpyAsync(d + L.act, h->actions, N * 16, cudaMemcpyHostToDevice, st));
    dn_step_io io = io_at(L, d);
    if (!h->terminal_obs) io.terminal_obs = nullptr;
    if (!h->found_targets) io.found_targets = nullptr;
    if (!h->episode_return) io.episode_return = nullptr;
    if (!h->episode_length) io.episode_length = nullptr;
    dn::StepIO k;
    rc = step_io(env, &io, 1, k);
    if (rc == DN_OK) rc = launch_step(env, k, 1, 1, st, true);
    if (rc != DN_OK) return rc;
    DN_CUDA(cudaMemcpyAsync(h->obs, io.obs, N * D * 4, cudaMemcpyDeviceToHost, st));
    DN_CUDA(cudaMemcpyAsync(h->reward, io.reward, N * 4, cudaMemcpyDeviceToHost, st));
    DN_CUDA(cudaMemcpyAsync(h->done, io.done, N, cudaMemcpyDeviceToHost, st));
    if (h->found_targets) DN_CUDA(cudaMemcpyAsync(h->found_targets, io.found_targets, N * 4, cudaMemcpyDeviceToHost, st));
    if (h->terminal_obs) DN_CUDA(cudaMemcpyAsync(h->terminal_obs, io.terminal_obs, N * D * 4, cudaMemcpyDeviceToHost, st));
    if (h->episode_return) DN_CUDA(cudaMemcpyAsync(h->episode_return, io.episode_return, N * 4, cudaMemcpyDeviceToHost, st));
    if (h->episode_length) DN_CUDA(cudaMemcpyAsync(h->episode_length, io.episode_length, N * 4, cudaMemcpyDeviceToHost, st));
    DN_CUDA(cudaStreamSynchronize(st));
    return DN_OK;
}

int dn_action_to_rpm(dn_env* env, const float* actions, float* rpm_out, int64_t n, void* stream) {
    if (!env || !actions || !rpm_out || n < 0) return fail(DN_EINVAL, "dn_action_to_rpm: bad argument");
    if (env->P.act_type >= DN_ACT_PID)
        return fail(DN_EINVAL, "dn_action_to_rpm: the PID action types are not elementwise maps (the RPMs depend on the drone and controller state)");
    if (n == 0) return DN_OK;
    DeviceGuard guard(env->device);
    dn::action_map_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(env->P, actions, rpm_out, n);
    DN_CUDA(cudaGetLastError());
    env->launches += 1;
    return DN_OK;
}

int dn_gae(const float* rewards, const float* values, const uint8_t* done, const float* last_values,
           float gamma, float gae_lambda, float* advantages_out, float* returns_out,
           int32_t num_steps, int32_t num_envs, void* stream) {
    if (!rewards || !values || !done || !last_values || !advantages_out || !returns_out || num_steps <= 0 || num_envs <= 0)
        return fail(DN_EINVAL, "dn_gae: bad argument");
    dn::gae_kernel<<<(num_envs + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
        rewards, values, done, last_values, gamma, gae_lambda, advantages_out, returns_out, num_steps, num_envs);
    DN_CUDA(cudaGetLastError());
    return DN_OK;
}

static int state_xfer(dn_env* env, const dn_state_view* v, bool set, void* stream) {
    if (!env || !v) return fail(DN_EINVAL, "dn_get/set_state: null argument");
    { const int rq = quiesce(env, set ? "dn_set_state" : "dn_get_state"); if (rq != DN_OK) return rq; }
    DeviceGuard guard(env->device);
    dn::StateView V;
    V.pos = v->pos; V.quat = v->quat; V.vel = v->vel; V.rpy_rates = v->rpy_rates; V.ang_v = v->ang_v;
    V.prev_vel = v->prev_vel; V.prev_ang_v = v->prev_ang_v; V.dist = v->dist; V.prev_dist = v->prev_dist;
    V.target_idx = v->target_idx; V.steps = v->steps; V.just_found = v->just_found; V.ep_return = v->ep_return;
    V.ep_length = v->ep_length; V.episode_count = v->episode_count; V.last_rpm_sum = v->last_rpm_sum; V.obs_rms = v->obs_rms;
    V.aux = v->aux; V.rew_rms = v->rew_rms; V.spawn = v->spawn; V.pid = v->pid;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int N = env->P.n;
    if (set) dn::state_xfer_kernel<true><<<(N + 255) / 256, 256, 0, st>>>(env->P, V);
    else dn::state_xfer_kernel<false><<<(N + 255) / 256, 256, 0, st>>>(env->P, V);
    DN_CUDA(cudaGetLastError());
    env->launches += 1;
    return DN_OK;
}

int dn_get_state(dn_env* env, const dn_state_view* view, void* stream) { return state_xfer(env, view, false, stream); }
int dn_set_state(dn_env* env, const dn_state_view* view, void* stream) { return state_xfer(env, view, true, stream); }

int dn_episode_stats(dn_env* env, dn_stats* host_out, int clear, void* stream) {
    if (!env || !host_out) return fail(DN_EINVAL, "dn_episode_stats: null argument");
    { const int rq = quiesce(env, "dn_episode_stats"); if (rq != DN_OK) return rq; }
    DeviceGuard guard(env->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dn::Stats h;
    dn::stats_reduce_kernel<<<1, 256, 0, st>>>(env->d_block_stats, env->n_slots, env->d_stats, clear ? 1 : 0);
    DN_CUDA(cudaGetLastError());
    env->launches += 1;
    DN_CUDA(cudaMemcpyAsync(&h, env->d_stats, sizeof(h), cudaMemcpyDeviceToHost, st));
    DN_CUDA(cudaStreamSynchronize(st));
    host_out->return_sum = h.return_sum; host_out->length_sum = h.length_sum; host_out->episodes = h.episodes;
    host_out->successes = h.successes; host_out->found_targets = h.found_targets; host_out->crashes = h.crashes;
    host_out->truncations = h.truncations;
    return DN_OK;
}

}  // extern "C"
