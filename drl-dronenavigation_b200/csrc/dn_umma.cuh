// dn_umma.cuh -- hand-written sm_100a GEMM building blocks for the PPO minibatch update:
// TMA (cp.async.bulk.tensor) operand loads into 128B-swizzled shared memory, tcgen05.mma (kind::f16, BF16 inputs,
// FP32 accumulation in TMEM) issued by one thread, tcgen05.ld epilogues fused with the elementwise work of the layer.
//
// One persistent, warp-specialised kernel template `umma_gemm<KIND, BN>` serves the three contractions of an MLP layer
//   FWD    Y  = tanh(X W^T + b)            A = X  [M,K]   K-major, B = W  [N,K]    K-major   (FWD_RELU: max(X W^T + b, 0))
//   DGRAD  dX = (dY W) * (1 - H^2)         A = dY [M,N]   K-major, B = W  [N,K]    MN-major (reduction over W's rows)
//   WGRAD  dW = dY^T X  (split over rows)  A = dY [m,N]   MN-major, B = X [m,K]    MN-major (reduction over the batch rows)
// so that no transposed copy of an activation, a gradient or a weight is ever written.
//
// FP32-faithful arithmetic on BF16 tensor cores: every FP32 matrix is stored as two BF16 planes, hi = bf16(x) and
// lo = bf16(x - hi) (plane 1 follows plane 0 in the same allocation), and a product is accumulated as
//   A B ~= A_hi B_hi + A_hi B_lo + A_lo B_hi          (3 passes over K into the same TMEM accumulator; the dropped
// lo*lo term and the rounding of lo are ~2^-16 relative to |a||b| per product, 7e-6 on the network's gradients).
// `passes = 1` is plain BF16 (hi planes only), offered as a labelled option.
//
// What the kernel is built around (ncu on the first version: L2 -> SM traffic at the ~12 TB/s slice limit, and the
// epilogue's per-row 16-byte global accesses throttling the LSU):
//   * a pipeline stage holds BOTH planes of the A and the B tile of one k-block; the three products of a k-block are
//     issued from that one copy (the first version re-loaded every plane per pass: 1.5x the L2 traffic);
//   * CG = 2: CTA pairs (cta_group::2, UMMA M = 256): each CTA loads its own 128 rows of A and HALF of the B tile, the
//     tensor cores of the pair read both halves -- B traffic per CTA halves, the 256-wide tile fits two pipeline stages
//     next to the epilogue buffers;
//   * epilogue through shared memory: every epilogue warp owns two 4 KB staging buffers; results leave as TMA bulk
//     tensor stores (full 64-byte rows, no LSU pressure), the tanh output the dgrad epilogue needs arrives the same way
//     one chunk ahead (TMA load + mbarrier), and the buffer it arrived in is reused for the result.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace dnmma {

constexpr int BM = 128;            // accumulator rows per CTA (= TMEM lanes)
constexpr int BK = 32;             // BF16 elements per k-block (pipeline stage).  64 left only two 64 KB stages in the ring: one stage
                                   // in flight cannot cover the TMA latency (probe: operand loads alone 25 us, MMAs alone 25 us, both 41 us)
constexpr int UK = 16;             // K of one tcgen05.mma.kind::f16
constexpr int NUM_THREADS = 384;   // warp 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 3 spare, 4..11 epilogue
constexpr int EPI_WARP0 = 4;
constexpr int EPI_WARPS = 8;
constexpr int MAX_STAGES = 8;
constexpr uint32_t RING_BYTES = 131072;              // operand ring (>= 2 stages of the largest configuration)
constexpr uint32_t EPI_BUF_BYTES = 4096;             // one chunk: 32 rows x 32 columns, hi plane (2 KB) | lo plane (2 KB)
constexpr uint32_t EPI_BYTES = EPI_WARPS * 2 * EPI_BUF_BYTES;
constexpr int MAX_COLSUM_COLS = 512;                 // widest DGRAD result whose column sums fit the shared-memory accumulator
constexpr int GROUP_FLOATS = 4 * MAX_COLSUM_COLS;      // shared-memory floats per problem of a launch (column sums [4][ld_out] / the bias vector)
constexpr int MAX_GROUPS = 2;                         // problems of identical shape in one launch (the policy and the value net)
constexpr uint32_t COLSUM_BYTES = MAX_GROUPS * GROUP_FLOATS * 4;
constexpr uint32_t BAR_BYTES = 512;
constexpr uint32_t SMEM_BYTES = 1024 /* alignment slack */ + RING_BYTES + EPI_BYTES + COLSUM_BYTES + BAR_BYTES;
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;      // shared::cluster address of the same offset in the even CTA of a pair

// K_FWD_RELU: the forward contraction with max(x, 0) as a compile-time epilogue (the SAC actor's latent layers).  A kind of
// its own rather than a third runtime value of GemmArgs::act, so that the K_FWD instantiations keep their code.
enum Kind { K_FWD = 0, K_DGRAD = 1, K_WGRAD = 2, K_FWD_RELU = 3 };

struct GemmArgs {
    int m_tiles, n_tiles, slices;   // tile grid: accumulator rows / (128 CG), accumulator columns / BN, split of the reduction
    int k_blocks;                   // BK-wide k-blocks of the reduction (WGRAD: of ALL slices; slice s takes [s KB / S, (s + 1) KB / S))
    int passes;                     // 1 (BF16) or 3 (hi*hi + hi*lo + lo*hi)
    int a_lo_row, b_lo_row;         // row of the lo plane inside the A / B tensor maps (rows of plane 0)
    int c_lo_row;                   // row of the lo plane inside the result / H tensor maps
    int act;                        // FWD: 1 = tanh, 0 = identity
    const float* bias;              // FWD: [N]
    int ld_out;                     // FWD / DGRAD: columns of the result (and of H)
    float* partial;                 // WGRAD: [slices][rows][ld_partial] FP32 partial products
    int ld_partial;
    long long slice_stride;         // elements between slices of `partial`
    float* colsum;                  // DGRAD, optional: [gridDim.x][ld_out] column sums of the FP32 result over this CTA's tiles
                                    // (= this CTA's share of the bias gradient of the layer below)
    // Two problems of IDENTICAL shape in one launch (the policy net's and the value net's layer l): tiles [0, T) belong to the
    // first problem (tensor maps 1..4 of the kernel, the pointers above), tiles [T, 2T) to the second (maps 5..8, the pointers
    // below).  One wave quantisation instead of two: 256 tiles on 74 CTA pairs are 4 rounds, 512 tiles are 7.
    int groups;                     // 1 or 2
    const float* bias2;
    float* partial2;
    float* colsum2;
};

// ------------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on the barrier at the same offset in the EVEN CTA of the pair (a no-op mask for that CTA itself)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded spin: a protocol error becomes a trap (an error the host sees) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 27)) __trap();
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load: the box lands densely in shared memory with the map's swizzle, bytes counted on `bar`.
// CG = 2: the bytes are counted on the barrier at the same offset in the even CTA of the pair (the one that issues the MMAs).
template <int CG>
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1) {
    if constexpr (CG == 1) {
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
            : "memory");
    } else {
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                smem_u32(dst)),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0), "r"(c1)
            : "memory");
    }
}
// 2-D tiled store of a shared-memory box (bulk async group of the issuing thread)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    if constexpr (CG == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
    else
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], BF16 inputs, FP32 accumulate.  CG = 2: one instruction drives the tensor cores of both
// CTAs of the pair (M = 256: each CTA's TMEM receives its 128 rows; each CTA's shared memory supplies its A rows and half of B).
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        const uint32_t z = 0;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z)
            : "memory");
    }
}
// mbarrier arrive once every MMA issued so far by this thread has completed (implies tcgen05.fence::before_thread_sync).
// CG = 2: the arrive is multicast to the barrier at the same offset in both CTAs of the pair.
template <int CG>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
    } else {
        const uint16_t mask = 3;
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                     "h"(mask)
                     : "memory");
    }
}

// 32 lanes x 32 consecutive FP32 columns of the accumulator -> 32 registers per thread (thread = accumulator row).
// Issue and completion are separate so that the next chunk's load is in flight while the current one is worked on;
// tmem_ld_wait names the registers as in/out operands: nothing may read them before the wait.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                   "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                   "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}

// ------------------------------------------------------------------------------------------------------------------
// descriptors (bit layouts: cute/arch/mma_sm100_desc.hpp of the CUTLASS tree vendored in this image)
// ------------------------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor; offsets in bytes; layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);              // [0,14)  start address >> 4
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;    // [16,30) leading-dimension byte offset >> 4
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;    // [32,46) stride-dimension byte offset >> 4
    d |= static_cast<uint64_t>(1) << 46;                            // [46,48) descriptor version 1 (Blackwell)
    d |= static_cast<uint64_t>(layout) << 61;                       // [61,64) layout type
    return d;
}
// K-major operand tile: rows x 32 BF16, each row one 64-byte line under the 64-byte swizzle; 8-row groups 512 bytes apart;
// the k-th UMMA_K slice (16 elements) starts 32 bytes further inside the line
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t tile, int k) { return smem_desc(tile + k * (UK * 2), 16, 512, 4); }
// MN-major operand tile: TMA boxes of 32 k-rows x 64 contiguous MN elements under the 128-byte swizzle (4096 bytes per box,
// boxes side by side along MN); 8-k-row groups 1024 bytes apart (SBO), 64-element MN chunks one box apart (LBO); the k-th
// UMMA_K slice starts 16 k-rows = 2048 bytes further
constexpr uint32_t MN_BOX_BYTES = BK * 128;
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t tile, int k) { return smem_desc(tile + k * (UK * 128), MN_BOX_BYTES, 1024, 2); }

// instruction descriptor: D = F32, A = B = BF16, M = m, N = n
__host__ __device__ constexpr uint32_t instr_desc(int m, int n, int a_mn_major, int b_mn_major) {
    return (1u << 4)                                  // [4,6)   D format F32
           | (1u << 7)                                // [7,10)  A format BF16
           | (1u << 10)                               // [10,13) B format BF16
           | (static_cast<uint32_t>(a_mn_major) << 15)  // [15]    A major (0 = K, 1 = MN)
           | (static_cast<uint32_t>(b_mn_major) << 16)  // [16]    B major
           | (static_cast<uint32_t>(n >> 3) << 17)      // [17,23) N >> 3
           | (static_cast<uint32_t>(m >> 4) << 24);     // [24,29) M >> 4
}

// ------------------------------------------------------------------------------------------------------------------
// helpers of the epilogues
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(__nv_bfloat16 a, __nv_bfloat16 b) {
    return static_cast<uint32_t>(__bfloat16_as_ushort(a)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b)) << 16);
}
__device__ __forceinline__ float bf16lo_f(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi_f(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }
// (a, b) -> packed hi pair and packed lo pair.  One packed conversion per pair (F2FP.BF16.F32.PACK_AB, an ALU instruction):
// converting element by element compiles to F2F.BF16.F32, which shares the quarter-rate pipe with MUFU -- ncu showed the
// 64 single conversions of a 32-column chunk costing as much as the chunk's 64 MUFU ops and the epilogue out-lasting the MMAs.
__device__ __forceinline__ void split_pair(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);          // .x = a in the low half
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(a - bf16lo_f(hi), b - bf16hi_f(hi));
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// tanh(x) = 1 - 2 / (1 + e^(2x)) with the two MUFU approximations (ex2, rcp): absolute error <= 3e-7 over the whole
// range (|tanh| <= 1, so this is the FP32-level accuracy the planes can carry anyway), saturates to +-1 without special
// cases, 5 instructions instead of libm's ~30
__device__ __forceinline__ float tanh_fast(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return fmaf(-2.0f, r, 1.0f);
}

// The staging buffers hold 32 rows of 64 bytes under the tensor maps' 64-byte swizzle: 16-byte piece j of row r sits at
// piece j ^ ((r >> 1) & 3) (address bits [4,6) xor bits [7,9)).
__device__ __forceinline__ uint32_t stage_off(int row, int piece) { return row * 64 + ((piece ^ ((row >> 1) & 3)) << 4); }

// 32 FP32 values of this lane's row -> hi / lo BF16 pieces in the staging buffer (hi plane at +0, lo plane at +2048)
__device__ __forceinline__ void stage_split32(const float (&y)[32], uint8_t* buf, int lane, bool write_lo) {
    uint32_t h[16], l[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) split_pair(y[2 * j], y[2 * j + 1], h[j], l[j]);
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(buf + stage_off(lane, q)) = make_uint4(h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]);
    if (write_lo) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(buf + 2048 + stage_off(lane, q)) = make_uint4(l[4 * q], l[4 * q + 1], l[4 * q + 2], l[4 * q + 3]);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// the kernel.  BN = accumulator columns of a tile; CG = CTAs that share a tile (1, or 2 = cta_group::2 pair).
// Tensor maps: tmA / tmB the operands (K-major: boxes of rows x 32 columns, 64-byte swizzle; MN-major: boxes of 32 rows x 64
// columns, 128-byte swizzle), tmC the result planes and tmH the
// tanh-output planes of DGRAD (64-byte swizzle, box 32 columns x 32 rows).
// ------------------------------------------------------------------------------------------------------------------
template <int KIND, int BN, int CG>
__global__ void __launch_bounds__(NUM_THREADS, 1)
umma_gemm(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
          const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
          const __grid_constant__ CUtensorMap tmC2, const __grid_constant__ CUtensorMap tmH2, const GemmArgs g) {
    static_assert(BN % 64 == 0 && BN >= 64 && BN <= 256 && (CG == 1 || CG == 2) && (BN / CG) % 64 == 0, "tile shape");
    constexpr int BNL = BN / CG;                          // rows (K-major) / columns (MN-major) of B this CTA loads
    constexpr uint32_t A_BYTES = BM * BK * 2;             // one plane of the A tile: 16 KB
    constexpr uint32_t B_BYTES = BNL * BK * 2;            // one plane of this CTA's share of the B tile
    constexpr uint32_t IDESC = instr_desc(BM * CG, BN, KIND == K_WGRAD, KIND != K_FWD && KIND != K_FWD_RELU);
    constexpr uint32_t TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* epi_base = smem + RING_BYTES;
    float* colsum_s = reinterpret_cast<float*>(epi_base + EPI_BYTES);             // [4][ld_out] (DGRAD with g.colsum)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_base + EPI_BYTES + COLSUM_BYTES);
    uint64_t* empty_bar = full_bar + MAX_STAGES;
    uint64_t* tfull_bar = empty_bar + MAX_STAGES;   // [2] accumulator stage ready for the epilogue
    uint64_t* tempty_bar = tfull_bar + 2;           // [2] accumulator stage drained (lives in the even CTA of a pair)
    uint64_t* h_bar = tempty_bar + 2;               // [EPI_WARPS][2] H chunk landed in the warp's staging buffer
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(h_bar + 2 * EPI_WARPS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (CG == 1) ? 0 : static_cast<int>(cluster_ctarank());
    const int cid = blockIdx.x / CG, ncl = gridDim.x / CG;            // tile loop: one tile per cluster per round
    const int planes = (g.passes == 3) ? 2 : 1;
    const uint32_t stage_bytes = planes * (A_BYTES + B_BYTES);
    const int stages = (RING_BYTES / stage_bytes) > MAX_STAGES ? MAX_STAGES : static_cast<int>(RING_BYTES / stage_bytes);
    const int group_tiles = g.m_tiles * g.n_tiles * g.slices;     // tiles of one problem
    const int total_tiles = group_tiles * g.groups;

    // Programmatic dependent launch (launch_one sets the attribute): the next kernel of the stream may be scheduled as soon as
    // this one's CTAs leave their SMs, and this kernel sets up (barriers, TMEM, descriptors) while its predecessor drains;
    // nothing below touches global memory before griddepcontrol.wait, which returns once the predecessor has completed and its
    // writes are visible.  Both instructions are no-ops for a normal launch.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if constexpr (KIND != K_WGRAD) tma_prefetch_desc(&tmC);
        if constexpr (KIND == K_DGRAD) tma_prefetch_desc(&tmH);
        if (g.groups > 1) {
            tma_prefetch_desc(&tmA2);
            tma_prefetch_desc(&tmB2);
            if constexpr (KIND != K_WGRAD) tma_prefetch_desc(&tmC2);
            if constexpr (KIND == K_DGRAD) tma_prefetch_desc(&tmH2);
        }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], CG);                 // one arrive per producer of the pair (+ the transaction bytes)
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], EPI_WARPS * CG);   // every epilogue warp of the pair
        }
        for (int s = 0; s < 2 * EPI_WARPS; ++s) mbar_init(&h_bar[s], 1);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) tmem_alloc<CG>(tmem_ptr, TMEM_COLS);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if constexpr (KIND == K_DGRAD) {
        if (g.colsum != nullptr)
            for (int gi = 0; gi < g.groups; ++gi)
                for (int i = threadIdx.x; i < 4 * g.ld_out; i += NUM_THREADS) colsum_s[gi * GROUP_FLOATS + i] = 0.0f;
    }
    if constexpr (KIND == K_FWD || KIND == K_FWD_RELU) {   // the layer's bias vector (<= 512 entries) next to the epilogue warps
        for (int gi = 0; gi < g.groups; ++gi)
            for (int i = threadIdx.x; i < g.ld_out; i += NUM_THREADS) colsum_s[gi * GROUP_FLOATS + i] = __ldg((gi ? g.bias2 : g.bias) + i);
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CG == 2) cluster_sync_all();           // the partner's barriers are initialised before anything remote
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===================================== TMA producer (every CTA) =====================================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = cid; t < total_tiles; t += ncl) {
                const bool g2 = t >= group_tiles;
                const int tt = g2 ? t - group_tiles : t;
                const CUtensorMap* mA = g2 ? &tmA2 : &tmA;
                const CUtensorMap* mB = g2 ? &tmB2 : &tmB;
                const int nt = tt % g.n_tiles, mt = (tt / g.n_tiles) % g.m_tiles, sl = tt / (g.n_tiles * g.m_tiles);
                const int m0 = (mt * CG + rank) * BM;             // this CTA's accumulator rows
                const int n0 = nt * BN + rank * BNL;              // this CTA's share of the B tile
                const int kb0 = (KIND == K_WGRAD) ? static_cast<int>(static_cast<long long>(sl) * g.k_blocks / g.slices) : 0;
                const int kb1 = (KIND == K_WGRAD) ? static_cast<int>(static_cast<long long>(sl + 1) * g.k_blocks / g.slices) : g.k_blocks;
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    uint8_t* sb = sa + planes * A_BYTES;
                    if (rank == 0) mbar_expect_tx(&full_bar[stage], stage_bytes * CG);
#pragma unroll 1
                    for (int p = 0; p < planes; ++p) {
                        const int a_row = p ? g.a_lo_row : 0, b_row = p ? g.b_lo_row : 0;
                        uint8_t* da = sa + p * A_BYTES;
                        uint8_t* db = sb + p * B_BYTES;
                        if constexpr (KIND == K_FWD || KIND == K_FWD_RELU) {
                            tma_load_2d<CG>(mA, &full_bar[stage], da, kb * BK, a_row + m0);                         // X rows, K slice
                            tma_load_2d<CG>(mB, &full_bar[stage], db, kb * BK, b_row + n0);                         // W rows, K slice
                        } else if constexpr (KIND == K_DGRAD) {
                            tma_load_2d<CG>(mA, &full_bar[stage], da, kb * BK, a_row + m0);                         // dY rows, N slice
#pragma unroll
                            for (int j = 0; j < BNL / 64; ++j)                                                       // W rows = reduction
                                tma_load_2d<CG>(mB, &full_bar[stage], db + j * MN_BOX_BYTES, n0 + j * 64, b_row + kb * BK);
                        } else {
                            const int r0 = kb * BK;                                                                  // batch rows = reduction
#pragma unroll
                            for (int j = 0; j < BM / 64; ++j)
                                tma_load_2d<CG>(mA, &full_bar[stage], da + j * MN_BOX_BYTES, m0 + j * 64, a_row + r0);
#pragma unroll
                            for (int j = 0; j < BNL / 64; ++j)
                                tma_load_2d<CG>(mB, &full_bar[stage], db + j * MN_BOX_BYTES, n0 + j * 64, b_row + r0);
                        }
                    }
                    if (CG == 2 && rank != 0) mbar_arrive_leader(&full_bar[stage]);
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================================== MMA issuer (even CTA of a pair) ===============================
        if (lane == 0 && rank == 0) {
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int t = cid; t < total_tiles; t += ncl) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                int n_kb = g.k_blocks;
                if constexpr (KIND == K_WGRAD) {
                    const int sl = (t >= group_tiles ? t - group_tiles : t) / (g.n_tiles * g.m_tiles);
                    n_kb = static_cast<int>(static_cast<long long>(sl + 1) * g.k_blocks / g.slices) - static_cast<int>(static_cast<long long>(sl) * g.k_blocks / g.slices);
                }
                for (int kb = 0; kb < n_kb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * stage_bytes), sb = sa + planes * A_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / UK; ++k) {
                        const uint64_t a_hi = (KIND == K_WGRAD) ? desc_mnmajor(sa, k) : desc_kmajor(sa, k);
                        const uint64_t b_hi = (KIND == K_FWD || KIND == K_FWD_RELU) ? desc_kmajor(sb, k) : desc_mnmajor(sb, k);
                        umma_bf16<CG>(d_tmem, a_hi, b_hi, IDESC, (kb | k) != 0);
                        if (planes == 2) {
                            const uint64_t a_lo = (KIND == K_WGRAD) ? desc_mnmajor(sa + A_BYTES, k) : desc_kmajor(sa + A_BYTES, k);
                            const uint64_t b_lo = (KIND == K_FWD || KIND == K_FWD_RELU) ? desc_kmajor(sb + B_BYTES, k) : desc_mnmajor(sb + B_BYTES, k);
                            umma_bf16<CG>(d_tmem, a_hi, b_lo, IDESC, 1);
                            umma_bf16<CG>(d_tmem, a_lo, b_hi, IDESC, 1);
                        }
                    }
                    umma_commit<CG>(&empty_bar[stage]);      // frees the slot (in both CTAs) when these MMAs have read it
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
                umma_commit<CG>(&tfull_bar[acc]);            // accumulator complete -> epilogue (of both CTAs)
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
        __syncwarp();
    } else if (warp >= EPI_WARP0) {
        // ===================================== epilogue (every CTA: its own 128 accumulator rows) ============
        const int ew = warp - EPI_WARP0;
        const int q = warp & 3;                              // TMEM lane quadrant this warp may read
        const int half = ew >> 2;                            // which half of the BN columns
        constexpr int CHUNKS = (BN / 2) / 32;                // 32-column chunks per warp per tile
        uint8_t* ebuf = epi_base + ew * 2 * EPI_BUF_BYTES;   // two staging buffers
        uint64_t* hb = h_bar + 2 * ew;
        uint32_t hphase = 0;                                 // bit b: parity the next wait on buffer b expects
        const bool write_lo = planes == 2;
        int acc = 0;
        uint32_t acc_phase = 0;
        int item = 0;                                        // running chunk counter: buffer = item & 1

        // (t is the launch-wide tile index; tiles of the second problem start at group_tiles)
        auto local = [&](int t) { return t >= group_tiles ? t - group_tiles : t; };
        auto tile_rows = [&](int t) { return (((local(t) / g.n_tiles) % g.m_tiles) * CG + rank) * BM + q * 32; };
        auto tile_col = [&](int t, int ci) { return (local(t) % g.n_tiles) * BN + half * (BN / 2) + ci * 32; };
        auto load_h = [&](int t, int ci, int b) {            // lane 0: H chunk (hi, lo) -> staging buffer b
            const CUtensorMap* mH = t >= group_tiles ? &tmH2 : &tmH;
            mbar_expect_tx(&hb[b], write_lo ? 4096u : 2048u);
            tma_load_2d<1>(mH, &hb[b], ebuf + b * EPI_BUF_BYTES, tile_col(t, ci), tile_rows(t));
            if (write_lo) tma_load_2d<1>(mH, &hb[b], ebuf + b * EPI_BUF_BYTES + 2048, tile_col(t, ci), g.c_lo_row + tile_rows(t));
        };
        if constexpr (KIND == K_DGRAD) {
            if (lane == 0 && cid < total_tiles) load_h(cid, 0, 0);
        }
        for (int t = cid; t < total_tiles; t += ncl) {
            const bool g2 = t >= group_tiles;
            const int sl = local(t) / (g.n_tiles * g.m_tiles);
            const CUtensorMap* mC = g2 ? &tmC2 : &tmC;
            float* const gsm = colsum_s + (g2 ? GROUP_FLOATS : 0);       // this problem's bias vector / column-sum accumulator
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + half * (BN / 2);
            const int row0 = tile_rows(t);
            uint32_t cur[32], nxt[32];
            tmem_ld32_issue(t_row, cur);
#pragma unroll 1
            for (int ci = 0; ci < CHUNKS; ++ci, ++item) {
                const int b = item & 1;
                uint8_t* buf = ebuf + b * EPI_BUF_BYTES;
                const int col = tile_col(t, ci);
                tmem_ld_wait(cur);
                if (ci + 1 < CHUNKS) {
                    tmem_ld32_issue(t_row + (ci + 1) * 32, nxt);    // in flight while this chunk is worked on
                } else {
                    // the whole accumulator stage is in registers: hand it back to the MMA issuer before the last chunk's work
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if constexpr (CG == 1) mbar_arrive(&tempty_bar[acc]);
                        else mbar_arrive_leader(&tempty_bar[acc]);
                    }
                }
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(cur[j]);
                if constexpr (KIND == K_WGRAD) {
                    float4* dst = reinterpret_cast<float4*>((g2 ? g.partial2 : g.partial) + sl * g.slice_stride + static_cast<long long>(row0 + lane) * g.ld_partial + col);
#pragma unroll
                    for (int qd = 0; qd < 8; ++qd) dst[qd] = make_float4(v[4 * qd], v[4 * qd + 1], v[4 * qd + 2], v[4 * qd + 3]);
                } else {
                    if constexpr (KIND == K_FWD || KIND == K_FWD_RELU) {
                        const float4* sbias = reinterpret_cast<const float4*>(gsm + col);
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4) {
                            const float4 bb = sbias[j4];
                            v[4 * j4] += bb.x; v[4 * j4 + 1] += bb.y; v[4 * j4 + 2] += bb.z; v[4 * j4 + 3] += bb.w;
                        }
                        if constexpr (KIND == K_FWD_RELU) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
                        } else if (g.act) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = tanh_fast(v[j]);
                        }
                        // the store that last read this buffer was issued two chunks ago
                        if (lane == 0) bulk_wait_read<1>();
                        __syncwarp();
                    } else {
                        // H chunk of this item: landed (or landing) in this buffer
                        mbar_wait(&hb[b], (hphase >> b) & 1u);
                        hphase ^= 1u << b;
                        uint32_t hw[16], lw[16];
#pragma unroll
                        for (int qd = 0; qd < 4; ++qd) {
                            const uint4 u = *reinterpret_cast<const uint4*>(buf + stage_off(lane, qd));
                            hw[4 * qd] = u.x; hw[4 * qd + 1] = u.y; hw[4 * qd + 2] = u.z; hw[4 * qd + 3] = u.w;
                        }
                        if (write_lo) {
#pragma unroll
                            for (int qd = 0; qd < 4; ++qd) {
                                const uint4 u = *reinterpret_cast<const uint4*>(buf + 2048 + stage_off(lane, qd));
                                lw[4 * qd] = u.x; lw[4 * qd + 1] = u.y; lw[4 * qd + 2] = u.z; lw[4 * qd + 3] = u.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) lw[j] = 0u;
                        }
                        __syncwarp();                        // every lane has its H row in registers: the buffer is free
                        // next item's H chunk -> the other buffer (its last store, issued one chunk ago, must have been read)
                        if (lane == 0) {
                            int nt_ = t, nci = ci + 1;
                            if (nci == CHUNKS) { nci = 0; nt_ = t + ncl; }
                            if (nt_ < total_tiles) {
                                bulk_wait_read<0>();
                                load_h(nt_, nci, b ^ 1);
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float h0 = bf16lo_f(hw[j]) + bf16lo_f(lw[j]), h1 = bf16hi_f(hw[j]) + bf16hi_f(lw[j]);
                            v[2 * j] *= fmaf(-h0, h0, 1.0f);
                            v[2 * j + 1] *= fmaf(-h1, h1, 1.0f);
                        }
                    }
                    stage_split32(v, buf, lane, write_lo);
                    fence_proxy_async();                     // generic-proxy writes -> visible to the TMA (async proxy)
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_2d(mC, buf, col, row0);
                        if (write_lo) tma_store_2d(mC, buf + 2048, col, g.c_lo_row + row0);
                        bulk_commit();
                    }
                    if constexpr (KIND == K_DGRAD) {
                        if (g.colsum != nullptr) {
                            // column sums over the warp's 32 rows by a transposing butterfly (31 shuffles): afterwards lane j
                            // holds the sum of column col + j.  This warp is the only writer of (quadrant q, these columns).
#pragma unroll
                            for (int s = 16; s >= 1; s >>= 1) {
                                const bool up = (lane & s) != 0;
#pragma unroll
                                for (int j = 0; j < s; ++j) {
                                    const float send = up ? v[j] : v[j + s];
                                    const float keep = up ? v[j + s] : v[j];
                                    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, s);
                                }
                            }
                            gsm[q * g.ld_out + col + lane] += v[0];
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) cur[j] = nxt[j];
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (lane == 0) bulk_wait_all();                      // the staging buffers outlive their stores
        __syncwarp();
        if constexpr (KIND == K_DGRAD) {
            if (g.colsum != nullptr) {
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");       // epilogue warps only
                for (int gi = 0; gi < g.groups; ++gi) {
                    const float* cs = colsum_s + gi * GROUP_FLOATS;
                    float* dstc = gi ? g.colsum2 : g.colsum;
                    for (int c = threadIdx.x - EPI_WARP0 * 32; c < g.ld_out; c += EPI_WARPS * 32)
                        dstc[static_cast<long long>(blockIdx.x) * g.ld_out + c] = ((cs[c] + cs[g.ld_out + c]) + cs[2 * g.ld_out + c]) + cs[3 * g.ld_out + c];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CG == 2) cluster_sync_all();               // the partner may still be reading this CTA's shared memory / TMEM
    if (warp == 2) tmem_dealloc<CG>(tmem_base, TMEM_COLS);
}

}  // namespace dnmma
