// ppo_update.cu -- the PPO minibatch update (include/dnppo.h) and the SAC actor (include/dnsac.h) on sm_100a: tensor-map
// construction, launchers of the tcgen05 contraction kernel (dn_umma.cuh) and the CUDA-core kernels around it.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <string>
#include <vector>

#include "../../include/dnppo.h"
#include "../../include/dnsac.h"
#include "../../include/dronenav.h"
#include "dn_umma.cuh"
#include "ppo_kernels.cuh"
#include "ppo_comm.cuh"
#include "sac_kernels.cuh"

int dn_internal_fail(int code, const std::string& msg);   // dronenav.cu: sets the thread-local dn_last_error message

#define PPO_CUDA(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            return dn_internal_fail(DN_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));  \
    } while (0)

namespace {

using namespace dnmma;

// ---- cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda) ----------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// BF16 row-major [rows, cols] tensor maps (dn_umma.cuh):
//   MAP_KMAJOR   operand read along its rows: box = box_rows x BK (32) columns, 64-byte swizzle (one swizzle row per box row)
//   MAP_MNMAJOR  operand read across its rows: box = BK (32) rows x 64 columns, 128-byte swizzle
//   MAP_EPILOGUE results / tanh outputs: box = 32 x 32, 64-byte swizzle (the per-warp staging buffers)
enum MapKind { MAP_KMAJOR, MAP_MNMAJOR, MAP_EPILOGUE };
int make_map(CUtensorMap* m, const void* base, long long rows, long long cols, int box_rows, MapKind kind) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return dn_internal_fail(DN_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
    cuuint32_t box[2] = {kind == MAP_MNMAJOR ? 64u : 32u, static_cast<cuuint32_t>(kind == MAP_MNMAJOR ? BK : (kind == MAP_EPILOGUE ? 32 : box_rows))};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    kind == MAP_MNMAJOR ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return dn_internal_fail(DN_ECUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
    return DN_OK;
}

// Tile shape of a contraction whose accumulator is `rows` x `n`: CTA pairs (CG = 2, 256 x BN tiles) whenever the row count
// allows it, else single CTAs (128 x BN).
void pick_tile(int rows, int n, int* cg, int* bn) {
    *cg = (rows % 256 == 0 && n % 128 == 0) ? 2 : 1;
    if (*cg == 2) *bn = (n % 256 == 0) ? 256 : 128;
    else *bn = (n % 128 == 0) ? 128 : 64;
}

struct GemmPlan {       // one contraction, ready to launch
    int kind = 0, bn = 0, cg = 1, grid = 0;
    int tiles_n = 0;    // accumulator columns / bn
    CUtensorMap ma, mb, mc, mh;
    CUtensorMap ma2, mb2, mc2, mh2;   // second problem of a grouped launch (args.groups == 2)
    GemmArgs args;
};

// persistent grid: one CTA (pair) per SM (pair) of a device with `sms` SMs, never more than there are tiles
int grid_for(int tiles, int cg, int sms) { return std::max(1, std::min(tiles, sms / cg)) * cg; }

typedef void (*GemmKernel)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap,
                           GemmArgs);

// the instantiation of umma_gemm for a kind and tile shape; nullptr if there is none
GemmKernel gemm_kernel(int kind, int bn, int cg) {
#define DN_CASE(K, B, G) \
    if (kind == K && bn == B && cg == G) return umma_gemm<K, B, G>;
    DN_CASE(K_FWD, 256, 2) DN_CASE(K_FWD, 128, 2) DN_CASE(K_FWD, 128, 1) DN_CASE(K_FWD, 64, 1)
    DN_CASE(K_DGRAD, 256, 2) DN_CASE(K_DGRAD, 128, 2) DN_CASE(K_DGRAD, 128, 1) DN_CASE(K_DGRAD, 64, 1)
    DN_CASE(K_WGRAD, 256, 2) DN_CASE(K_WGRAD, 128, 2) DN_CASE(K_WGRAD, 128, 1) DN_CASE(K_WGRAD, 64, 1)
    DN_CASE(K_FWD_RELU, 256, 2) DN_CASE(K_FWD_RELU, 128, 2) DN_CASE(K_FWD_RELU, 128, 1) DN_CASE(K_FWD_RELU, 64, 1)
#undef DN_CASE
    return nullptr;
}

// umma_gemm needs more than the default 48 KB of dynamic shared memory.  That limit belongs to the function on the device that is
// current when it is set, so it is set on every device that launches the kernel: by each handle on its own device at create time,
// for every tile shape pick_tile can return.
int allow_gemm_smem(std::initializer_list<int> kinds) {
    const int tiles[4][2] = {{256, 2}, {128, 2}, {128, 1}, {64, 1}};
    for (int kind : kinds)
        for (const auto& t : tiles)
            PPO_CUDA(cudaFuncSetAttribute(gemm_kernel(kind, t[0], t[1]), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(SMEM_BYTES)));
    return DN_OK;
}

int launch_gemm(const GemmPlan& p, cudaStream_t st) {
    const GemmKernel kern = gemm_kernel(p.kind, p.bn, p.cg);
    if (!kern) return dn_internal_fail(DN_EINVAL, "launch_gemm: no such kernel instantiation");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = p.cg;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    // programmatic dependent launch: the kernel's set-up overlaps the tail of its predecessor in the stream (umma_gemm waits
    // with griddepcontrol.wait before its first global access)
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    if (p.args.groups == 2) PPO_CUDA(cudaLaunchKernelEx(&cfg, kern, p.ma, p.mb, p.mc, p.mh, p.ma2, p.mb2, p.mc2, p.mh2, p.args));
    else PPO_CUDA(cudaLaunchKernelEx(&cfg, kern, p.ma, p.mb, p.mc, p.mh, p.ma, p.mb, p.mc, p.mh, p.args));
    return DN_OK;
}

// Plans.  `*_planes` point at the hi plane; the lo plane starts `plane_rows * cols` elements later.  `rows_now` <= plane_rows
// is the number of rows the launch covers (tile counts); the tensor maps always span the whole planes.  `sms`: SMs of the
// device the plan launches on.
void set_grid(GemmPlan* p, int sms) {
    const GemmArgs& g = p->args;
    p->grid = grid_for(g.m_tiles * g.n_tiles * g.slices, p->cg, sms);
}
// forward: out[M,N] = act(A[M,K] W[N,K]^T + bias); act 0 identity, 1 tanh, 2 ReLU (the K_FWD_RELU instantiations)
int plan_fwd(GemmPlan* p, int sms, int passes, int M, int N, int K, const void* a, const void* w, const float* bias, int act, void* out,
             int rows_now = 0) {
    if (!rows_now) rows_now = M;
    if (M % BM || rows_now % BM || N % 64 || K % 64) return dn_internal_fail(DN_EINVAL, "mlp forward: M % 128, N % 64, K % 64 must be 0");
    p->kind = (act == 2) ? K_FWD_RELU : K_FWD;
    pick_tile(rows_now, N, &p->cg, &p->bn);
    int rc;
    if ((rc = make_map(&p->ma, a, 2LL * M, K, BM, MAP_KMAJOR)) || (rc = make_map(&p->mb, w, 2LL * N, K, p->bn / p->cg, MAP_KMAJOR)) ||
        (rc = make_map(&p->mc, out, 2LL * M, N, 32, MAP_EPILOGUE)))
        return rc;
    p->mh = p->mc;
    GemmArgs& g = p->args;
    memset(&g, 0, sizeof(g));
    g.m_tiles = rows_now / (BM * p->cg); g.n_tiles = N / p->bn; g.slices = 1; g.k_blocks = K / BK; g.passes = passes;
    g.a_lo_row = M; g.b_lo_row = N; g.c_lo_row = M; g.act = act; g.bias = bias; g.ld_out = N; g.groups = 1;
    set_grid(p, sms);
    return DN_OK;
}
// dgrad: out[M,N] = (A[M,K] W[K,N]) * (1 - H[M,N]^2)
int plan_dgrad(GemmPlan* p, int sms, int passes, int M, int N, int K, const void* a, const void* w, const void* h, void* out, int rows_now = 0) {
    if (!rows_now) rows_now = M;
    if (M % BM || rows_now % BM || N % 64 || K % 64) return dn_internal_fail(DN_EINVAL, "mlp dgrad: M % 128, N % 64, K % 64 must be 0");
    p->kind = K_DGRAD;
    pick_tile(rows_now, N, &p->cg, &p->bn);
    int rc;
    if ((rc = make_map(&p->ma, a, 2LL * M, K, BM, MAP_KMAJOR)) || (rc = make_map(&p->mb, w, 2LL * K, N, 0, MAP_MNMAJOR)) ||
        (rc = make_map(&p->mc, out, 2LL * M, N, 32, MAP_EPILOGUE)) || (rc = make_map(&p->mh, h, 2LL * M, N, 32, MAP_EPILOGUE)))
        return rc;
    GemmArgs& g = p->args;
    memset(&g, 0, sizeof(g));
    g.m_tiles = rows_now / (BM * p->cg); g.n_tiles = N / p->bn; g.slices = 1; g.k_blocks = K / BK; g.passes = passes;
    g.a_lo_row = M; g.b_lo_row = K; g.c_lo_row = M; g.ld_out = N; g.groups = 1;
    set_grid(p, sms);
    return DN_OK;
}
// wgrad: partial[s][Mo][No] = A[rows_s, Mo]^T B[rows_s, No], rows split into `slices`
int plan_wgrad(GemmPlan* p, int sms, int passes, int Mo, int No, int rows, int slices, const void* a, const void* b, float* partial, int rows_now = 0) {
    if (!rows_now) rows_now = rows;
    if (Mo % BM || No % 64 || slices < 1 || rows_now % 64 || rows_now / BK < slices)
        return dn_internal_fail(DN_EINVAL, "mlp wgrad: Mo % 128, No % 64, rows % 64 must be 0 and every slice needs at least one k-block");
    p->kind = K_WGRAD;
    pick_tile(Mo, No, &p->cg, &p->bn);
    int rc;
    if ((rc = make_map(&p->ma, a, 2LL * rows, Mo, 0, MAP_MNMAJOR)) || (rc = make_map(&p->mb, b, 2LL * rows, No, 0, MAP_MNMAJOR))) return rc;
    p->mc = p->ma;
    p->mh = p->ma;
    GemmArgs& g = p->args;
    memset(&g, 0, sizeof(g));
    g.m_tiles = Mo / (BM * p->cg); g.n_tiles = No / p->bn; g.slices = slices; g.k_blocks = rows_now / BK; g.passes = passes;
    g.a_lo_row = rows; g.b_lo_row = rows;
    g.partial = partial; g.ld_partial = No; g.slice_stride = static_cast<long long>(Mo) * No; g.groups = 1;
    set_grid(p, sms);
    return DN_OK;
}

// One launch for two problems of identical shape (layer l of the policy and of the value net): `out` = a's problem + b's.
// false if the two plans differ in anything but their pointers.
bool merge_plans(GemmPlan* out, const GemmPlan& a, const GemmPlan& b, int sms) {
    const GemmArgs &x = a.args, &y = b.args;
    if (a.kind != b.kind || a.bn != b.bn || a.cg != b.cg || x.m_tiles != y.m_tiles || x.n_tiles != y.n_tiles || x.slices != y.slices ||
        x.k_blocks != y.k_blocks || x.passes != y.passes || x.a_lo_row != y.a_lo_row || x.b_lo_row != y.b_lo_row || x.c_lo_row != y.c_lo_row ||
        x.act != y.act || x.ld_out != y.ld_out || x.ld_partial != y.ld_partial || x.slice_stride != y.slice_stride ||
        (x.colsum == nullptr) != (y.colsum == nullptr))
        return false;
    *out = a;
    out->ma2 = b.ma; out->mb2 = b.mb; out->mc2 = b.mc; out->mh2 = b.mh;
    out->args.groups = 2; out->args.bias2 = y.bias; out->args.partial2 = y.partial; out->args.colsum2 = y.colsum;
    out->grid = grid_for(2 * x.m_tiles * x.n_tiles * x.slices, a.cg, sms);
    return true;
}

// ====================================================================================================================
// the update handle
// ====================================================================================================================
using namespace dnppo;

struct Net {                      // one MLP (pi or vf)
    int L = 0;                    // hidden layers
    int n[MAX_LAYERS + 1] = {};   // n[0] = XPAD (padded observation), n[l] = width of hidden layer l
    long long w_off[MAX_LAYERS + 1] = {}, b_off[MAX_LAYERS + 1] = {};   // flat offsets; index L = head
    __nv_bfloat16* h[MAX_LAYERS + 1] = {};     // activation planes [2][max_rows][n[l]] (h[0] = shared observation planes)
    __nv_bfloat16* dz[MAX_LAYERS + 1] = {};    // pre-activation gradient planes
    __nv_bfloat16* w[MAX_LAYERS + 1] = {};     // weight planes [2][n[l]][n[l-1]]
    float* wpart[MAX_LAYERS + 1] = {};         // split-K partials of the weight gradient [slices][n[l]][n[l-1]]
    float* bpart[MAX_LAYERS + 1] = {};         // column-sum partials of the bias gradient [COLSUM_CHUNKS][n[l]]
    int slices_max[MAX_LAYERS + 1] = {};
    GemmPlan fwd[MAX_LAYERS + 1], dgrad[MAX_LAYERS + 1], wgrad[MAX_LAYERS + 1];
};

// What the PPO handle and the SAC actor share: the device, the observation planes the first layer reads, the table that
// refreshes the BF16 weight planes from the flat FP32 parameters, and the device allocations, which go with the handle.
struct MlpCore {
    int device = 0, passes = 3, sms = 148;
    int max_rows = 0, cur_rows = -1;   // cur_rows: the (padded) row count the forward plans were built for
    float* params = nullptr;
    __nv_bfloat16* x = nullptr;
    PlaneSeg* psegs_dev = nullptr; int* pseg_of_block_dev = nullptr; int plane_blocks = 0;
    std::vector<void*> allocs;
    ~MlpCore() {                        // the handle's device is current
        for (void* p : allocs) cudaFree(p);
        if (psegs_dev) cudaFree(psegs_dev);
        if (pseg_of_block_dev) cudaFree(pseg_of_block_dev);
    }
};

typedef void (*HeadKernel)(HeadArgs);
typedef void (*SacHeadKernel)(dnsac::SacHeadArgs);

}  // namespace

struct dn_ppo : MlpCore {
    dn_ppo_config cfg;
    float *grads = nullptr, *exp_avg = nullptr, *exp_avg_sq = nullptr, *step = nullptr;
    Net pi, vf;
    HeadKernel head[2] = {};        // head_kernel for this act_dim and width: [0] dn_ppo_forward / training, [1] sampling
    float *m_act = nullptr, *m_logp = nullptr, *m_val = nullptr, *m_adv = nullptr, *m_ret = nullptr;
    double *adv_partial = nullptr, *norm_partial = nullptr;
    float* head_partial = nullptr;
    int head_blocks_max = 0, head_psize = 0;
    size_t head_smem = 0;
    Ctrl* ctrl = nullptr;
    int* mirror = nullptr;          // pinned + mapped
    int* mirror_dev = nullptr;
    Seg* segs_dev = nullptr; int* seg_of_block_dev = nullptr; int n_segs = 0, reduce_blocks = 0;
    std::vector<Seg> segs_host;
    int table_rows = -1;
    // the policy and the value net have the same hidden widths (PBDroneSimulator.py:251-258): layer l of both runs as ONE launch
    // gradient all-reduce over NVLink peer memory (ppo_comm.cuh); comm_base == nullptr: not set up
    char* comm_base = nullptr;
    size_t comm_bytes = 0;
    dncomm::CommArgs comm;
    bool comm_connected = false;
    std::vector<void*> comm_opened;
    bool grouped = false;
    GemmPlan gfwd[MAX_LAYERS + 1], gdgrad[MAX_LAYERS + 1], gwgrad[MAX_LAYERS + 1];
};

// the SAC actor (include/dnsac.h): the latent ReLU layers on the forward contraction, then sac_head_kernel
struct dn_sac_actor : MlpCore {
    dn_sac_actor_config cfg;
    Net net;                          // h, w and fwd of the latent layers (the training buffers stay unallocated)
    SacHeadKernel head = nullptr;     // sac_head_kernel for this act_dim and width
    float *mu = nullptr, *log_std = nullptr;
};

namespace {

// split of the batch rows of a weight-gradient contraction: as many slices as it takes to give every CTA (pair) a work item
// (slices need not divide the rows: slice s covers k-blocks [s KB / S, (s + 1) KB / S) of the KB = rows / BK blocks), but every
// slice keeps at least 256 rows so that the partial-sum traffic stays small against the contraction
int wgrad_slices(int rows, int tiles, int units) {
    const int target = std::max(1, units / std::max(tiles, 1));
    return std::max(1, std::min(target, rows / 256));
}

template <typename T>
int dev_alloc(MlpCore* h, T** p, size_t count) {
    void* q = nullptr;
    PPO_CUDA(cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
    PPO_CUDA(cudaMemset(q, 0, std::max<size_t>(count, 1) * sizeof(T)));
    h->allocs.push_back(q);
    *p = static_cast<T*>(q);
    return DN_OK;
}

// Makes `device` current after checking that it exists and is an sm_100 part; *sms = its SM count.  `who` (the entry point) and
// `kernels` word the messages.
int open_device(const char* who, const char* kernels, int device, int* sms) {
    const std::string w(who);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return dn_internal_fail(DN_ECUDA, w + ": no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return dn_internal_fail(DN_EINVAL, w + ": bad device index");
    PPO_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    PPO_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return dn_internal_fail(DN_ECUDA, w + ": " + kernels + " are sm_100a only (tcgen05 / TMEM / TMA)");
    *sms = prop.multiProcessorCount;
    return DN_OK;
}

// the shared part of a new handle on the device open_device made current, with its observation planes [2][max_rows][XPAD]
int init_core(MlpCore* h, int device, int sms, int precision, int max_rows, float* params) {
    h->device = device;
    h->sms = sms;
    h->passes = (precision == DN_MLP_BF16X3) ? 3 : 1;
    h->max_rows = max_rows;
    h->params = params;
    return dev_alloc(h, &h->x, 2LL * max_rows * XPAD);
}

// tiles of the weight-gradient contraction of a layer [N, K] (accumulator N x K) and the CTAs (pairs) available for them
int wgrad_tiles(int N, int K, int sms, int* units) {
    int cg, bn;
    pick_tile(N, K, &cg, &bn);
    *units = sms / cg;
    return (N / (BM * cg)) * (K / bn);
}

// The hidden layers of one MLP: widths, flat offsets, activation and weight planes.  `train` adds the buffers of the backward
// pass: pre-activation gradient planes and the partials of the weight and bias gradients.
int setup_net(MlpCore* h, Net& net, int L, const int32_t* hidden, const int64_t* w_off, const int64_t* b_off, bool train) {
    net.L = L;
    net.n[0] = XPAD;
    net.h[0] = h->x;
    const long long R = h->max_rows;
    int rc;
    for (int l = 1; l <= L; ++l) {
        const int N = hidden[l - 1], K = net.n[l - 1];
        net.n[l] = N;
        net.w_off[l - 1] = w_off[l - 1];
        net.b_off[l - 1] = b_off[l - 1];
        if ((rc = dev_alloc(h, &net.h[l], 2 * R * N)) || (train && (rc = dev_alloc(h, &net.dz[l], 2 * R * N))) ||
            (rc = dev_alloc(h, &net.w[l], 2LL * N * K)))
            return rc;
        if (!train) continue;
        int units = 0;
        const int wt = wgrad_tiles(N, K, h->sms, &units);
        net.slices_max[l] = wgrad_slices(h->max_rows, wt, units);
        if ((rc = dev_alloc(h, &net.wpart[l], static_cast<size_t>(net.slices_max[l]) * N * K)) ||
            (rc = dev_alloc(h, &net.bpart[l], static_cast<size_t>(h->sms) * N)))
            return rc;
    }
    return DN_OK;
}

// Plans for `rows` rows: tensor maps over the full workspaces (lo plane max_rows rows after the hi plane), tile shapes and
// counts for this row count (CTA pairs need multiples of 256 rows).  plan_forward: the forward contractions of `net`, act 1 tanh
// (the PPO nets) or 2 ReLU (the SAC actor); build_plans adds the backward contractions of a PPO net.
int plan_forward(const MlpCore* h, Net& net, int rows, int act) {
    int rc;
    for (int l = 1; l <= net.L; ++l)
        if ((rc = plan_fwd(&net.fwd[l], h->sms, h->passes, h->max_rows, net.n[l], net.n[l - 1], net.h[l - 1], net.w[l],
                           h->params + net.b_off[l - 1], act, net.h[l], rows)))
            return rc;
    return DN_OK;
}

int build_plans(dn_ppo* h, Net& net, int rows, int groups) {
    int rc;
    if ((rc = plan_forward(h, net, rows, 1))) return rc;
    for (int l = 1; l <= net.L; ++l) {
        const int N = net.n[l], K = net.n[l - 1];
        if (l > 1) {
            if ((rc = plan_dgrad(&net.dgrad[l], h->sms, h->passes, h->max_rows, K, N, net.dz[l], net.w[l], net.h[l - 1], net.dz[l - 1], rows)))
                return rc;
            net.dgrad[l].args.colsum = net.bpart[l - 1];      // bias gradient of layer l-1 = column sums of dz[l-1], per CTA
        }
        int units = 0;
        const int wt = wgrad_tiles(N, K, h->sms, &units);
        const int slices = std::min(wgrad_slices(rows, wt * groups, units), net.slices_max[l]);   // one work item per CTA (pair) per launch
        if ((rc = plan_wgrad(&net.wgrad[l], h->sms, h->passes, N, K, h->max_rows, slices, net.dz[l], net.h[l - 1], net.wpart[l], rows)))
            return rc;
    }
    return DN_OK;
}

// reduction table: every parameter tensor <- its partials
void add_seg(std::vector<Seg>& v, const float* src, long long stride, int n_slices, int rows, int cols, int ld, long long dst) {
    Seg s;
    s.src = src; s.slice_stride = stride; s.dst_off = dst; s.n_slices = n_slices; s.rows = rows; s.cols = cols; s.ld = ld;
    s.first_block = 0; s.n_blocks = 0; s.deep = 0;
    v.push_back(s);
}

int build_reduce_table(dn_ppo* h, int rows) {
    std::vector<Seg>& v = h->segs_host;
    v.clear();
    const int A = h->cfg.act_dim, npi = h->pi.n[h->pi.L], nvf = h->vf.n[h->vf.L];
    const int head_blocks = std::min(std::max(rows / HEAD_WARPS, 1), h->head_blocks_max);
    Net* nets[2] = {&h->pi, &h->vf};
    for (Net* net : nets) {
        for (int l = 1; l <= net->L; ++l) {
            const int N = net->n[l], K = net->n[l - 1];
            const int cols = (l == 1) ? h->cfg.obs_dim : K;                         // the first layer's padding columns are dropped
            add_seg(v, net->wpart[l], static_cast<long long>(N) * K, net->wgrad[l].args.slices, N, cols, K, net->w_off[l - 1]);
            if (l < net->L)      // per-CTA column sums written by the dgrad launch that produced dz[l]; layer L: head kernel, below
                add_seg(v, net->bpart[l], N, net->dgrad[l + 1].grid, 1, N, N, net->b_off[l - 1]);
        }
    }
    const long long P = h->head_psize;
    const float* hp = h->head_partial;
    add_seg(v, hp, P, head_blocks, A, npi, npi, h->pi.w_off[h->pi.L]);
    add_seg(v, hp + A * npi, P, head_blocks, 1, A, A, h->pi.b_off[h->pi.L]);
    add_seg(v, hp + A * npi + A, P, head_blocks, 1, nvf, nvf, h->vf.w_off[h->vf.L]);
    add_seg(v, hp + A * npi + A + nvf, P, head_blocks, 1, 1, 1, h->vf.b_off[h->vf.L]);
    add_seg(v, hp + A * npi + A + nvf + 1, P, head_blocks, 1, A, A, h->cfg.log_std_off);
    add_seg(v, hp + A * npi + A + nvf + 1 + A, P, head_blocks, 1, npi, npi, h->pi.b_off[h->pi.L - 1]);
    add_seg(v, hp + A * npi + A + nvf + 1 + A + npi, P, head_blocks, 1, nvf, nvf, h->vf.b_off[h->vf.L - 1]);
    std::vector<int> sob;
    for (size_t i = 0; i < v.size(); ++i) {
        const long long count = static_cast<long long>(v[i].rows) * v[i].cols;
        v[i].first_block = static_cast<int>(sob.size());
        v[i].deep = v[i].n_slices >= REDUCE_DEEP_MIN_SLICES;
        const int per = v[i].deep ? REDUCE_DEEP_PER_BLOCK : REDUCE_PER_BLOCK;
        v[i].n_blocks = static_cast<int>((count + per - 1) / per);
        for (int b = 0; b < v[i].n_blocks; ++b) sob.push_back(static_cast<int>(i));
    }
    if (static_cast<int>(v.size()) > h->n_segs || static_cast<int>(sob.size()) > h->reduce_blocks) {
        if (h->segs_dev) { cudaFree(h->segs_dev); cudaFree(h->seg_of_block_dev); }
        PPO_CUDA(cudaMalloc(&h->segs_dev, v.size() * sizeof(Seg)));
        PPO_CUDA(cudaMalloc(&h->seg_of_block_dev, sob.size() * sizeof(int)));
    }
    h->n_segs = static_cast<int>(v.size());
    h->reduce_blocks = static_cast<int>(sob.size());
    // synchronous copies: this runs only when the minibatch size changes (never inside a captured graph)
    PPO_CUDA(cudaMemcpy(h->segs_dev, v.data(), v.size() * sizeof(Seg), cudaMemcpyHostToDevice));
    PPO_CUDA(cudaMemcpy(h->seg_of_block_dev, sob.data(), sob.size() * sizeof(int), cudaMemcpyHostToDevice));
    return DN_OK;
}

// the table planes_kernel walks: every hidden weight of `nets` -> its BF16 planes
int build_plane_table(MlpCore* h, const Net* const* nets, int n_nets, int obs_dim) {
    std::vector<PlaneSeg> v;
    std::vector<int> sob;
    for (int k = 0; k < n_nets; ++k) {
        const Net* net = nets[k];
        for (int l = 1; l <= net->L; ++l) {
            PlaneSeg s;
            s.param_off = net->w_off[l - 1]; s.rows = net->n[l]; s.ld = net->n[l - 1];
            s.cols = (l == 1) ? obs_dim : net->n[l - 1];
            s.planes = net->w[l];
            const long long count = static_cast<long long>(s.rows) * s.ld / 2;
            s.first_block = static_cast<int>(sob.size());
            s.n_blocks = static_cast<int>((count + 255) / 256);
            for (int b = 0; b < s.n_blocks; ++b) sob.push_back(static_cast<int>(v.size()));
            v.push_back(s);
        }
    }
    PPO_CUDA(cudaMalloc(&h->psegs_dev, v.size() * sizeof(PlaneSeg)));
    PPO_CUDA(cudaMalloc(&h->pseg_of_block_dev, sob.size() * sizeof(int)));
    PPO_CUDA(cudaMemcpy(h->psegs_dev, v.data(), v.size() * sizeof(PlaneSeg), cudaMemcpyHostToDevice));
    PPO_CUDA(cudaMemcpy(h->pseg_of_block_dev, sob.data(), sob.size() * sizeof(int), cudaMemcpyHostToDevice));
    h->plane_blocks = static_cast<int>(sob.size());
    return DN_OK;
}

// FP32 parameters -> the BF16 weight planes the contractions read
int refresh_planes(const MlpCore* h, cudaStream_t st) {
    planes_kernel<<<h->plane_blocks, 256, 0, st>>>(h->psegs_dev, h->pseg_of_block_dev, h->params, h->passes > 1);
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

int check_rows(const MlpCore* h, const char* who, int rows) {
    if (rows < 1 || rows > h->max_rows) return dn_internal_fail(DN_EINVAL, std::string(who) + ": rows must be within max_rows");
    return DN_OK;
}

// a drawing call's one step of the device draw counter (enqueued, so graph replays advance it too)
int advance_counter(void* counter, cudaStream_t st) {
    counter_advance_kernel<<<1, 32, 0, st>>>(static_cast<long long*>(counter));
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

// (re)plans the contractions for `rows` rows; the reduction table of the partial gradients only when training with a new row count
int ensure_rows(dn_ppo* h, int rows, bool train) {
    int rc;
    if (rows != h->cur_rows) {
        bool same = h->pi.L == h->vf.L;
        for (int l = 1; same && l <= h->pi.L; ++l) same = h->pi.n[l] == h->vf.n[l];
        if ((rc = build_plans(h, h->pi, rows, same ? 2 : 1)) || (rc = build_plans(h, h->vf, rows, same ? 2 : 1))) return rc;
        for (int l = 1; same && l <= h->pi.L; ++l) {
            same = merge_plans(&h->gfwd[l], h->pi.fwd[l], h->vf.fwd[l], h->sms) &&
                   merge_plans(&h->gwgrad[l], h->pi.wgrad[l], h->vf.wgrad[l], h->sms);
            if (same && l > 1) {
                same = merge_plans(&h->gdgrad[l], h->pi.dgrad[l], h->vf.dgrad[l], h->sms);
                // the reduction table sums one column-sum row per CTA of the launch that wrote them
                h->pi.dgrad[l].grid = h->vf.dgrad[l].grid = h->gdgrad[l].grid;
            }
        }
        if (!same && h->pi.L == h->vf.L) {
            // shapes differ after all: plans with per-net slice counts
            if ((rc = build_plans(h, h->pi, rows, 1)) || (rc = build_plans(h, h->vf, rows, 1))) return rc;
        }
        h->grouped = same;
        h->cur_rows = rows;                        // (the reduction table depends on the row count alone and is keyed by it below)
    }
    if (train && rows != h->table_rows) {
        if ((rc = build_reduce_table(h, rows))) return rc;
        h->table_rows = rows;
    }
    return DN_OK;
}

// f(NP) for the head kernels' NP = column pairs per lane = width / 64, rounded up to the instantiated 2, 4 or 8 (widths are
// multiples of 128, at most 512)
template <typename F>
auto with_np(int width, F&& f) {
    const int np = width / 64;
    if (np <= 2) return f(std::integral_constant<int, 2>());
    if (np <= 4) return f(std::integral_constant<int, 4>());
    return f(std::integral_constant<int, 8>());
}

// the PPO head for act_dim 1, 3 or 4 and the wider of the two last hidden layers; `sample`: dn_ppo_act's instantiation
HeadKernel ppo_head_for(int act_dim, int width, bool sample) {
    return with_np(width, [&](auto np) -> HeadKernel {
        constexpr int NP = decltype(np)::value;
        switch (act_dim) {
            case 1: return sample ? head_kernel<1, NP, true> : head_kernel<1, NP, false>;
            case 3: return sample ? head_kernel<3, NP, true> : head_kernel<3, NP, false>;
            case 4: return sample ? head_kernel<4, NP, true> : head_kernel<4, NP, false>;
            default: return nullptr;
        }
    });
}

// h->head: the two instantiations for this handle's act_dim and width, allowed the dynamic shared memory head_smem may take (at
// most 200 KB) on the handle's device
int setup_heads(dn_ppo* h, int width) {
    for (int s = 0; s < 2; ++s) {
        h->head[s] = ppo_head_for(h->cfg.act_dim, width, s);
        PPO_CUDA(cudaFuncSetAttribute(h->head[s], cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    return DN_OK;
}

// a.out_action set: the sampling instantiation (dn_ppo_act)
int run_head(dn_ppo* h, const HeadArgs& a, int blocks, cudaStream_t st) {
    h->head[a.out_action != nullptr]<<<blocks, HEAD_WARPS * 32, h->head_smem, st>>>(a);
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

// observation rows -> the padded BF16 planes `x` [2][max_rows][XPAD] the first layer reads
void gather_obs_args(GatherArgs& g, const MlpCore* h, const float* obs, int rows, int obs_dim) {
    memset(&g, 0, sizeof(g));
    g.obs = obs; g.rows = rows; g.obs_dim = obs_dim;
    g.x_hi = h->x; g.x_lo = (h->passes > 1) ? h->x + static_cast<long long>(h->max_rows) * XPAD : nullptr;
}
int launch_gather(const GatherArgs& g, cudaStream_t st) {
    const int blocks = (g.rows * 8 + 255) / 256;
    gather_kernel<<<blocks, 256, 0, st>>>(g);
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

int run_gather(dn_ppo* h, const float* obs, const dn_ppo_rollout* r, const long long* idx, int rows, bool train, cudaStream_t st) {
    GatherArgs g;
    gather_obs_args(g, h, obs, rows, h->cfg.obs_dim);
    g.idx = idx; g.act_dim = h->cfg.act_dim;
    if (train) {
        g.act = r->actions; g.logp = r->old_log_prob; g.val = r->old_values; g.adv = r->advantages; g.ret = r->returns;
        g.m_act = h->m_act; g.m_logp = h->m_logp; g.m_val = h->m_val; g.m_adv = h->m_adv; g.m_ret = h->m_ret;
        g.adv_partial = h->adv_partial;
    }
    return launch_gather(g, st);
}

int launch_forward(const Net& net, cudaStream_t st) {
    int rc;
    for (int l = 1; l <= net.L; ++l)
        if ((rc = launch_gemm(net.fwd[l], st))) return rc;
    return DN_OK;
}

int run_forward_chain(dn_ppo* h, cudaStream_t st) {
    int rc;
    if (h->grouped) {
        for (int l = 1; l <= h->pi.L; ++l)
            if ((rc = launch_gemm(h->gfwd[l], st))) return rc;
        return DN_OK;
    }
    if ((rc = launch_forward(h->pi, st))) return rc;
    return launch_forward(h->vf, st);
}

void fill_head_common(dn_ppo* h, HeadArgs& a, int rows) {
    memset(&a, 0, sizeof(a));
    const long long R = h->max_rows;
    const int npi = h->pi.n[h->pi.L], nvf = h->vf.n[h->vf.L];
    a.rows = rows; a.act_dim = h->cfg.act_dim; a.n_pi = npi; a.n_vf = nvf;
    a.hp_hi = h->pi.h[h->pi.L]; a.hp_lo = (h->passes > 1) ? a.hp_hi + R * npi : nullptr;
    a.hv_hi = h->vf.h[h->vf.L]; a.hv_lo = (h->passes > 1) ? a.hv_hi + R * nvf : nullptr;
    a.w_pi = h->params + h->pi.w_off[h->pi.L]; a.b_pi = h->params + h->pi.b_off[h->pi.L];
    a.w_vf = h->params + h->vf.w_off[h->vf.L]; a.b_vf = h->params + h->vf.b_off[h->vf.L];
    a.log_std = h->params + h->cfg.log_std_off;
    a.partial_size = h->head_psize;
}

// the BF16 plane pairs of `net` the buffer entry points expose: "h<l>", "w<l>" and, of a training net, "dz<l>"
bool find_planes(const MlpCore* h, const Net& net, const std::string& s, void** ptr, int64_t* elems) {
    const int l = s.empty() ? 0 : s.back() - '0';
    if (l < 1 || l > net.L) return false;
    const std::string kind = s.substr(0, s.size() - 1);
    const long long R = h->max_rows;
    if (kind == "h") { *ptr = net.h[l]; *elems = 2 * R * net.n[l]; }
    else if (kind == "w") { *ptr = net.w[l]; *elems = 2LL * net.n[l] * net.n[l - 1]; }
    else if (kind == "dz" && net.dz[l]) { *ptr = net.dz[l]; *elems = 2 * R * net.n[l]; }
    else return false;
    return true;
}

}  // namespace

extern "C" {

int dn_mlp_gemm(int kind, int passes, int M, int N, int K, int slices, const void* a, const void* b, const float* bias, int act,
                const void* h, void* out, float* partial, void* stream) {
    if (passes != 1 && passes != 3) return dn_internal_fail(DN_EINVAL, "dn_mlp_gemm: passes must be 1 or 3");
    if (!a || !b) return dn_internal_fail(DN_EINVAL, "dn_mlp_gemm: null operand");
    if (kind == 0 && (!bias || !out)) return dn_internal_fail(DN_EINVAL, "dn_mlp_gemm: forward needs bias and out");
    if (kind == 1 && (!h || !out)) return dn_internal_fail(DN_EINVAL, "dn_mlp_gemm: dgrad needs h and out");
    if (kind == 2 && !partial) return dn_internal_fail(DN_EINVAL, "dn_mlp_gemm: wgrad needs partial");
    if (kind < 0 || kind > 2) return dn_internal_fail(DN_EINVAL, "dn_mlp_gemm: kind must be 0, 1 or 2");
    // the contraction runs on the caller's current device: its SM count sizes the grid, and the kernel gets its shared memory there
    int dev = 0, sms = 0;
    PPO_CUDA(cudaGetDevice(&dev));
    PPO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GemmPlan p;
    int rc = (kind == 0) ? plan_fwd(&p, sms, passes, M, N, K, a, b, bias, act, out)
           : (kind == 1) ? plan_dgrad(&p, sms, passes, M, N, K, a, b, h, out)
                         : plan_wgrad(&p, sms, passes, M, N, K, slices, a, b, partial);
    if (rc || (rc = allow_gemm_smem({p.kind}))) return rc;
    return launch_gemm(p, static_cast<cudaStream_t>(stream));
}

int dn_ppo_create(const dn_ppo_config* cfg, int device, float* params, float* grads, float* exp_avg, float* exp_avg_sq, float* step,
                  dn_ppo** out) {
    if (!cfg || !out || !params || !grads || !exp_avg || !exp_avg_sq || !step) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: null argument");
    *out = nullptr;
    if (cfg->abi_version != DN_ABI_VERSION) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: abi_version mismatch");
    if (cfg->obs_dim < 1 || cfg->obs_dim > XPAD) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: obs_dim must be 1..64");
    if (cfg->act_dim != 1 && cfg->act_dim != 3 && cfg->act_dim != 4) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: act_dim must be 1, 3 or 4");
    if (cfg->max_rows < BM || cfg->max_rows % BM) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: max_rows must be a positive multiple of 128");
    if (cfg->n_pi < 1 || cfg->n_pi > MAX_LAYERS || cfg->n_vf < 1 || cfg->n_vf > MAX_LAYERS)
        return dn_internal_fail(DN_EINVAL, "dn_ppo_create: 1..4 hidden layers per network");
    for (int l = 0; l < cfg->n_pi; ++l)
        if (cfg->pi_hidden[l] < 128 || cfg->pi_hidden[l] % 128) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: hidden widths must be multiples of 128");
    for (int l = 0; l < cfg->n_vf; ++l)
        if (cfg->vf_hidden[l] < 128 || cfg->vf_hidden[l] % 128) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: hidden widths must be multiples of 128");
    for (int l = 0; l < cfg->n_pi; ++l)
        if (cfg->pi_hidden[l] > MAX_COLSUM_COLS) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: hidden widths may be at most 512");
    for (int l = 0; l < cfg->n_vf; ++l)
        if (cfg->vf_hidden[l] > MAX_COLSUM_COLS) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: hidden widths may be at most 512");
    if (cfg->pi_hidden[cfg->n_pi - 1] > MAX_HEAD_COLS || cfg->vf_hidden[cfg->n_vf - 1] > MAX_HEAD_COLS)
        return dn_internal_fail(DN_EINVAL, "dn_ppo_create: the last hidden layer may be at most 512 wide");
    if (cfg->precision != DN_MLP_BF16X3 && cfg->precision != DN_MLP_BF16) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: unknown precision");
    if (cfg->world_size < 1) return dn_internal_fail(DN_EINVAL, "dn_ppo_create: world_size must be >= 1");
    int sms = 0, rc;
    if ((rc = open_device("dn_ppo_create", "the update kernels", device, &sms))) return rc;

    dn_ppo* h = new dn_ppo();
    auto bail = [&](int code) { dn_ppo_destroy(h); return code; };
    h->cfg = *cfg;
    h->grads = grads; h->exp_avg = exp_avg; h->exp_avg_sq = exp_avg_sq; h->step = step;
    const long long R = cfg->max_rows;
    const int A = cfg->act_dim;
    if ((rc = init_core(h, device, sms, cfg->precision, cfg->max_rows, params))) return bail(rc);
    if ((rc = setup_net(h, h->pi, cfg->n_pi, cfg->pi_hidden, cfg->pi_w_off, cfg->pi_b_off, true))) return bail(rc);
    if ((rc = setup_net(h, h->vf, cfg->n_vf, cfg->vf_hidden, cfg->vf_w_off, cfg->vf_b_off, true))) return bail(rc);
    h->pi.w_off[cfg->n_pi] = cfg->pi_w_off[cfg->n_pi]; h->pi.b_off[cfg->n_pi] = cfg->pi_b_off[cfg->n_pi];    // index L: the heads
    h->vf.w_off[cfg->n_vf] = cfg->vf_w_off[cfg->n_vf]; h->vf.b_off[cfg->n_vf] = cfg->vf_b_off[cfg->n_vf];
    if ((rc = dev_alloc(h, &h->m_act, R * A)) || (rc = dev_alloc(h, &h->m_logp, R)) || (rc = dev_alloc(h, &h->m_val, R)) ||
        (rc = dev_alloc(h, &h->m_adv, R)) || (rc = dev_alloc(h, &h->m_ret, R)))
        return bail(rc);
    if ((rc = dev_alloc(h, &h->adv_partial, 2 * ((R * 8 + 255) / 256))) || (rc = dev_alloc(h, &h->norm_partial, NORM_BLOCKS))) return bail(rc);
    const int npi = h->pi.n[h->pi.L], nvf = h->vf.n[h->vf.L];
    h->head_psize = head_partial_size(A, npi, nvf);
    h->head_blocks_max = 3 * h->sms;
    h->head_smem = static_cast<size_t>(A * npi + nvf + HEAD_WARPS * h->head_psize) * sizeof(float);
    if (h->head_smem > 200 * 1024) return bail(dn_internal_fail(DN_EINVAL, "dn_ppo_create: head kernel shared memory exceeds 200 KB"));
    if ((rc = dev_alloc(h, &h->head_partial, static_cast<size_t>(h->head_blocks_max) * h->head_psize))) return bail(rc);
    if ((rc = dev_alloc(h, &h->ctrl, 1))) return bail(rc);
    {
        void* m = nullptr;
        cudaError_t e = cudaHostAlloc(&m, 4 * sizeof(int), cudaHostAllocMapped);
        if (e != cudaSuccess) return bail(dn_internal_fail(DN_ECUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)));
        h->mirror = static_cast<int*>(m);
        memset(h->mirror, 0, 4 * sizeof(int));
        void* d = nullptr;
        e = cudaHostGetDevicePointer(&d, m, 0);
        if (e != cudaSuccess) return bail(dn_internal_fail(DN_ECUDA, std::string("cudaHostGetDevicePointer: ") + cudaGetErrorString(e)));
        h->mirror_dev = static_cast<int*>(d);
    }
    {
        const Net* nets[2] = {&h->pi, &h->vf};
        if ((rc = build_plane_table(h, nets, 2, cfg->obs_dim))) return bail(rc);
    }
    if ((rc = allow_gemm_smem({K_FWD, K_DGRAD, K_WGRAD})) || (rc = setup_heads(h, std::max(npi, nvf)))) return bail(rc);
    if ((rc = ensure_rows(h, h->max_rows, true))) return bail(rc);
    if ((rc = dn_ppo_sync_weights(h, nullptr))) return bail(rc);
    PPO_CUDA(cudaStreamSynchronize(nullptr));
    *out = h;
    return DN_OK;
}

int dn_ppo_destroy(dn_ppo* h) {
    if (!h) return DN_OK;
    cudaSetDevice(h->device);
    for (void* p : h->comm_opened) cudaIpcCloseMemHandle(p);
    if (h->comm_base) cudaFree(h->comm_base);
    if (h->mirror) cudaFreeHost(h->mirror);
    if (h->segs_dev) cudaFree(h->segs_dev);
    if (h->seg_of_block_dev) cudaFree(h->seg_of_block_dev);
    delete h;
    return DN_OK;
}

// ---- gradient all-reduce over peer memory (ppo_comm.cuh) ----
int dn_ppo_comm_create(dn_ppo* h, int32_t rank, int32_t world, unsigned char* handle_out) {
    if (!h || !handle_out) return dn_internal_fail(DN_EINVAL, "dn_ppo_comm_create: null argument");
    if (world < 2 || world > dncomm::MAX_RANKS || rank < 0 || rank >= world)
        return dn_internal_fail(DN_EINVAL, "dn_ppo_comm_create: world must be 2..16 and 0 <= rank < world");
    if (h->comm_base) return dn_internal_fail(DN_EINVAL, "dn_ppo_comm_create: already created");
    static_assert(sizeof(cudaIpcMemHandle_t) == DN_PPO_COMM_HANDLE_BYTES, "IPC handle size");
    cudaSetDevice(h->device);
    const long long n = h->cfg.n_params + 1, q = 4ll * world;
    const long long n_pad = (n + q - 1) / q * q;
    h->comm_bytes = dncomm::FLAG_BYTES + 2 * static_cast<size_t>(n_pad) * sizeof(float) + 256;
    PPO_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->comm_base), h->comm_bytes));
    PPO_CUDA(cudaMemset(h->comm_base, 0, h->comm_bytes));
    memset(&h->comm, 0, sizeof(h->comm));
    h->comm.grads = h->grads; h->comm.n = n; h->comm.n_pad = n_pad; h->comm.rank = rank; h->comm.world = world;
    // the epoch word and the CTA counter live behind the buffers (never touched by peers)
    char* tail = h->comm_base + dncomm::FLAG_BYTES + 2 * static_cast<size_t>(n_pad) * sizeof(float);
    h->comm.epoch = reinterpret_cast<uint32_t*>(tail);
    h->comm.counter = reinterpret_cast<unsigned int*>(tail + 64);
    h->comm.peer[rank] = h->comm_base;
    cudaIpcMemHandle_t mh;
    PPO_CUDA(cudaIpcGetMemHandle(&mh, h->comm_base));
    memcpy(handle_out, &mh, sizeof(mh));
    PPO_CUDA(cudaDeviceSynchronize());
    return DN_OK;
}

int dn_ppo_comm_connect(dn_ppo* h, const unsigned char* handles) {
    if (!h || !handles) return dn_internal_fail(DN_EINVAL, "dn_ppo_comm_connect: null argument");
    if (!h->comm_base) return dn_internal_fail(DN_EINVAL, "dn_ppo_comm_connect: dn_ppo_comm_create first");
    if (h->comm_connected) return DN_OK;
    cudaSetDevice(h->device);
    for (int p = 0; p < h->comm.world; ++p) {
        if (p == h->comm.rank) continue;
        cudaIpcMemHandle_t mh;
        memcpy(&mh, handles + static_cast<size_t>(p) * DN_PPO_COMM_HANDLE_BYTES, sizeof(mh));
        void* ptr = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return dn_internal_fail(DN_ECUDA, std::string("dn_ppo_comm_connect: cudaIpcOpenMemHandle (peer-to-peer over NVLink / PCIe is required): ") +
                                                  cudaGetErrorString(e));
        }
        h->comm_opened.push_back(ptr);
        h->comm.peer[p] = static_cast<char*>(ptr);
    }
    h->comm_connected = true;
    return DN_OK;
}

int dn_ppo_allreduce(dn_ppo* h, void* stream) {
    if (!h) return dn_internal_fail(DN_EINVAL, "dn_ppo_allreduce: null handle");
    if (!h->comm_connected) return dn_internal_fail(DN_EINVAL, "dn_ppo_allreduce: dn_ppo_comm_create + dn_ppo_comm_connect first");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const dncomm::CommArgs& a = h->comm;
    const int T = dncomm::AR_THREADS;
    const int blocks = static_cast<int>(std::max<long long>(1, std::min<long long>((a.n_pad / 4 + T - 1) / T, h->sms)));   // all resident
    dncomm::allreduce_kernel<<<blocks, T, 0, st>>>(a);
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

int dn_ppo_sync_weights(dn_ppo* h, void* stream) {
    if (!h) return dn_internal_fail(DN_EINVAL, "dn_ppo_sync_weights: null handle");
    return refresh_planes(h, static_cast<cudaStream_t>(stream));
}

int dn_ppo_begin_update(dn_ppo* h, void* stream) {
    if (!h) return dn_internal_fail(DN_EINVAL, "dn_ppo_begin_update: null handle");
    PPO_CUDA(cudaMemsetAsync(h->ctrl, 0, sizeof(Ctrl), static_cast<cudaStream_t>(stream)));
    h->mirror[0] = h->mirror[1] = h->mirror[2] = 0;
    return DN_OK;
}

int dn_ppo_minibatch_grad(dn_ppo* h, const dn_ppo_rollout* r, const int64_t* idx, int32_t rows, void* stream) {
    if (!h || !r || !idx) return dn_internal_fail(DN_EINVAL, "dn_ppo_minibatch_grad: null argument");
    if (rows < BM || rows % BM || rows > h->max_rows) return dn_internal_fail(DN_EINVAL, "dn_ppo_minibatch_grad: rows must be a multiple of 128 within max_rows");
    if (!r->obs || !r->actions || !r->old_log_prob || !r->old_values || !r->advantages || !r->returns)
        return dn_internal_fail(DN_EINVAL, "dn_ppo_minibatch_grad: null rollout array");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc;
    if ((rc = ensure_rows(h, rows, true))) return rc;
    if ((rc = run_gather(h, r->obs, r, reinterpret_cast<const long long*>(idx), rows, true, st))) return rc;
    if ((rc = run_forward_chain(h, st))) return rc;
    // heads, losses, gradients w.r.t. the last hidden pre-activations
    const long long R = h->max_rows;
    const int npi = h->pi.n[h->pi.L], nvf = h->vf.n[h->vf.L];
    const int head_blocks = std::min(std::max(rows / HEAD_WARPS, 1), h->head_blocks_max);
    HeadArgs a;
    fill_head_common(h, a, rows);
    a.train = 1;
    a.m_act = h->m_act; a.m_logp = h->m_logp; a.m_val = h->m_val; a.m_adv = h->m_adv; a.m_ret = h->m_ret;
    a.adv_partial = h->adv_partial; a.adv_blocks = (rows * 8 + 255) / 256;
    a.normalize_adv = h->cfg.normalize_advantage && rows > 1;
    a.clip_range = h->cfg.clip_range; a.clip_range_vf = h->cfg.clip_range_vf; a.vf_coef = h->cfg.vf_coef;
    a.dzp_hi = h->pi.dz[h->pi.L]; a.dzp_lo = (h->passes > 1) ? a.dzp_hi + R * npi : nullptr;
    a.dzv_hi = h->vf.dz[h->vf.L]; a.dzv_lo = (h->passes > 1) ? a.dzv_hi + R * nvf : nullptr;
    a.partial = h->head_partial;
    if ((rc = run_head(h, a, head_blocks, st))) return rc;
    // backward through the hidden layers
    // bias gradients ride along: layer L's in the head kernel, layer l-1's in the epilogue of the dgrad of layer l
    if (h->grouped) {
        for (int l = h->pi.L; l >= 1; --l) {
            if ((rc = launch_gemm(h->gwgrad[l], st))) return rc;
            if (l > 1 && (rc = launch_gemm(h->gdgrad[l], st))) return rc;
        }
    } else {
        Net* nets[2] = {&h->pi, &h->vf};
        for (Net* net : nets)
            for (int l = net->L; l >= 1; --l) {
                if ((rc = launch_gemm(net->wgrad[l], st))) return rc;
                if (l > 1 && (rc = launch_gemm(net->dgrad[l], st))) return rc;
            }
    }
    // every partial -> the flat bucket; statistics; early-stop vote
    ReduceArgs ra;
    memset(&ra, 0, sizeof(ra));
    ra.segs = h->segs_dev; ra.n_segs = h->n_segs; ra.seg_of_block = h->seg_of_block_dev;
    ra.grads = h->grads; ra.n_params = h->cfg.n_params;
    ra.head_partial = h->head_partial; ra.head_blocks = head_blocks; ra.head_psize = h->head_psize;
    ra.head_stats_off = h->head_psize - 4;
    ra.ent_coef = h->cfg.ent_coef; ra.act_dim = h->cfg.act_dim; ra.log_std_off = h->cfg.log_std_off;
    ra.kl_limit = (h->cfg.target_kl >= 0.0f) ? 1.5f * h->cfg.target_kl : -1.0f;
    ra.rows = rows; ra.ctrl = h->ctrl;
    reduce_kernel<<<h->reduce_blocks + 1, 256, 0, st>>>(ra);
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

int dn_ppo_minibatch_apply(dn_ppo* h, void* stream) {
    if (!h) return dn_internal_fail(DN_EINVAL, "dn_ppo_minibatch_apply: null handle");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n = h->cfg.n_params;
    norm_kernel<<<NORM_BLOCKS, 256, 0, st>>>(h->grads, n, h->norm_partial);
    PPO_CUDA(cudaGetLastError());
    AdamArgs a;
    a.params = h->params; a.grads = h->grads; a.exp_avg = h->exp_avg; a.exp_avg_sq = h->exp_avg_sq; a.step = h->step; a.n = n;
    a.norm_partial = h->norm_partial;
    a.lr = h->cfg.learning_rate; a.beta1 = h->cfg.beta1; a.beta2 = h->cfg.beta2; a.eps = h->cfg.adam_eps;
    a.max_grad_norm = h->cfg.max_grad_norm; a.inv_world = 1.0f / static_cast<float>(h->cfg.world_size);
    a.ctrl = h->ctrl;
    adam_kernel<<<std::min<long long>((n + 255) / 256, 4 * h->sms), 256, 0, st>>>(a);
    PPO_CUDA(cudaGetLastError());
    // the planes are refreshed unconditionally (a stopped step leaves the parameters, hence the planes, unchanged)
    int rc;
    if ((rc = refresh_planes(h, st))) return rc;
    ctrl_commit_kernel<<<1, 32, 0, st>>>(h->ctrl, h->grads, n, h->step, h->norm_partial, a.inv_world, h->mirror_dev);
    PPO_CUDA(cudaGetLastError());
    return DN_OK;
}

int dn_ppo_get_stats(dn_ppo* h, dn_ppo_stats* out, void* stream) {
    if (!h || !out) return dn_internal_fail(DN_EINVAL, "dn_ppo_get_stats: null argument");
    Ctrl c;
    PPO_CUDA(cudaMemcpyAsync(&c, h->ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
    PPO_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    const double inv = 1.0 / std::max(c.n_done, 1);
    out->policy_gradient_loss = c.stats[0] * inv; out->value_loss = c.stats[1] * inv;
    out->approx_kl = c.stats[2] * inv; out->clip_fraction = c.stats[3] * inv;
    out->minibatches = c.n_done; out->optimizer_steps = c.n_applied; out->early_stop = c.stopped;
    out->last_approx_kl = c.last_kl; out->last_grad_norm = c.last_norm;
    return DN_OK;
}

int dn_ppo_poll(dn_ppo* h, int32_t* early_stop, int32_t* minibatches, int32_t* optimizer_steps) {
    if (!h) return dn_internal_fail(DN_EINVAL, "dn_ppo_poll: null handle");
    volatile int* m = h->mirror;
    if (early_stop) *early_stop = m[0];
    if (minibatches) *minibatches = m[1];
    if (optimizer_steps) *optimizer_steps = m[2];
    return DN_OK;
}

int dn_ppo_forward(dn_ppo* h, const float* obs, int32_t rows, float* mean, float* value, void* stream) {
    if (!h || !obs || !mean || !value) return dn_internal_fail(DN_EINVAL, "dn_ppo_forward: null argument");
    int rc;
    if ((rc = check_rows(h, "dn_ppo_forward", rows))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rows_pad = (rows + BM - 1) / BM * BM;
    if ((rc = ensure_rows(h, rows_pad, false))) return rc;
    if ((rc = run_gather(h, obs, nullptr, nullptr, rows, false, st))) return rc;
    if ((rc = run_forward_chain(h, st))) return rc;
    HeadArgs a;
    fill_head_common(h, a, rows);
    a.train = 0; a.out_mean = mean; a.out_value = value;
    const int head_blocks = std::min(std::max((rows + HEAD_WARPS - 1) / HEAD_WARPS, 1), h->head_blocks_max);
    return run_head(h, a, head_blocks, st);
}

int dn_ppo_act(dn_ppo* h, const float* obs, int32_t rows, const dn_ppo_sample* s, float* action, float* clipped_action, float* log_prob,
               float* value, void* stream) {
    if (!h || !obs || !s || !action || !log_prob || !value) return dn_internal_fail(DN_EINVAL, "dn_ppo_act: null argument");
    if (s->deterministic != 0 && s->deterministic != 1) return dn_internal_fail(DN_EINVAL, "dn_ppo_act: deterministic must be 0 or 1");
    if (!s->deterministic && !s->counter) return dn_internal_fail(DN_EINVAL, "dn_ppo_act: a sampling call needs the device counter (null counter)");
    if (s->row_id_offset < 0) return dn_internal_fail(DN_EINVAL, "dn_ppo_act: row_id_offset must be >= 0");
    if (!(s->low <= s->high)) return dn_internal_fail(DN_EINVAL, "dn_ppo_act: low must not exceed high (and neither may be NaN)");
    int rc;
    if ((rc = check_rows(h, "dn_ppo_act", rows))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rows_pad = (rows + BM - 1) / BM * BM;
    if ((rc = ensure_rows(h, rows_pad, false))) return rc;
    if ((rc = run_gather(h, obs, nullptr, nullptr, rows, false, st))) return rc;
    if ((rc = run_forward_chain(h, st))) return rc;
    HeadArgs a;
    fill_head_common(h, a, rows);
    a.train = 0; a.out_value = value;
    a.out_action = action; a.out_clipped = clipped_action; a.out_logp = log_prob;
    a.counter = s->deterministic ? nullptr : reinterpret_cast<const long long*>(s->counter);
    a.seed = s->seed; a.row_id_offset = s->row_id_offset; a.low = s->low; a.high = s->high;
    const int head_blocks = std::min(std::max((rows + HEAD_WARPS - 1) / HEAD_WARPS, 1), h->head_blocks_max);
    if ((rc = run_head(h, a, head_blocks, st))) return rc;
    return s->deterministic ? DN_OK : advance_counter(s->counter, st);
}

int dn_ppo_buffer(dn_ppo* h, const char* name, void** ptr, int64_t* elems) {
    if (!h || !name || !ptr || !elems) return dn_internal_fail(DN_EINVAL, "dn_ppo_buffer: null argument");
    const std::string s(name);
    if (s == "x") { *ptr = h->x; *elems = 2LL * h->max_rows * XPAD; return DN_OK; }
    const bool pi = s.compare(0, 3, "pi.") == 0, vf = s.compare(0, 3, "vf.") == 0;
    if ((pi || vf) && find_planes(h, pi ? h->pi : h->vf, s.substr(3), ptr, elems)) return DN_OK;
    return dn_internal_fail(DN_EINVAL, "dn_ppo_buffer: unknown buffer name");
}

}  // extern "C"

// ---- the SAC actor (include/dnsac.h) ----
namespace {

int sac_check_config(const dn_sac_actor_config* c) {
    if (c->abi_version != DN_ABI_VERSION) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: abi_version mismatch");
    if (c->obs_dim < 1 || c->obs_dim > XPAD) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: obs_dim must be 1..64");
    if (c->act_dim < 1 || c->act_dim > 4) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: act_dim must be 1..4");
    if (c->max_rows < BM || c->max_rows % BM) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: max_rows must be a positive multiple of 128");
    if (c->n_hidden < 1 || c->n_hidden > DN_SAC_MAX_LAYERS) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: 1..4 hidden layers");
    for (int l = 0; l < c->n_hidden; ++l)
        if (c->hidden[l] < 128 || c->hidden[l] > 512 || c->hidden[l] % 128)
            return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: hidden widths must be multiples of 128 between 128 and 512");
    if (c->precision != DN_MLP_BF16X3 && c->precision != DN_MLP_BF16) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: unknown precision");
    const long long A = c->act_dim, last = c->hidden[c->n_hidden - 1];
    auto inside = [&](long long off, long long count) { return off >= 0 && count <= c->n_params && off <= c->n_params - count; };
    bool ok = c->n_params > 0;
    for (int l = 0; l < c->n_hidden; ++l) {
        const long long in = l ? c->hidden[l - 1] : c->obs_dim;
        ok = ok && inside(c->w_off[l], c->hidden[l] * in) && inside(c->b_off[l], c->hidden[l]);
    }
    ok = ok && inside(c->mu_w_off, A * last) && inside(c->mu_b_off, A) && inside(c->log_std_w_off, A * last) && inside(c->log_std_b_off, A);
    if (!ok) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: a parameter tensor lies outside [0, n_params)");
    return DN_OK;
}

int sac_ensure_rows(dn_sac_actor* h, int rows_pad) {
    if (rows_pad == h->cur_rows) return DN_OK;
    int rc;
    if ((rc = plan_forward(h, h->net, rows_pad, 2))) return rc;
    h->cur_rows = rows_pad;
    return DN_OK;
}

// the SAC head for act_dim 1..4 and the last hidden width
SacHeadKernel sac_head_for(int act_dim, int width) {
    return with_np(width, [&](auto np) -> SacHeadKernel {
        constexpr int NP = decltype(np)::value;
        switch (act_dim) {
            case 1: return dnsac::sac_head_kernel<1, NP>;
            case 2: return dnsac::sac_head_kernel<2, NP>;
            case 3: return dnsac::sac_head_kernel<3, NP>;
            case 4: return dnsac::sac_head_kernel<4, NP>;
            default: return nullptr;
        }
    });
}

}  // namespace

extern "C" {

int dn_sac_actor_create(const dn_sac_actor_config* cfg, int device, const float* params, dn_sac_actor** out) {
    if (!cfg || !params || !out) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_create: null argument");
    *out = nullptr;
    int rc;
    if ((rc = sac_check_config(cfg))) return rc;
    int sms = 0;
    if ((rc = open_device("dn_sac_actor_create", "the kernels", device, &sms))) return rc;

    dn_sac_actor* h = new dn_sac_actor();
    auto bail = [&](int code) { dn_sac_actor_destroy(h); return code; };
    h->cfg = *cfg;
    h->head = sac_head_for(cfg->act_dim, cfg->hidden[cfg->n_hidden - 1]);
    const long long R = cfg->max_rows;
    // (the actor only reads the parameters)
    if ((rc = init_core(h, device, sms, cfg->precision, cfg->max_rows, const_cast<float*>(params))) ||
        (rc = setup_net(h, h->net, cfg->n_hidden, cfg->hidden, cfg->w_off, cfg->b_off, false)))
        return bail(rc);
    if ((rc = dev_alloc(h, &h->mu, R * cfg->act_dim)) || (rc = dev_alloc(h, &h->log_std, R * cfg->act_dim))) return bail(rc);
    const Net* nets[1] = {&h->net};
    if ((rc = build_plane_table(h, nets, 1, cfg->obs_dim))) return bail(rc);
    if ((rc = allow_gemm_smem({K_FWD_RELU}))) return bail(rc);
    if ((rc = sac_ensure_rows(h, h->max_rows))) return bail(rc);
    if ((rc = dn_sac_actor_sync_weights(h, nullptr))) return bail(rc);
    PPO_CUDA(cudaStreamSynchronize(nullptr));
    *out = h;
    return DN_OK;
}

int dn_sac_actor_destroy(dn_sac_actor* h) {
    if (!h) return DN_OK;
    cudaSetDevice(h->device);
    delete h;
    return DN_OK;
}

int dn_sac_actor_sync_weights(dn_sac_actor* h, void* stream) {
    if (!h) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_sync_weights: null handle");
    return refresh_planes(h, static_cast<cudaStream_t>(stream));
}

int dn_sac_act(dn_sac_actor* h, const float* obs, int32_t rows, const dn_sac_sample* s, float* action, float* log_prob, void* stream) {
    if (!h || !obs || !s || !action) return dn_internal_fail(DN_EINVAL, "dn_sac_act: null argument");
    if (s->mode != DN_SAC_SAMPLE && s->mode != DN_SAC_DETERMINISTIC && s->mode != DN_SAC_UNIFORM)
        return dn_internal_fail(DN_EINVAL, "dn_sac_act: mode must be DN_SAC_SAMPLE, DN_SAC_DETERMINISTIC or DN_SAC_UNIFORM");
    if (s->mode != DN_SAC_DETERMINISTIC && !s->counter) return dn_internal_fail(DN_EINVAL, "dn_sac_act: a drawing call needs the device counter (null counter)");
    if (s->row_id_offset < 0) return dn_internal_fail(DN_EINVAL, "dn_sac_act: row_id_offset must be >= 0");
    int rc;
    if ((rc = check_rows(h, "dn_sac_act", rows))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long* counter = reinterpret_cast<const long long*>(s->counter);
    if (s->mode == DN_SAC_UNIFORM) {
        dnsac::sac_uniform_kernel<<<(rows + 255) / 256, 256, 0, st>>>(rows, h->cfg.act_dim, counter, s->seed, s->row_id_offset, action, log_prob);
        PPO_CUDA(cudaGetLastError());
    } else {
        if ((rc = sac_ensure_rows(h, (rows + BM - 1) / BM * BM))) return rc;
        GatherArgs g;
        gather_obs_args(g, h, obs, rows, h->cfg.obs_dim);
        if ((rc = launch_gather(g, st)) || (rc = launch_forward(h->net, st))) return rc;
        const Net& net = h->net;
        const int n = net.n[net.L];
        dnsac::SacHeadArgs a;
        memset(&a, 0, sizeof(a));
        a.rows = rows; a.n = n; a.mode = s->mode;
        a.h_hi = net.h[net.L]; a.h_lo = (h->passes > 1) ? a.h_hi + static_cast<long long>(h->max_rows) * n : nullptr;
        const dn_sac_actor_config& c = h->cfg;
        a.w_mu = h->params + c.mu_w_off; a.b_mu = h->params + c.mu_b_off;
        a.w_ls = h->params + c.log_std_w_off; a.b_ls = h->params + c.log_std_b_off;
        a.mu = h->mu; a.log_std = h->log_std; a.action = action; a.log_prob = log_prob;
        a.counter = (s->mode == DN_SAC_SAMPLE) ? counter : nullptr;
        a.seed = s->seed; a.row_id_offset = s->row_id_offset;
        const int blocks = std::min((rows + HEAD_WARPS - 1) / HEAD_WARPS, 3 * h->sms);
        h->head<<<blocks, HEAD_WARPS * 32, 2 * c.act_dim * n * sizeof(float), st>>>(a);
        PPO_CUDA(cudaGetLastError());
    }
    return (s->mode == DN_SAC_DETERMINISTIC) ? DN_OK : advance_counter(s->counter, st);
}

int dn_sac_actor_buffer(dn_sac_actor* h, const char* name, void** ptr, int64_t* elems) {
    if (!h || !name || !ptr || !elems) return dn_internal_fail(DN_EINVAL, "dn_sac_actor_buffer: null argument");
    const long long R = h->max_rows;
    const std::string s(name);
    if (s == "x") { *ptr = h->x; *elems = 2 * R * XPAD; return DN_OK; }
    if (s == "mu") { *ptr = h->mu; *elems = R * h->cfg.act_dim; return DN_OK; }
    if (s == "log_std") { *ptr = h->log_std; *elems = R * h->cfg.act_dim; return DN_OK; }
    if (find_planes(h, h->net, s, ptr, elems)) return DN_OK;
    return dn_internal_fail(DN_EINVAL, "dn_sac_actor_buffer: unknown buffer name");
}

}  // extern "C"
