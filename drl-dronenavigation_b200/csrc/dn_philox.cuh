// dn_philox.cuh -- the counter-based generator shared by the env step kernel (random spawn, dn_device.cuh) and the PPO
// sampler (dn_ppo_act, ppo_kernels.cuh).  Host-compilable through tests/host_emu/cuda_shim.h.
//
// Philox4x32-10 (Salmon et al., SC'11), key = seed.  The same function is restated in oracle/dyn_oracle.py for the
// parity tests.  Every caller puts a GLOBAL id (env id, row id) in the last two counter words, so results do not
// depend on how the rows are sharded over GPUs; the second word tells the streams apart (spawn draws use 0 and 1,
// the PPO sampler DN_PPO_ACT_TAG of include/dnppo.h).
#pragma once
#include <stdint.h>

namespace dn {

struct U4 { uint32_t x, y, z, w; };
__device__ __forceinline__ void mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
    const unsigned long long p = static_cast<unsigned long long>(a) * b;
    hi = static_cast<uint32_t>(p >> 32); lo = static_cast<uint32_t>(p);
}
__device__ __forceinline__ U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t h0, l0, h1, l1;
        mulhilo32(0xD2511F53u, c.x, h0, l0);
        mulhilo32(0xCD9E8D57u, c.z, h1, l1);
        c = U4{h1 ^ c.y ^ k0, l1, h0 ^ c.w ^ k1, l0};
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c;
}
// 24-bit uniforms: exact in FP32
__device__ __forceinline__ float u01(uint32_t x) { return static_cast<float>(x >> 8) * (1.0f / 16777216.0f); }          // [0, 1)
__device__ __forceinline__ float u01_open(uint32_t x) { return (static_cast<float>(x >> 8) + 1.0f) * (1.0f / 16777216.0f); }  // (0, 1]

}  // namespace dn
