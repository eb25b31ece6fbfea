// mc3_b200 -- shared device helpers (sm_100a only).
#pragma once
#ifndef __CUDACC_RTC__          // NVRTC (user models, jit.cu) has none of these headers
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#endif
#include "../../include/mc3b200.h"

#ifndef __CUDA_ARCH__
#define MC3B_HOST 1
#endif

#ifndef __CUDACC_RTC__
// ---- error plumbing (C-ABI returns int, message via mc3b_last_error) ------
void mc3b_set_error(const char* fmt, ...);
#define MC3B_CHECK_ARG(cond, ...)                                      \
    do { if (!(cond)) { mc3b_set_error(__VA_ARGS__); return MC3B_ERR_ARG; } } while (0)
#define MC3B_CHECK_LAUNCH(what)                                        \
    do { cudaError_t e_ = cudaGetLastError();                          \
         if (e_ != cudaSuccess) {                                      \
             mc3b_set_error("%s: %s", what, cudaGetErrorString(e_));   \
             return MC3B_ERR_CUDA; } } while (0)
#define MC3B_CUDA(call)                                                \
    do { cudaError_t e_ = (call);                                      \
         if (e_ != cudaSuccess) {                                      \
             mc3b_set_error("%s: %s", #call, cudaGetErrorString(e_));  \
             return MC3B_ERR_CUDA; } } while (0)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
int mc3b_sm_count();
#endif

// ---- TMA bulk copy (1-D, no tensor map) + mbarrier -------------------------
// cp.async.bulk global->shared completes on an mbarrier by byte count; SASS:
// UBLKCP + SYNCS.  Addresses and sizes must be multiples of 16 bytes.
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
// order generic-proxy shared-memory writes before later async-proxy (TMA) writes
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- Philox4x32-10 counter-based generator ---------------------------------
// Stream layout used by the sampler: key = 64-bit seed; counter =
// (global chain id, draw slot, generation lo, generation hi).  A chain's
// stream therefore does not depend on how chains are spread over GPUs.
struct Philox {
    uint32_t k0, k1;
    __device__ __forceinline__ Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
    __device__ __forceinline__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
        const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; r++) {
            uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
            uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
            uint32_t n0 = hi1 ^ c1 ^ a, n2 = hi0 ^ c3 ^ b;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            a += W0; b += W1;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};
// 53-bit uniform in [0,1) from two 32-bit words (same construction as
// numpy's random_double: (a>>5, b>>6)).
__device__ __forceinline__ double u01(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}
// integer in [0, n) from 64 random bits (multiply-high; bias < n / 2^64).
__device__ __forceinline__ int64_t ubelow(uint32_t a, uint32_t b, int64_t n) {
    uint64_t r = ((uint64_t)a << 32) | b;
    return (int64_t)__umul64hi(r, (uint64_t)n);
}
