// Shared device/host helpers for the fastllm_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <stdexcept>
#include <string>

namespace fl {

constexpr int kNumSMs = 148;          // B200: 2 dies x 74 SMs; grids are sized in multiples of this
constexpr int kKvPage = 64;           // tokens per KV page
constexpr int kMaxBatch = 256;

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define FL_CUDA(expr)                                                                                  \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            throw ::fl::Error(-2, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + \
                                      ":" + std::to_string(__LINE__) + ")");                           \
    } while (0)

#define FL_CHECK(cond, code, msg)                       \
    do {                                                \
        if (!(cond)) throw ::fl::Error((code), (msg));  \
    } while (0)

// ---- device helpers ----------------------------------------------------------------------------------

// 128-bit streaming load through the read-only path without polluting L1 (weights are read exactly once per step).
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// bf16 pair packed in a u32 -> two f32 (exact: bf16 is the top half of an f32)
__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

__device__ __forceinline__ uint16_t f32_to_bf16_rne(float f) {
    uint32_t b = __float_as_uint(f);
    return (uint16_t)((b + 0x7FFFu + ((b >> 16) & 1u)) >> 16);
}

// two f32 -> packed bf16x2 (lo in bits 0-15), round-to-nearest-even, ONE instruction (same rounding as f32_to_bf16_rne)
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// ---- FP8 e4m3 KV elements (FL_KV_FP8_E4M3).  Kernels that read or write K/V pages are templated on the element type KV:
// uint16_t = bf16, uint8_t = e4m3.
template <typename KV>
constexpr bool kv_is_fp8 = sizeof(KV) == 1;

// two f32 -> packed e4m3x2 (lo in bits 0-7): round-to-nearest-even, saturating (|x| > 448 -> +-448, never NaN)
__device__ __forceinline__ uint16_t f32x2_to_e4m3x2(float lo, float hi) {
    uint16_t r;
    asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(hi), "f"(lo));
    return r;
}
// packed e4m3x2 -> packed bf16x2, exact (every e4m3 value is a bf16 value): e4m3 -> f16 -> f32 -> bf16
__device__ __forceinline__ uint32_t e4m3x2_to_bf16x2(uint16_t v) {
    uint32_t h;
    asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h) : "h"(v));
    float lo, hi;
    asm("cvt.f32.f16 %0, %1;" : "=f"(lo) : "h"((uint16_t)(h & 0xFFFFu)));
    asm("cvt.f32.f16 %0, %1;" : "=f"(hi) : "h"((uint16_t)(h >> 16)));
    return pack_bf16x2(lo, hi);
}
// the value a K/V element of type KV holds for x, as the bf16 bits the attention operands carry
template <typename KV>
__device__ __forceinline__ uint16_t kv_round_bf16(float x) {
    if constexpr (kv_is_fp8<KV>) return (uint16_t)e4m3x2_to_bf16x2(f32x2_to_e4m3x2(x, 0.f));
    else return f32_to_bf16_rne(x);
}
// two K/V elements of type KV for (lo, hi), packed as KV's storage of a pair
template <typename KV>
__device__ __forceinline__ uint32_t kv_pack2(float lo, float hi) {
    if constexpr (kv_is_fp8<KV>) return f32x2_to_e4m3x2(lo, hi);
    else return (uint32_t)f32_to_bf16_rne(lo) | ((uint32_t)f32_to_bf16_rne(hi) << 16);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}

// Programmatic dependent launch (PDL): the consumer kernel may start early; everything that depends on the
// producer's output must come after pdl_wait().  Weights never depend on a previous kernel, so GEMV kernels
// issue their first weight loads BEFORE pdl_wait() and overlap them with the producer's tail.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- mbarrier / bulk-copy (TMA engine, 1-D) helpers ------------------------------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// non-blocking probe of the phase with the given parity
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
// global -> shared bulk async copy (the TMA engine's 1-D mode; SASS: UBLKCP); bytes % 16 == 0, 16-B aligned both sides.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

}  // namespace fl
