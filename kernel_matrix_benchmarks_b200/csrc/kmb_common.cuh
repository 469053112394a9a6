// Shared device/host helpers for libkmb_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kmb_b200.h"

namespace kmb {

// ---- host-side error plumbing (defined in kmb_api.cu) -------------------------------------
int set_error(int code, const char* fmt, ...);
void count_launch(int n = 1);
// Per-(kernel function, device) launch state, thread-safe (kmb_api.cu).  cudaFuncSetAttribute is a per-device
// setting and occupancy a per-device answer, so neither may be cached per process: one process may drive
// several GPUs (B200Product(n_gpus=...), one host thread or many).
int ensure_dyn_smem(const void* fn, int smem_bytes);                             // opt-in dynamic shared memory
int resident_ctas(const void* fn, int threads, int smem_bytes, int* per_sm);     // also ensures the opt-in
int device_sm_count(int* sms);

#define KMB_CUDA_CHECK(expr)                                                                         \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess)                                                                       \
            return kmb::set_error(KMB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                  __FILE__, __LINE__);                                               \
    } while (0)

// coordinate scale folded into x and y so the exponential is a bare ex2
__host__ __device__ constexpr float coord_scale(int kid) {
    if (kid == KMB_KERNEL_GAUSSIAN) return 1.2011224087864498f;             // sqrt(log2 e)
    if (kid == KMB_KERNEL_ABSOLUTE_EXPONENTIAL) return 1.4426950408889634f; // log2 e
    return 1.0f;
}

// ---- PTX helpers ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "KMB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra KMB_DONE;\n"
        "bra KMB_WAIT;\n"
        "KMB_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// Producer-side wait: the slot frees once per ~10^4 cycles, so sleep between probes instead of
// competing with the consumer warps for issue slots.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    while (true) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(256);
    }
}
// TMA 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// Named barrier over a subset of the CTA's warps.
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ float ex2_approx(float x) {  // one MUFU.EX2
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {  // one MUFU.RSQ
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {  // one MUFU.RSQ + one FMUL, x >= 0
    // sqrt.approx.ftz expands to MUFU.RSQ + FMUL + two FSETP/SEL fix-ups for 0 and inf; clamping the
    // argument away from zero keeps rsqrt finite and needs no fix-up (sqrt(1e-30) = 1e-15 is below FP32
    // resolution of the exponents it feeds)
    const float c = fminf(fmaxf(x, 1.0e-30f), 3.0e38f);   // one FMNMX3; inf would give inf * 0
    return c * rsqrt_approx(c);
}

// Packed FP32 pairs (Blackwell FADD2 / FMUL2 / FFMA2: two lanes of work per issue slot).
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

}  // namespace kmb
