// common.cuh -- shared helpers for the sm_100a kernels of libpiml_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/piml_b200.h"

namespace piml {

// ---- host side: error reporting and launch accounting ---------------------------------------------------------
int fail(int code, const char *fmt, ...);       // records the thread-local message, returns `code`
void count_launch(int n = 1);                    // piml_launch_count()
int check_launch(const char *what);              // cudaGetLastError after a launch -> PIML_OK / PIML_ERR_CUDA
int sm_count();                                  // SMs of the current device (cached)

#define PIML_REQUIRE(cond, ...)                                   \
    do {                                                          \
        if (!(cond)) return piml::fail(PIML_ERR_INVALID, __VA_ARGS__); \
    } while (0)

#define PIML_CUDA(expr)                                                                        \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return piml::fail(PIML_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- device side: exact fp32 building blocks (SURVEY.md Appendix A.1) ---------------------------------------------
// Every expression on a neighbour-selection / gate path goes through explicit round-to-nearest intrinsics so that
// nvcc can never contract a*b+c into an FMA the reference does not perform.

__device__ __forceinline__ float norm2_rn(float x, float y) {       // torch.norm(p=2) over a 2-vector
    return __fsqrt_rn(__fmaf_rn(y, y, __fmul_rn(x, x)));
}

__device__ __forceinline__ float nan_to_zero(float x) { return (x != x) ? 0.0f : x; }

// ---- device side: mbarrier + TMA bulk copy (cp.async.bulk, SASS UBLKCP) -----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// Bounded variant for bring-up / self tests: gives up after ~`spins` polls and returns false instead of hanging the GPU.
__device__ __forceinline__ bool mbar_wait_bounded(uint64_t *bar, uint32_t parity, uint32_t spins) {
    for (uint32_t i = 0; i < spins; ++i) {
        uint32_t ok;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) return true;
    }
    return false;
}

// global -> shared bulk copy of `bytes` (multiple of 16, both addresses 16B aligned), completion on `bar`
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// One thread's asynchronous 16 B global -> shared copy (cp.async, L2 only; both addresses 16 B aligned), completed by
// cp_async_wait<k> (k = commit groups left in flight) followed by a barrier between the threads that read it.
__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int K>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(K) : "memory"); }

// Stage `n` 8-byte elements (float2) from gmem into smem.  Called by ALL threads of the CTA with identical
// arguments.  If `src` is 16B aligned one elected thread issues a TMA bulk copy that completes on `bar` (and copies
// an odd trailing element by hand); otherwise the CTA copies cooperatively.  Returns true if the consumer must wait
// on `bar`; in either case a __syncthreads() (or the barrier wait plus a later __syncthreads) must separate this
// call from the first read of `dst`.
__device__ __forceinline__ bool stage_float2(float2 *dst, const float2 *src, int n, uint64_t *bar) {
    const bool tma = (reinterpret_cast<uintptr_t>(src) & 15u) == 0 && n >= 2;
    if (tma) {
        if (threadIdx.x == 0) {
            const uint32_t bytes = static_cast<uint32_t>(n & ~1) * 8u;
            mbar_expect_tx(bar, bytes);
            tma_bulk_g2s(dst, src, bytes, bar);
            if (n & 1) dst[n - 1] = src[n - 1];
        }
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    }
    return tma;
}

}  // namespace piml
