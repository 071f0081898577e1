// tc.cuh -- thin inline-PTX layer over the Blackwell 5th-generation tensor cores (tcgen05) for sm_100a:
// TMEM allocation, UMMA shared-memory / instruction descriptors, tcgen05.mma (kind::tf32, A from TMEM, B from shared
// memory), tcgen05.commit, tcgen05.ld / tcgen05.st and the fences that order them against mbarriers.
//
// Operand conventions used by the kernels in this library (all K-major, no swizzle):
//   * B (weights, N x K): shared-memory image of 16-byte cells [K/4][N][4 tf32]; a core matrix (8 rows x 16 B) is 128
//     contiguous bytes, so SBO (8-row groups) = 128 B and LBO (the two 16-byte K cells of one K = 8 MMA) = N * 16 B;
//   * A (activations, 128 x K): TMEM, lane = row, column = k (one 32-bit tf32 per column);
//   * D (accumulator, 128 x N fp32): TMEM, lane = row, column = n.
#pragma once
#include <stdint.h>

namespace piml {
namespace tc {

__device__ __forceinline__ uint32_t smem_addr(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One full warp allocates `ncols` (power of two >= 32) TMEM columns; the base address lands in *slot (shared memory).
__device__ __forceinline__ void tmem_alloc(uint32_t *slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(slot)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major, SWIZZLE_NONE (bit layout: cute::UMMA::SmemDescriptor).
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3fffu);            // start address      bits [0,14)
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;  // leading byte offset bits [16,30)
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;  // stride byte offset  bits [32,46)
    d |= static_cast<uint64_t>(1) << 46;                           // descriptor version (Blackwell)
    return d;                                                      // base offset 0, layout type 0 = no swizzle
}

// Instruction descriptor for kind::tf32, fp32 accumulate, M = 128, both operands K-major (cute::UMMA::InstrDescriptor).
__host__ __device__ __forceinline__ uint32_t idesc_tf32(int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | ((128u >> 4) << 24);
}

// Instruction descriptor for kind::f16 with fp16 A / B, fp32 accumulate, M = 128, both operands K-major.
__host__ __device__ __forceinline__ uint32_t idesc_f16(int N) {
    return (1u << 4) | (0u << 7) | (0u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | ((128u >> 4) << 24);
}

// D[tmem] (+)= A[tmem] * B[smem]^T, M = 128, K = 16 (fp16 operands, two per 32-bit TMEM column / eight per 16-byte
// shared-memory cell).  Issued by ONE thread.
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                           bool accumulate) {
    const uint32_t acc = accumulate ? 1u : 0u;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem]^T, M = 128, K = 8 (tf32).  Issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            bool accumulate) {
    const uint32_t acc = accumulate ? 1u : 0u;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}

// One lane of a converged warp (PTX elect.sync): a warp-UNIFORM predicate, so that code under it keeps its operands in
// uniform registers.  tcgen05.mma takes its descriptors from uniform registers: when the issuing code is divergent
// (`if (lane == 0)`) ptxas wraps EVERY MMA in an ELECT / 5 x R2UR.BROADCAST / branch "waterfall" loop, which costs
// ~100 cycles per MMA in the issuing thread -- more than the MMA itself (65 cycles for M = 128, K = 16 fp16).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// All previously issued tcgen05.mma of this thread arrive (once) on `bar` when they complete.
__device__ __forceinline__ void commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(bar))
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}

// 32 lanes x 32 consecutive columns: thread i of the warp gets TMEM lane (taddr.lane + i), columns taddr.col .. +31.
__device__ __forceinline__ void ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// x = hi + lo (+ O(2^-22 |x|)) with hi, lo exactly representable in tf32 (round to nearest): the 3xTF32 split.
__device__ __forceinline__ void split_tf32(float x, uint32_t &hi, uint32_t &lo) {
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hi) : "f"(x));
    const float rest = x - __uint_as_float(hi);
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lo) : "f"(rest));
}

// x = hi + lo (+ O(2^-22 |x|)) with hi, lo fp16 (round to nearest): the 3xFP16 split.  Two values at a time:
// returns the packed pairs {hi(x0), hi(x1)} and {lo(x0), lo(x1)} (x0 in the low half = the even K index).
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t &hi, uint32_t &lo) {
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));          // d.hi = cvt(a), d.lo = cvt(b)
    float h0, h1;
    asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}"
        : "=f"(h0), "=f"(h1) : "r"(hi));
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - h1), "f"(x0 - h0));
}
__device__ __forceinline__ void split_f16(float x, uint16_t &hi, uint16_t &lo) {
    uint32_t h, l;
    split_f16x2(x, 0.f, h, l);
    hi = static_cast<uint16_t>(h & 0xffffu); lo = static_cast<uint16_t>(l & 0xffffu);
}

}  // namespace tc
}  // namespace piml
