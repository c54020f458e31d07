// Packed-FP32 register pairs and 1-D TMA bulk copies into shared memory, shared by the all-pairs kernels (the
// brute-force k-NN of spx_knn.cu, the RANSAC plane scoring of spx_plane.cu).
#pragma once

#include "spx_common.cuh"

namespace spx {

// Two fp32 values in one 64-bit register pair, the operand of sm_100's FADD2 / FMUL2 / FFMA2 (sub/mul/fma.rn.f32x2:
// IEEE round-to-nearest per element, so results stay bit-identical to the scalar instructions).
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}

// ---- tiles through the TMA engine: 1-D bulk copies (cp.async.bulk, completion counted in bytes on an mbarrier) into
// a double-buffered shared-memory tile, issued by one thread a whole tile ahead of the compute, so the global-load
// latency of the staging (the long-scoreboard + barrier stalls of the synchronous version:
// profiles/r2g_ncu_bf_p4.txt) hides behind the work on the previous tile.  Source and size must be 16-byte aligned.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

}  // namespace spx
