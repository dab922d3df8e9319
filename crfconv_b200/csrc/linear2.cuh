// Fast-path Linear kernels (second generation) for the shapes that carry the bytes of the hot path:
// Cout <= 64, Cin_total <= 128, channel counts multiples of 4 (every Linear of the CRF layers and ResNet blocks at the two
// finest levels).  Differences from the generic kernels of linear.cu:
//   * persistent CTAs (a multiple of the 148 SMs) that stream 128/64/32-row tiles through a 3-stage cp.async ring, so
//     HBM/L2 latency is hidden by copies in flight instead of by occupancy;
//   * the weight matrix is split ONCE per CTA into bf16 (hi, lo) pairs kept in shared memory, so the inner loop issues
//     only LDS + mma for the B operand;
//   * contractions on mma.sync m16n8k16 bf16 with bf16x3 error compensation: a·b ≈ a_hi·b_hi + a_hi·b_lo + a_lo·b_hi,
//     16 mantissa bits per operand → relative error ≈ 2^-16, well inside the 1e-3 parity budget, at twice the MAC rate of
//     3xTF32 on this part (measured: 557 vs 278 TFLOP/s dense for single-pass bf16 / tf32 mma.sync, profiles/).
//     precision 2 selects a single bf16 pass (stated tolerance 2e-2, see DESIGN.md §5); fwd2_kernel exists only in that form,
//     the fp32-grade forward is the 3xTF32 fwd2t_kernel.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace crf {
namespace lin2 {

constexpr int kThreads = 256;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool pred) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    const int sz = pred ? 16 : 0;   // src-size 0 ⇒ zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void split2(float x, float y, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x, y);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x - __low2float(h), y - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// D += A·B with (hi, lo) operands.  X3 = false ⇒ single bf16 pass.
template <bool X3>
__device__ __forceinline__ void mma3(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0, uint32_t bh1,
                                     uint32_t bl0, uint32_t bl1) {
    if constexpr (X3) {
        mma_bf16(d, al, bh0, bh1);
        mma_bf16(d, ah, bl0, bl1);
    }
    mma_bf16(d, ah, bh0, bh1);
}

}  // namespace lin2
}  // namespace crf
