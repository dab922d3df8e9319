// Shared helpers for the sm_100a kernels of crfconv_b200.  Not a compatibility layer: everything here assumes
// compute capability 10.0 (B200), 32-wide warps, 148 SMs.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

// ---- C-ABI status codes (include/crfconv_b200.h) -------------------------------------------------------
#define CRF_OK 0
#define CRF_ERR_INVALID_ARG (-1)
#define CRF_ERR_WORKSPACE (-2)
#define CRF_ERR_UNSUPPORTED (-3)
#define CRF_ERR_NO_DEVICE (-4)

// Positive return values are cudaError_t.
#define CRF_CUDA(call)                                         \
    do {                                                       \
        cudaError_t _e = (call);                               \
        if (_e != cudaSuccess) return (int)_e;                 \
    } while (0)
#define CRF_LAUNCH_CHECK()                                     \
    do {                                                       \
        cudaError_t _e = cudaPeekAtLastError();                \
        if (_e != cudaSuccess) return (int)_e;                 \
    } while (0)

namespace crf {

constexpr int kNumSMs = 148;   // B200

// Same-address global atomics serialise in L2 at ≈40 ns each (measured: 1.8 M float atomics on 256 addresses = 290 µs),
// so a per-CTA epilogue that adds into ONE result vector costs (#CTAs × 40 ns) of serial tail per kernel.  Reductions over
// CTAs therefore go through kStatSlots / kGradSlots partial copies (CTA b adds into slot b % slots: chain depth <= 5-30 instead of 300-2000) that a
// tiny follow-up kernel sums in a fixed order.
constexpr int kStatSlots = 64;    // BatchNorm Σ/Σ² and backward Σ partials: buffers are [kStatSlots][2·C] doubles
constexpr int kGradSlots = 32;    // weight-gradient partials: scratch is [kGradSlots][Cout·Ktot] floats

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace; 256-byte aligned slices.
struct Carver {
    char* base;
    size_t off = 0;
    explicit Carver(void* p) : base(reinterpret_cast<char*>(p)) {}
    template <typename T>
    T* take(size_t count) {
        T* r = reinterpret_cast<T*>(base + off);
        off += align_up(count * sizeof(T), 256);
        return r;
    }
};

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// order-preserving float <-> uint mapping for atomicMin/atomicMax on floats
__device__ __forceinline__ unsigned f2ord(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

}  // namespace crf
