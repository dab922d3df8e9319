// tcgen05 / TMEM / mbarrier primitives for the sm_100a Linear kernels (linear3.cu).  Bring-up and the descriptor encodings
// were validated on a B200 with scripts/micro/umma_test.cu (exact results on tf32-representable inputs; 3xTF32 = 1.7e-6).
//   * operands live in shared memory in the K-major SWIZZLE_128B canonical layout: a "slab" is [rows][32 floats], one
//     128-byte line per row, the 16-byte chunk c of row r stored at chunk position c ^ (r & 7); 8-row groups are 1024 B
//     apart (the descriptor's stride byte offset); slabs are 1024-byte aligned;
//   * MN-major tf32 operands (the contraction runs along the rows, linear3w.cu / linear3b.cu) exist only in the
//     SWIZZLE_128B_BASE32B layout: a block is [rows][32 channels], one 128-byte line per row, the 32-byte chunk c of row r
//     stored at chunk position c ^ (r & 3); 4-row atoms are 512 B apart (descriptor SBO), 32-channel blocks LBO bytes apart;
//   * one thread issues tcgen05.mma (kind::tf32, M = 128, N = 16..256, K = 8 per instruction); the fp32 accumulator lives in
//     TMEM: row i of D on lane i, column j at column base + j;
//   * completion is tracked with tcgen05.commit → mbarrier; every wait is bounded and traps instead of hanging the GPU.
#pragma once
#include <cstdint>
#include <cstdio>

namespace crf {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Waits are bounded by TIME (≈2 s of SM clock): a mis-programmed pipeline traps (surfacing as a CUDA error at the C ABI)
// instead of hanging the device.  The slow path is kept out of line: the kernels' three warp roles share a small instruction
// cache, and an inlined printf call site per wait would triple the size of the issue loop.
static __device__ __noinline__ void mbar_timeout() {
    printf("crfconv_b200: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
    __trap();
}
static __device__ __noinline__ void mbar_wait_slow(uint64_t* bar, uint32_t parity, unsigned sleep_ns) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (sleep_ns) __nanosleep(sleep_ns);
        if (clock64() - t0 > 4000000000LL) mbar_timeout();
    }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity, 0);
}
// Same, for warps that can afford a slower wake-up: sleeps between polls so that waiting warps leave the issue slots to the
// warps that are converting / storing.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
    if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity, 40);
}
// Same bound, inline and without the printf: no call site, so a warp that keeps many registers live across the wait does not
// spill them around a call (the trap still surfaces as a CUDA error).
__device__ __forceinline__ void mbar_wait_relaxed_nocall(uint64_t* bar, uint32_t parity) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(40);
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}

// one lane of a converged warp; unlike `lane == 0` the compiler knows the region is single-threaded and issues tcgen05
// instructions without a per-instruction election loop
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// whole warp; writes the TMEM base address (lane 0, column c) to *slot
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (descriptor version 1 = sm_100)
__device__ __forceinline__ uint64_t smem_desc_k128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// byte offset of the 16-byte chunk c16 (0..7) of row r inside a SWIZZLE_128B_BASE32B block (32-byte chunks XOR (r & 3))
__device__ __forceinline__ uint32_t blk_off(int r, int c16) { return (uint32_t)(r * 128 + ((((c16 >> 1) ^ (r & 3)) << 5) | ((c16 & 1) << 4))); }
// MN-major SWIZZLE_128B_BASE32B descriptor: LBO = stride between 32-channel blocks, SBO = 512 B between 4-row atoms
__device__ __forceinline__ uint64_t desc_mn(uint32_t saddr, uint32_t lbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)1 << 61);
}
// instruction descriptor: D f32, A and B tf32, both K-major
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on `bar` once every tcgen05.mma issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes × 16 consecutive columns: thread l of warp w (w % 4 selects the lane quarter) gets row 32·(w%4)+l
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// split form: issue several loads, then one tmem_ld_wait()
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// byte offset of the 16-byte chunk c (4 floats) of row r inside a slab
__device__ __forceinline__ uint32_t slab_chunk_off(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

// tf32 split: hi keeps the top 10 mantissa bits (what the tensor core reads), lo = x − hi exactly
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    lo = x - hi;
}

}  // namespace umma
}  // namespace crf
