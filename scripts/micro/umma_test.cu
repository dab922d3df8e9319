// Bring-up test for the tcgen05 path: D[128,N] = A[128,K] · B[N,K]^T with kind::tf32, operands written to shared memory by
// CUDA cores in the K-major SWIZZLE_128B canonical layout, accumulator in TMEM, read back with tcgen05.ld.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o scripts/micro/umma_test scripts/micro/umma_test.cu
// Every wait is bounded (trap after ~1e7 polls) so a wrong descriptor cannot hang the box.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
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
__device__ __forceinline__ void mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
    for (uint32_t i = 0; i < (1u << 24); ++i)
        if (mbar_try_wait(bar, parity)) return;
    printf("mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
    __trap();
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"): rows are 128 bytes, 8-row groups are 1024 bytes apart.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);          // start address
    d |= (uint64_t)0 << 16;                          // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset: 8 rows × 128 B
    d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
    return d;
}

// instruction descriptor: D = f32, A = B = tf32, both K-major, M = 128
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
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

// element (r, k) of a K-major SW128 slab of 32 floats per row
__device__ __forceinline__ uint32_t sw128_off(int r, int k) { return (uint32_t)(r * 128 + ((((k >> 2) ^ (r & 7)) << 4) | ((k & 3) << 2))); }

template <int N, int KSLABS, bool X3>
__global__ void __launch_bounds__(128) umma_test_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ D) {
    constexpr int K = 32 * KSLABS;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    // [A hi slabs][A lo slabs][B hi slabs][B lo slabs]
    uint8_t* a_hi = smem;
    uint8_t* a_lo = a_hi + KSLABS * 128 * 128;
    uint8_t* b_hi = a_lo + KSLABS * 128 * 128;
    uint8_t* b_lo = b_hi + KSLABS * N * 128;
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base;

    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(64));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // operands → swizzled shared memory, split into tf32 hi + remainder lo
    for (int i = tid; i < 128 * K; i += 128) {
        const int r = i / K, k = i % K;
        const float x = A[i];
        const float hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
        const uint32_t off = (k / 32) * (128 * 128) + sw128_off(r, k % 32);
        *(float*)(a_hi + off) = X3 ? hi : x;
        *(float*)(a_lo + off) = x - hi;
    }
    for (int i = tid; i < N * K; i += 128) {
        const int r = i / K, k = i % K;
        const float x = B[i];
        const float hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
        const uint32_t off = (k / 32) * (N * 128) + sw128_off(r, k % 32);
        *(float*)(b_hi + off) = X3 ? hi : x;
        *(float*)(b_lo + off) = x - hi;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes → visible to the tensor core's async proxy
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;

    if (tid == 0) {
        constexpr uint32_t idesc = make_idesc(128, N);
        uint32_t acc = 0;
        for (int s = 0; s < KSLABS; ++s) {
            for (int k8 = 0; k8 < 4; ++k8) {
                const uint32_t ao = s * 128 * 128 + k8 * 32, bo = s * N * 128 + k8 * 32;
                const uint64_t ah = make_desc(smem_u32(a_hi + ao)), al = make_desc(smem_u32(a_lo + ao));
                const uint64_t bh = make_desc(smem_u32(b_hi + bo)), bl = make_desc(smem_u32(b_lo + bo));
                if (X3) {
                    umma_tf32(tmem, al, bh, idesc, acc); acc = 1;
                    umma_tf32(tmem, ah, bl, idesc, acc);
                }
                umma_tf32(tmem, ah, bh, idesc, acc); acc = 1;
            }
        }
        umma_commit(&bar);
    }
    mbar_wait_bounded(&bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // warp w reads TMEM lanes 32w .. 32w+31 (one accumulator row per thread)
    const int row = warp * 32 + (tid & 31);
    for (int c = 0; c < N; c += 16) {
        float v[16];
        tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) D[row * N + c + i] = v[i];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(64));
}

template <int N, int KSLABS, bool X3>
static int run(const char* name, bool exact_inputs) {
    constexpr int K = 32 * KSLABS;
    std::vector<float> A(128 * K), B(N * K), D(128 * N), ref(128 * N);
    srand(1234);
    for (auto& x : A) x = exact_inputs ? (float)((rand() % 17) - 8) * 0.25f : (float)rand() / RAND_MAX * 2.f - 1.f;
    for (auto& x : B) x = exact_inputs ? (float)((rand() % 17) - 8) * 0.5f : (float)rand() / RAND_MAX * 2.f - 1.f;
    double amax = 0;
    for (int i = 0; i < 128; ++i)
        for (int j = 0; j < N; ++j) {
            double s = 0;
            for (int k = 0; k < K; ++k) s += (double)A[i * K + k] * (double)B[j * K + k];
            ref[i * N + j] = (float)s;
            amax = fmax(amax, fabs(s));
        }
    float *dA, *dB, *dD;
    cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, D.size() * 4);
    cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
    cudaMemset(dD, 0xff, D.size() * 4);
    const size_t smem = 2 * KSLABS * 128 * 128 + 2 * KSLABS * N * 128 + 1024;
    auto kern = umma_test_kernel<N, KSLABS, X3>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<1, 128, smem>>>(dA, dB, dD);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: CUDA error %s\n", name, cudaGetErrorString(e)); return 1; }
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    double err = 0;
    int bad = 0;
    for (int i = 0; i < 128 * N; ++i) {
        const double d = fabs((double)D[i] - (double)ref[i]);
        if (!(d <= 1e30)) { ++bad; continue; }
        err = fmax(err, d);
    }
    printf("%s: N=%d K=%d x3=%d  max|err|=%.3e (max|ref|=%.3e, rel %.3e) nan=%d   D[0..3]=%g %g %g %g  ref=%g %g %g %g\n", name, N, K, (int)X3,
           err, amax, err / amax, bad, D[0], D[1], D[2], D[3], ref[0], ref[1], ref[2], ref[3]);
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
    return 0;
}


// ---- throughput probe: one elected lane issues `iters` MMAs back to back (descriptors precomputed, loop unrolled by 4) ----
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
template <int M, int N, int NACC>
__global__ void __launch_bounds__(128) umma_rate_kernel(int iters, long long* out) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* a_s = smem;                  // 128 × 128 B
    uint8_t* b_s = smem + 128 * 128;      // N × 128 B
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    for (int i = tid; i < (128 + N) * 32; i += 128) ((float*)smem)[i] = 0.001f * (i % 7);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    if (warp == 1) {
        constexpr uint32_t idesc = make_idesc(M, N);
        const uint64_t a0 = make_desc(smem_u32(a_s)), b0 = make_desc(smem_u32(b_s));
        long long t0 = 0, t1 = 0;
        if (elect_one()) {
            t0 = clock64();
            for (int i = 0; i < iters; i += 4) {
#pragma unroll
                for (int j = 0; j < 4; ++j) umma_tf32(tmem + (uint32_t)((j % NACC) * N), a0 + 2 * j, b0 + 2 * j, idesc, 1);
            }
            t1 = clock64();
            umma_commit(&bar);
        }
        __syncwarp();
        mbar_wait_bounded(&bar, 0);
        const long long t2 = clock64();
        if (t0) { out[0] = t1 - t0; out[1] = t2 - t0; }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

template <int M, int N, int NACC>
static void rate() {
    long long* d;
    cudaMalloc(&d, 16);
    const size_t smem = (128 + N) * 128 + 1024;
    auto kern = umma_rate_kernel<M, N, NACC>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int iters = 4096;
    kern<<<1, 128, smem>>>(iters, d);
    kern<<<1, 128, smem>>>(iters, d);
    cudaError_t e = cudaDeviceSynchronize();
    long long h[2] = {0, 0};
    cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
    printf("rate M=%3d N=%3d nacc=%d: issue %.1f cyc/MMA, complete %.1f cyc/MMA  (math floor max(M,128)*N/256 = %d)  %s\n", M, N, NACC,
           (double)h[0] / iters, (double)h[1] / iters, (M > 128 ? M : 128) * N / 256, e == cudaSuccess ? "" : cudaGetErrorString(e));
    cudaFree(d);
}


// ---- issuer-loop probe: per "slab" 12 MMAs + commit, optionally an (already satisfied) mbarrier wait, syncwarp and a fresh election ----
template <int N, int MODE, int SPIN>
__global__ void __launch_bounds__(256) umma_loop_kernel(int slabs, long long* out) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    uint8_t* a_s = smem_dyn;
    uint8_t* b_s = smem_dyn + 128 * 128;
    __shared__ uint64_t bar_commit, bar_ready, bar_never;
    __shared__ volatile int stop_flag;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) { stop_flag = 0; mbar_init(&bar_never, 1); mbar_init(&bar_commit, 1); mbar_init(&bar_ready, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    for (int i = tid; i < (128 + N) * 32; i += 256) ((float*)smem_dyn)[i] = 0.001f * (i % 7);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    if (warp >= 2 && SPIN > 0) {            // 6 bystander warps: 1 = tight mbarrier polling, 2 = polling with nanosleep(40), 3 = shared-memory store traffic, 4 = ALU spin
        float* scratch = (float*)(smem_dyn + (128 + N) * 128);
        float acc = 0.f;
        while (!stop_flag) {
            if (SPIN == 1) { mbar_try_wait(&bar_never, 0); }
            if (SPIN == 2) { mbar_try_wait(&bar_never, 0); __nanosleep(40); }
            if (SPIN == 3) { for (int r = 0; r < 8; ++r) *(float4*)(scratch + ((tid - 64) * 4 + r * 768)) = make_float4(acc, 1.f, 2.f, 3.f); }
            if (SPIN == 4) { for (int r = 0; r < 64; ++r) acc = fmaf(acc, 1.0001f, 0.5f); }
            if (SPIN == 7) { for (int r = 0; r < 8; ++r) *(float4*)(scratch + ((tid - 64) * 4 + r * 768)) = make_float4(acc, 1.f, 2.f, 3.f); asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
            if (SPIN == 5) { mbar_try_wait(&bar_commit, 0); }                       // poll the barrier the commits arrive on
            if (SPIN == 6) { mbar_try_wait(&bar_commit, 0); mbar_try_wait(&bar_ready, 1); }   // ... and the one the issuer waits on
        }
        if (acc == 12345.f) out[1] = 0;
    }
    if (warp == 1) {
        constexpr uint32_t idesc = make_idesc(128, N);
        const uint64_t a0 = make_desc(smem_u32(a_s)), b0 = make_desc(smem_u32(b_s));
        const long long t0 = clock64();
        for (int s = 0; s < slabs; ++s) {
            if (MODE >= 1) { while (!mbar_try_wait(&bar_ready, 1)) {} if (MODE == 4) asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < 12; ++j) umma_tf32(tmem, a0 + 2 * (j & 3), b0 + 2 * (j & 3), idesc, 1);
                if (MODE != 3) umma_commit(&bar_commit);
            }
            if (MODE >= 2) __syncwarp();
        }
        const long long t1 = clock64();
        if (elect_one()) umma_commit(&bar_ready);     // final: wait for everything
        __syncwarp();
        // bar_ready phase 0 completes when all MMAs are done
        for (uint32_t i = 0; i < (1u << 24); ++i) if (mbar_try_wait(&bar_ready, 0)) break;
        const long long t2 = clock64();
        if ((tid & 31) == 0) { out[0] = t1 - t0; out[1] = t2 - t0; }
        stop_flag = 1;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}
template <int N, int MODE, int SPIN>
static void loop_rate() {
    long long* d;
    cudaMalloc(&d, 16);
    const size_t smem = (128 + N) * 128 + 8 * 768 * 4 + 4096;
    auto kern = umma_loop_kernel<N, MODE, SPIN>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int slabs = 512;
    kern<<<1, 256, smem>>>(slabs, d);
    kern<<<1, 256, smem>>>(slabs, d);
    cudaError_t e = cudaDeviceSynchronize();
    long long h[2] = {0, 0};
    cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
    printf("issuer loop N=%3d mode=%d bystanders=%d (0 blocked, 1 mbarrier poll, 2 poll+nanosleep, 3 STS traffic, 4 ALU): issue %.0f cyc/slab, complete %.0f cyc/slab  %s\n", N, MODE, SPIN,
           (double)h[0] / slabs, (double)h[1] / slabs, e == cudaSuccess ? "" : cudaGetErrorString(e));
    cudaFree(d);
}


// ---- MN-major bring-up: D[M, N] = Σ_k A[k][m] · B[k][n], operands stored "row = k" exactly like an activation tile ----
// slab image: [channel block of 32][KR rows × 128 B], chunk c of row r at c ^ (r & 7): the SAME bytes the K-major kernels use.
// tf32 MN-major operands only exist in the SWIZZLE_128B_BASE32B layout (type 1): rows (k) of 128 bytes, 32-byte chunk c of row k at
// position c ^ (k & 3); an atom is 4 rows (512 B); SBO = stride between K atoms, LBO = stride between 32-channel blocks.
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr, uint32_t lbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)1 << 61);
}
__device__ __forceinline__ uint32_t sw32_off(int r, int k) {      // element k (0..31) of row r
    const int c32 = (k >> 3) ^ (r & 3);
    return (uint32_t)(r * 128 + (c32 << 5) + ((k & 7) << 2));
}
template <int M, int N, int KR>
__global__ void __launch_bounds__(128) umma_mn_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ D) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    constexpr int SLAB = KR * 128;
    uint8_t* a_s = smem_dyn;                       // [M/32][KR][128 B]
    uint8_t* b_s = smem_dyn + (M / 32) * SLAB;     // [N/32][KR][128 B]
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(64));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    for (int i = tid; i < KR * M; i += 128) {      // A is [KR][M] row-major in global
        const int r = i / M, m = i % M;
        *(float*)(a_s + (m / 32) * SLAB + sw32_off(r, m % 32)) = A[i];
    }
    for (int i = tid; i < KR * N; i += 128) {
        const int r = i / N, n = i % N;
        *(float*)(b_s + (n / 32) * SLAB + sw32_off(r, n % 32)) = B[i];
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    if (warp == 1) {
        if (elect_one()) {
            constexpr uint32_t idesc = make_idesc(M, N) | (1u << 15) | (1u << 16);      // A and B MN-major
            for (int j = 0; j < KR / 8; ++j)
                umma_tf32(tmem, make_desc_mn(smem_u32(a_s) + j * 1024, SLAB), make_desc_mn(smem_u32(b_s) + j * 1024, SLAB), idesc, j > 0);
            umma_commit(&bar);
        }
        __syncwarp();
    }
    mbar_wait_bounded(&bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = warp * 32 + (tid & 31);
    for (int c = 0; c < N; c += 16) {
        float v[16];
        tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c, v);
        if (row < M)
            for (int i = 0; i < 16; ++i) D[row * N + c + i] = v[i];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(64));
}
template <int M, int N, int KR>
static void run_mn() {
    std::vector<float> A(KR * M), B(KR * N), D(128 * N, -1.f), ref(M * N);
    srand(7);
    for (auto& x : A) x = (float)((rand() % 17) - 8) * 0.25f;
    for (auto& x : B) x = (float)((rand() % 17) - 8) * 0.5f;
    for (int m = 0; m < M; ++m)
        for (int n = 0; n < N; ++n) {
            double s = 0;
            for (int k = 0; k < KR; ++k) s += (double)A[k * M + m] * (double)B[k * N + n];
            ref[m * N + n] = (float)s;
        }
    float *dA, *dB, *dD;
    cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, D.size() * 4);
    cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dD, D.data(), D.size() * 4, cudaMemcpyHostToDevice);
    const size_t smem = (size_t)(M / 32 + N / 32) * KR * 128;
    auto kern = umma_mn_kernel<M, N, KR>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<1, 128, smem>>>(dA, dB, dD);
    cudaError_t e = cudaDeviceSynchronize();
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    double err = 0;
    for (int i = 0; i < M * N; ++i) err = fmax(err, fabs((double)D[i] - (double)ref[i]));
    printf("MN-major M=%d N=%d Krows=%d: max|err| = %.3e   D[0..3] = %g %g %g %g  ref = %g %g %g %g   D[33*N+5]=%g ref %g  %s\n", M, N, KR, err, D[0], D[1], D[2],
           D[3], ref[0], ref[1], ref[2], ref[3], D[33 * N + 5], ref[33 * N + 5], e == cudaSuccess ? "" : cudaGetErrorString(e));
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
}


// ---- mixed majors: D[128, N] = Σ_k A[k][m] · B[n][k], A MN-major BASE32B (lines = k), B K-major (lines = n), instruction-descriptor
// bit 15 only.  This is the input-gradient product of csrc/linear3b.cu (A = Wᵀ, lines = output channels; B = dH, lines = rows).
// B is in K-major SWIZZLE_128B slabs (16-byte chunk c of line n at c ^ (n & 7), SBO = 1024 B).  Inputs are tf32-representable: exact.
template <int N, int K>
__global__ void __launch_bounds__(128) umma_mixed_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ D) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    constexpr int ASLAB = K * 128, BSLAB = N * 128;
    uint8_t* a_s = smem_dyn;                       // [4 channel blocks][K lines × 128 B]
    uint8_t* b_s = smem_dyn + 4 * ASLAB;           // [K / 32 slabs][N lines × 128 B]
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(64));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    for (int i = tid; i < K * 128; i += 128) {     // A is [K][128] row-major in global
        const int k = i / 128, m = i % 128;
        *(float*)(a_s + (m / 32) * ASLAB + sw32_off(k, m % 32)) = A[i];
    }
    for (int i = tid; i < N * K; i += 128) {       // B is [N][K] row-major in global
        const int n = i / K, k = i % K;
        *(float*)(b_s + (k / 32) * BSLAB + sw128_off(n, k % 32)) = B[i];
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    if (warp == 1) {
        if (elect_one()) {
            constexpr uint32_t idesc = make_idesc(128, N) | (1u << 15);                // A MN-major, B K-major
            for (int k8 = 0; k8 < K / 8; ++k8) {
                const uint64_t bdesc = make_desc(smem_u32(b_s) + (k8 / 4) * BSLAB + (k8 % 4) * 32);
                umma_tf32(tmem, make_desc_mn(smem_u32(a_s) + k8 * 1024, ASLAB), bdesc, idesc, k8 > 0);
            }
            umma_commit(&bar);
        }
        __syncwarp();
    }
    mbar_wait_bounded(&bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = warp * 32 + (tid & 31);
    for (int c = 0; c < N; c += 16) {
        float v[16];
        tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c, v);
        for (int i = 0; i < 16; ++i) D[row * N + c + i] = v[i];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(64));
}
template <int N, int K>
static int run_mixed() {
    std::vector<float> A(K * 128), B(N * K), D(128 * N, -1.f), ref(128 * N);
    srand(11);
    for (auto& x : A) x = (float)((rand() % 17) - 8) * 0.25f;
    for (auto& x : B) x = (float)((rand() % 17) - 8) * 0.5f;
    for (int m = 0; m < 128; ++m)
        for (int n = 0; n < N; ++n) {
            double s = 0;
            for (int k = 0; k < K; ++k) s += (double)A[k * 128 + m] * (double)B[n * K + k];
            ref[m * N + n] = (float)s;
        }
    float *dA, *dB, *dD;
    cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, D.size() * 4);
    cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dD, D.data(), D.size() * 4, cudaMemcpyHostToDevice);
    const size_t smem = (size_t)4 * K * 128 + (size_t)(K / 32) * N * 128;
    auto kern = umma_mixed_kernel<N, K>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<1, 128, smem>>>(dA, dB, dD);
    cudaError_t e = cudaDeviceSynchronize();
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    double err = 0;
    for (int i = 0; i < 128 * N; ++i) err = fmax(err, fabs((double)D[i] - (double)ref[i]));
    printf("mixed majors (A MN-major BASE32B, B K-major SWIZZLE_128B) M=128 N=%d K=%d: max|err| = %.3e  %s  %s\n", N, K, err,
           err == 0.0 ? "EXACT" : "WRONG", e == cudaSuccess ? "" : cudaGetErrorString(e));
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
    return e == cudaSuccess ? 0 : 1;
}

int main() {
    if (run_mixed<32, 64>()) return 1;
    run_mn<128, 64, 64>();

    loop_rate<64, 2, 0>(); loop_rate<64, 4, 0>(); loop_rate<64, 2, 7>(); loop_rate<64, 4, 7>();

    rate<128, 16, 1>(); rate<128, 64, 1>(); rate<128, 256, 1>(); rate<64, 64, 1>();
    int rc = 0;
    rc |= run<64, 1, false>("exact  ", true);
    rc |= run<64, 2, false>("exact2 ", true);
    rc |= run<16, 1, false>("exactN16", true);
    rc |= run<64, 4, false>("tf32x1 ", false);
    rc |= run<64, 4, true>("tf32x3 ", false);
    rc |= run<16, 4, true>("tf32x3 N16", false);
    return rc;
}
