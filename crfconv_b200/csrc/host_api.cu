// Host-pointer entry points of the C ABI (include/crfconv_b200.h): the literal drop-ins for the reference's C++
// functions, which take host buffers (knn_.h:13-15; wrapper.cpp:205-229).  They stage through a grow-only
// per-thread device arena, run the device entry points on a private stream and synchronise before returning.
// There is NO CPU fallback: without a CUDA device these calls return CRFCONV_ERR_NO_DEVICE / a cudaError_t.
#include <algorithm>
#include <atomic>
#include <cstring>
#include <thread>
#include <vector>

#include "../../include/crfconv_b200.h"
#include "common.cuh"

namespace {

struct Arena {
    void* ptr = nullptr;
    size_t bytes = 0;
    cudaStream_t stream = nullptr;
    int device = -1;

    int ensure(size_t need) {
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return CRF_ERR_NO_DEVICE; }
        if (dev != device) {   // arena belongs to one device
            if (ptr) cudaFree(ptr);
            ptr = nullptr; bytes = 0;
            if (stream) cudaStreamDestroy(stream);
            stream = nullptr;
            device = dev;
        }
        if (!stream) CRF_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        if (need > bytes) {
            if (ptr) CRF_CUDA(cudaFree(ptr));
            ptr = nullptr; bytes = 0;
            size_t want = crf::align_up(need + need / 4, (size_t)1 << 20);
            CRF_CUDA(cudaMalloc(&ptr, want));
            bytes = want;
        }
        return CRF_OK;
    }
};

thread_local Arena g_arena;

// narrow one contiguous span; returns the OR of all source values (range check by the caller: no branch in the loop, vectorisable)
template <typename T>
uint64_t pack_span(const int64_t* src, T* dst, int64_t n) {
    uint64_t seen = 0;
    for (int64_t i = 0; i < n; ++i) {
        const uint64_t v = (uint64_t)src[i];
        seen |= v;
        dst[i] = (T)v;
    }
    return seen;
}

template <typename T>
__global__ void __launch_bounds__(256) unpack_index_kernel(const T* __restrict__ src, int64_t* __restrict__ dst, int64_t n) {
    // 4 indices per thread: one 8- / 16-byte load, two 128-bit stores
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n) {
        alignas(16) T v[4];
        if constexpr (sizeof(T) == 2) *reinterpret_cast<uint2*>(v) = __ldg(reinterpret_cast<const uint2*>(src + i));
        else *reinterpret_cast<uint4*>(v) = __ldg(reinterpret_cast<const uint4*>(src + i));
        longlong2 a, b;
        a.x = (long long)v[0]; a.y = (long long)v[1]; b.x = (long long)v[2]; b.y = (long long)v[3];
        *reinterpret_cast<longlong2*>(dst + i) = a;
        *reinterpret_cast<longlong2*>(dst + i + 2) = b;
    } else {
        for (int64_t j = i; j < n; ++j) dst[j] = (int64_t)src[j];
    }
}

}  // namespace

using namespace crf;

extern "C" {

int crfconv_abi_version(void) { return 2; }

const char* crfconv_status_string(int status) {
    switch (status) {
        case CRFCONV_OK: return "ok";
        case CRFCONV_ERR_INVALID_ARG: return "invalid argument";
        case CRFCONV_ERR_WORKSPACE: return "workspace too small";
        case CRFCONV_ERR_UNSUPPORTED: return "unsupported configuration";
        case CRFCONV_ERR_NO_DEVICE: return "no CUDA device";
        default: return status > 0 ? cudaGetErrorString((cudaError_t)status) : "unknown status";
    }
}

int crfconv_pack_index_host(const int64_t* idx, int64_t n, int bits, void* out, int threads) {
    if (n < 0 || (bits != 16 && bits != 32)) return CRF_ERR_INVALID_ARG;
    if (n == 0) return CRF_OK;
    if (!idx || !out) return CRF_ERR_INVALID_ARG;
    const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(threads, 64), n >> 16));   // >= 64 Ki indices per thread
    std::atomic<uint64_t> seen{0};
    auto work = [&](int t) {
        const int64_t per = ((n + nt - 1) / nt + 15) & ~(int64_t)15, lo = std::min(n, per * t), hi = std::min(n, lo + per);
        const uint64_t s = bits == 16 ? pack_span(idx + lo, (uint16_t*)out + lo, hi - lo) : pack_span(idx + lo, (uint32_t*)out + lo, hi - lo);
        seen.fetch_or(s, std::memory_order_relaxed);
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
    // a negative index has bit 63 set, one that does not fit has a bit at or above `bits`: either shows up in the OR
    return (seen.load() >> bits) ? CRF_ERR_INVALID_ARG : CRF_OK;
}

int crfconv_unpack_index(const void* packed, int64_t n, int bits, int64_t* out, void* stream) {
    if (n < 0 || (bits != 16 && bits != 32)) return CRF_ERR_INVALID_ARG;
    if (n == 0) return CRF_OK;
    if (!packed || !out || (reinterpret_cast<uintptr_t>(packed) & 15) || (reinterpret_cast<uintptr_t>(out) & 15)) return CRF_ERR_INVALID_ARG;
    const unsigned grid = (unsigned)((n + 1023) / 1024);
    if (bits == 16) unpack_index_kernel<uint16_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)packed, out, n);
    else unpack_index_kernel<uint32_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)packed, out, n);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

int crfconv_cpp_knn_batch(const float* batch_data, size_t batch_size, size_t npts, size_t dim, const float* queries,
                          size_t nqueries, size_t K, int64_t* batch_indices) {
    if (dim != 3) return CRF_ERR_UNSUPPORTED;
    if (batch_size == 0 || nqueries == 0 || K == 0) return CRF_OK;
    if (!batch_data || !queries || !batch_indices || npts == 0) return CRF_ERR_INVALID_ARG;
    if (K > 1024) return CRF_ERR_UNSUPPORTED;
    const int64_t B = (int64_t)batch_size, N = (int64_t)npts, Q = (int64_t)nqueries, Kk = (int64_t)K;
    const size_t pts_b = align_up((size_t)B * N * 3 * sizeof(float), 256);
    const size_t q_b = align_up((size_t)B * Q * 3 * sizeof(float), 256);
    const size_t out_b = align_up((size_t)B * Q * Kk * sizeof(int64_t), 256);
    const size_t ws_b = crfconv_knn_workspace_bytes(B, N, Q, Kk);
    int rc = g_arena.ensure(pts_b + q_b + out_b + ws_b);
    if (rc != CRF_OK) return rc;
    char* base = (char*)g_arena.ptr;
    float* d_pts = (float*)base;
    float* d_q = (float*)(base + pts_b);
    int64_t* d_out = (int64_t*)(base + pts_b + q_b);
    void* d_ws = base + pts_b + q_b + out_b;
    cudaStream_t st = g_arena.stream;
    CRF_CUDA(cudaMemcpyAsync(d_pts, batch_data, (size_t)B * N * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    const bool same = (queries == batch_data) && (Q == N);
    if (!same) CRF_CUDA(cudaMemcpyAsync(d_q, queries, (size_t)B * Q * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
    rc = crfconv_knn_batch(d_pts, B, N, same ? d_pts : d_q, Q, Kk, d_out, d_ws, ws_b, st);
    if (rc != CRF_OK) return rc;
    CRF_CUDA(cudaMemcpyAsync(batch_indices, d_out, (size_t)B * Q * Kk * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CRF_CUDA(cudaStreamSynchronize(st));
    return CRF_OK;
}

int crfconv_grid_subsample_host(const float* points, int64_t N, const float* features, int64_t fdim,
                                const int32_t* classes, int64_t ldim, float sampleDl, int order, float* out_points,
                                float* out_features, int32_t* out_classes, int64_t* M_out) {
    if (!M_out) return CRF_ERR_INVALID_ARG;
    *M_out = 0;
    if (N < 0 || fdim < 0 || ldim < 0) return CRF_ERR_INVALID_ARG;
    if (N == 0) return CRF_OK;
    if (!points || !out_points) return CRF_ERR_INVALID_ARG;
    if (!features) fdim = 0;
    if (!classes) ldim = 0;
    const size_t p_b = align_up((size_t)N * 3 * 4, 256), f_b = align_up((size_t)N * std::max<int64_t>(fdim, 1) * 4, 256),
                 c_b = align_up((size_t)N * std::max<int64_t>(ldim, 1) * 4, 256);
    const size_t ws_b = crfconv_grid_subsample_workspace_bytes(N, fdim, ldim);
    int rc = g_arena.ensure(2 * (p_b + f_b + c_b) + ws_b);
    if (rc != CRF_OK) return rc;
    char* base = (char*)g_arena.ptr;
    float* d_p = (float*)base;           base += p_b;
    float* d_f = (float*)base;           base += f_b;
    int32_t* d_c = (int32_t*)base;       base += c_b;
    float* d_op = (float*)base;          base += p_b;
    float* d_of = (float*)base;          base += f_b;
    int32_t* d_oc = (int32_t*)base;      base += c_b;
    void* d_ws = base;
    cudaStream_t st = g_arena.stream;
    CRF_CUDA(cudaMemcpyAsync(d_p, points, (size_t)N * 3 * 4, cudaMemcpyHostToDevice, st));
    if (fdim) CRF_CUDA(cudaMemcpyAsync(d_f, features, (size_t)N * fdim * 4, cudaMemcpyHostToDevice, st));
    if (ldim) CRF_CUDA(cudaMemcpyAsync(d_c, classes, (size_t)N * ldim * 4, cudaMemcpyHostToDevice, st));
    int64_t M = 0;
    rc = crfconv_grid_subsample(d_p, N, fdim ? d_f : nullptr, fdim, ldim ? d_c : nullptr, ldim, sampleDl, order, d_op,
                                fdim ? d_of : nullptr, ldim ? d_oc : nullptr, nullptr, &M, d_ws, ws_b, st);
    if (rc != CRF_OK) return rc;
    CRF_CUDA(cudaMemcpyAsync(out_points, d_op, (size_t)M * 3 * 4, cudaMemcpyDeviceToHost, st));
    if (fdim && out_features) CRF_CUDA(cudaMemcpyAsync(out_features, d_of, (size_t)M * fdim * 4, cudaMemcpyDeviceToHost, st));
    if (ldim && out_classes) CRF_CUDA(cudaMemcpyAsync(out_classes, d_oc, (size_t)M * ldim * 4, cudaMemcpyDeviceToHost, st));
    CRF_CUDA(cudaStreamSynchronize(st));
    *M_out = M;
    return CRF_OK;
}

}  // extern "C"
