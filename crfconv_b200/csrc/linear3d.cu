// Input gradient of a Linear layer on the 5th-generation tensor cores:  [dX1 | dX2] (+)= dH · W,  dH = BatchNorm(+LeakyReLU)-backward
// transform of dY applied on the fly (linear_args.cuh DgradArgs; same contract as dgrad2_kernel / dgrad_kernel).
// Same machinery as the forward kernel (linear3.cu): persistent CTA per SM, producer groups → 3-slot ring of K-major SWIZZLE_128B
// slabs → one issuing lane (tcgen05.mma kind::tf32, M = 128, 3xTF32) → two TMEM accumulator buffers → epilogue warps.
//   A = dH tile [128 rows × Cout] (K = Cout, ≤ 2 slabs of 32 channels), built by the producers from dY and H;
//   B = Wᵀ [N = input channels (≤ 128) × K = Cout], split once per CTA;
//   D = [128 rows × N] → dX1 (first C1 columns) and dX2 (the rest), written through a 64-column staging buffer in coalesced rows,
//       optionally accumulated onto the destination (residual / concat branches).
// What bounds it: rows × (2·Cout + Ktot) × 4 bytes of HBM traffic (dY, H read; dX written).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "linear_args.cuh"
#include "umma.cuh"

namespace crf {
namespace lin3d {

using lin::DgradArgs;
using namespace umma;

constexpr int kEpiWarps = 4, kProdWarps = 12, kGroupWarps = 4, kGroups = kProdWarps / kGroupWarps;
constexpr int kThreads = (kEpiWarps + 1 + kProdWarps) * 32;      // 544
constexpr int kRowsPerPass = kGroupWarps * 4;                    // 16
constexpr int kLoadsPerSlab = 128 / kRowsPerPass;                // 8 float4 per thread, slab and array
constexpr int BM = 128, BK = 32, RING = 3;
static_assert(kGroups == RING, "group g owns ring slot g");
constexpr int kSlabBytes = BM * 128, kSlotBytes = 2 * kSlabBytes;
constexpr int kStageCols = 64, kStageLd = kStageCols + 4;        // the epilogue handles the accumulator in column blocks of 64
constexpr int BN = 128;                                          // N = input channels, padded (64 < Ktot <= 128)
constexpr uint32_t kTmemCols = 2 * BN;
inline size_t smem_bytes(int nch) {
    return (size_t)RING * kSlotBytes + (size_t)2 * nch * BN * 128 + (size_t)BM * kStageLd * 4 + (size_t)4 * nch * BK * 4 + (size_t)(2 * RING + 4) * 8 + 16;
}

__global__ void __launch_bounds__(kThreads, 1) dgrad3_kernel(const DgradArgs a, const int ntiles) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int C = a.Cout, Ktot = a.C1 + a.C2;
    const int nch = (C + BK - 1) / BK, Kpad = nch * BK;               // K dimension = output channels of the layer
    uint8_t* ring = smem;
    uint8_t* w_hi = ring + RING * kSlotBytes;                          // [nch][BN rows × 128 B]: Wᵀ, row n = input channel
    uint8_t* w_lo = w_hi + nch * BN * 128;
    float* stage = reinterpret_cast<float*>(w_lo + nch * BN * 128);    // [BM][64 + 4]
    float* s_par = stage + BM * kStageLd;                              // [4][Kpad]: sc, sh, pz, pw of the BN-backward transform
    uint64_t* full = reinterpret_cast<uint64_t*>(s_par + 4 * Kpad);
    uint64_t* empty = full + RING;
    uint64_t* tfull = empty + RING;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool plain = a.bn.scale == nullptr;
    if (warp == 0) tmem_alloc(tmem_slot, kTmemCols);
    if (tid == kEpiWarps * 32) {
        for (int i = 0; i < RING; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, kEpiWarps); }
        mbar_init_fence();
    }
    {   // B[n][k] = W[k][n]: loads batched ahead of their uses
        constexpr int WPT = (BN * 64 + kThreads - 1) / kThreads;       // Kpad <= 64
        float wv[WPT];
        const int total = BN * Kpad;
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * kThreads;
            float w = 0.f;
            if (e < total) {
                const int k = e / BN, n = e - k * BN;                  // consecutive threads → consecutive n: coalesced rows of W
                if (k < C && n < Ktot) w = __ldg(a.W + (int64_t)k * Ktot + n);
            }
            wv[i] = w;
        }
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * kThreads;
            if (e < total) {
                const int k = e / BN, n = e - k * BN, c = k / BK, kk = k % BK;
                float hi, lo;
                split_tf32(wv[i], hi, lo);
                const uint32_t off = (uint32_t)(c * BN * 128) + slab_chunk_off(n, kk >> 2) + ((kk & 3) << 2);
                *reinterpret_cast<float*>(w_hi + off) = hi;
                *reinterpret_cast<float*>(w_lo + off) = lo;
            }
        }
    }
    for (int k = tid; k < Kpad; k += kThreads) {
        const float4 p = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);
        s_par[k] = p.x; s_par[Kpad + k] = p.y; s_par[2 * Kpad + k] = p.z; s_par[3 * Kpad + k] = p.w;
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp > kEpiWarps) {
        // ===================================================================== producers: dH slabs from dY (and H)
        const int g = (warp - (kEpiWarps + 1)) / kGroupWarps;
        const int t = tid - (kEpiWarps + 1) * 32 - g * (kGroupWarps * 32);
        const int c4 = t & 7, rb = t >> 3;
        const int Q = my_tiles * nch;
        uint8_t* hi_slab = ring + g * kSlotBytes;
        const float slope = a.bn.slope;
        for (int q = g; q < Q; q += kGroups) {
            const int lt = q / nch, lc = q - lt * nch;
            const uint32_t use = (uint32_t)(q / RING);
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)lt * gridDim.x) * BM;
            const int col = lc * BK + 4 * c4;
            const bool cok = col < C;
            const int64_t left = a.M - m0 - rb;
            const int64_t base = (m0 + rb) * C + col;
            float4 dv[kLoadsPerSlab], hv[kLoadsPerSlab];
#pragma unroll
            for (int j = 0; j < kLoadsPerSlab; ++j) {
                const bool ok = cok && (kRowsPerPass * j < left);
                const int64_t off = ok ? base + (int64_t)(kRowsPerPass * j) * C : 0;
                dv[j] = ok ? __ldg(reinterpret_cast<const float4*>(a.dY + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                hv[j] = (ok && !plain) ? __ldg(reinterpret_cast<const float4*>(a.H + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (!plain) {
                const float4 sc = *reinterpret_cast<const float4*>(s_par + col), sh = *reinterpret_cast<const float4*>(s_par + Kpad + col);
                const float4 pz = *reinterpret_cast<const float4*>(s_par + 2 * Kpad + col), pw = *reinterpret_cast<const float4*>(s_par + 3 * Kpad + col);
#pragma unroll
                for (int j = 0; j < kLoadsPerSlab; ++j) {
                    const bool ok = cok && (kRowsPerPass * j < left);
                    const float4 d = dv[j], h = hv[j];
                    float4 o;
                    o.x = fmaf(sc.x, fmaf(h.x, sc.x, sh.x) > 0.f ? d.x : d.x * slope, fmaf(pz.x, h.x, pw.x));
                    o.y = fmaf(sc.y, fmaf(h.y, sc.y, sh.y) > 0.f ? d.y : d.y * slope, fmaf(pz.y, h.y, pw.y));
                    o.z = fmaf(sc.z, fmaf(h.z, sc.z, sh.z) > 0.f ? d.z : d.z * slope, fmaf(pz.z, h.z, pw.z));
                    o.w = fmaf(sc.w, fmaf(h.w, sc.w, sh.w) > 0.f ? d.w : d.w * slope, fmaf(pz.w, h.w, pw.w));
                    dv[j] = ok ? o : make_float4(0.f, 0.f, 0.f, 0.f);      // the additive terms must not leak into padding rows / columns
                }
            }
            mbar_wait_relaxed(empty + g, (use & 1) ^ 1);
#pragma unroll
            for (int j = 0; j < kLoadsPerSlab; ++j) {
                float4 h, l;
                split_tf32(dv[j].x, h.x, l.x); split_tf32(dv[j].y, h.y, l.y); split_tf32(dv[j].z, h.z, l.z); split_tf32(dv[j].w, h.w, l.w);
                const uint32_t off = slab_chunk_off(rb + kRowsPerPass * j, c4);
                *reinterpret_cast<float4*>(hi_slab + off) = h;
                *reinterpret_cast<float4*>(hi_slab + kSlabBytes + off) = l;
            }
            asm volatile("bar.sync %0, %1;" ::"r"(2 + g), "n"(kGroupWarps * 32) : "memory");
            if (t == 0) mbar_arrive(full + g);
        }
    } else if (warp == kEpiWarps) {
        // ===================================================================== MMA issuer
        constexpr uint32_t idesc = idesc_tf32(BM, BN);
        const uint64_t a_desc0 = smem_desc_k128(smem_u32(ring));
        const uint64_t bh_desc0 = smem_desc_k128(smem_u32(w_hi)), bl_desc0 = smem_desc_k128(smem_u32(w_lo));
        int slot = 0;
        uint32_t use = 0;
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int buf = ti & 1;
            mbar_wait(tempty + buf, ((uint32_t)(ti >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d = tmem + (uint32_t)(buf * BN);
            for (int c = 0; c < nch; ++c) {
                mbar_wait(full + slot, use & 1);
                fence_async_smem();                                      // producers' generic-proxy stores → async proxy
                tc_fence_after();
                const int nk8 = (min(BK, C - c * BK) + 7) >> 3;
                if (elect_one()) {
                    const uint64_t ah0 = a_desc0 + (uint64_t)(slot * (kSlotBytes / 16)), al0 = ah0 + kSlabBytes / 16;
                    const uint64_t bh0 = bh_desc0 + (uint64_t)(c * (BN * 128 / 16)), bl0 = bl_desc0 + (uint64_t)(c * (BN * 128 / 16));
#pragma unroll
                    for (int k8 = 0; k8 < 4; ++k8) {
                        if (k8 < nk8) {
                            mma_tf32(d, al0 + 2 * k8, bh0 + 2 * k8, idesc, (c | k8) != 0);
                            mma_tf32(d, ah0 + 2 * k8, bl0 + 2 * k8, idesc, 1);
                            mma_tf32(d, ah0 + 2 * k8, bh0 + 2 * k8, idesc, 1);
                        }
                    }
                    mma_commit(empty + slot);
                    if (c == nch - 1) mma_commit(tfull + buf);
                }
                if (++slot == RING) { slot = 0; ++use; }
            }
        }
    } else {
        // ===================================================================== epilogue: [128 × BN] accumulator → dX1 | dX2
        const int row = tid;
        constexpr int CB = BN < kStageCols ? BN : kStageCols;            // columns per staging pass
        constexpr int CH = CB / 4, RPP = BM / CH;
        const int ochunk = tid % CH, orow = tid / CH;
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int buf = ti & 1;
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
            const int valid = (int)min((int64_t)BM, a.M - m0);
            mbar_wait_relaxed(tfull + buf, (uint32_t)(ti >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int n0 = 0; n0 < BN; n0 += CB) {
                {
                    uint32_t v[CB / 16][16];
#pragma unroll
                    for (int cb = 0; cb < CB / 16; ++cb) tmem_ld16_issue(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * BN + n0 + cb * 16), v[cb]);
                    tmem_ld_wait();
                    if (n0 + CB >= BN) {                                 // last column block read: the accumulator buffer is free
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(tempty + buf);
                    }
#pragma unroll
                    for (int cb = 0; cb < CB / 16; ++cb)
#pragma unroll
                        for (int i = 0; i < 16; i += 4)
                            *reinterpret_cast<float4*>(stage + row * kStageLd + cb * 16 + i) =
                                make_float4(__uint_as_float(v[cb][i]), __uint_as_float(v[cb][i + 1]), __uint_as_float(v[cb][i + 2]), __uint_as_float(v[cb][i + 3]));
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                const int n = n0 + 4 * ochunk;                           // input-channel index of this thread's 16-byte chunk
                float* dst = nullptr;
                int ld = 0, acc = 0;
                if (n < a.C1) { if (a.dX1) { dst = a.dX1 + n; ld = a.C1; acc = a.acc1; } }
                else if (n < Ktot) { if (a.dX2) { dst = a.dX2 + (n - a.C1); ld = a.C2; acc = a.acc2; } }
                if (dst) {
                    for (int r = orow; r < valid; r += RPP) {
                        float4 o = *reinterpret_cast<const float4*>(stage + r * kStageLd + 4 * ochunk);
                        float* p = dst + (m0 + r) * ld;
                        if (acc) { const float4 old = *reinterpret_cast<const float4*>(p); o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
                        *reinterpret_cast<float4*>(p) = o;
                    }
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

}  // namespace lin3d

namespace lin {

int try_dgrad3(const DgradArgs& a, int precision, cudaStream_t st) {
    using namespace lin3d;
    if (precision != 0) return kDeclined;
    const int Ktot = a.C1 + a.C2;
    if (a.Cout > 64 || (a.Cout & 3) || Ktot > BN || (a.C1 & 3) || (a.C2 & 3) || a.bn.act_ref) return kDeclined;
    if (!aligned16(a.dY) || (a.bn.scale && !aligned16(a.H))) return kDeclined;
    if ((a.dX1 && !aligned16(a.dX1)) || (a.dX2 && !aligned16(a.dX2))) return kDeclined;
    if (!a.dX1 && !a.dX2) return kDeclined;
    if (Ktot <= 64 || a.Cout <= 32) return kDeclined;  // narrower products: the mma.sync kernel is as fast or faster (measured)
    const int ntiles = (int)ceil_div(a.M, BM);
    if (ntiles <= 0) return kDeclined;
    return launch(dgrad3_kernel, dim3(std::min(ntiles, kNumSMs)), dim3(kThreads), smem_bytes((a.Cout + BK - 1) / BK), st, a, ntiles);
}

}  // namespace lin
}  // namespace crf
