// Weight gradient of a Linear layer on the 5th-generation tensor cores:
//     dWᵀ[k, co] = Σ_rows Xin[r, k] · dH[r, co]        (Xin = [lrelu(X1·scale1+shift1) | X2], dH = BatchNorm-backward transform of dY)
// The contraction runs over ROWS, so both operands are "MN-major" for tcgen05.mma: an activation tile is stored row by row
// exactly as it lies in global memory, and one MMA (kind::tf32, K = 8) consumes 8 rows of it.  tf32 MN-major operands exist
// only in the SWIZZLE_128B_BASE32B shared-memory layout (validated in scripts/micro/umma_test.cu): a block is [rows][32
// channels], one 128-byte line per row, the 32-byte chunk c of row r stored at chunk position c ^ (r & 3); 4-row atoms are
// 512 B apart (descriptor SBO), 32-channel blocks one block apart (LBO).  A = Xin (M = input channels, padded to 128 with
// blocks that stay zero), B = dH (N = Cout padded to 32 / 64), D = dWᵀ accumulates in TMEM over ALL the tiles of the CTA and is
// read out once at the end into the caller's weight-gradient partial slot.  3xTF32 (hi·hi + hi·lo + lo·hi) for fp32 parity.
//
// Persistent CTA per SM, 64-row stages, two stages in shared memory (2 × 96 KB for 128 input / 64 output channels):
//   warps 5..16  producers : 6 groups of 2 warps.  A stage is cut into tasks of [32 rows × 32 channels] (X blocks with the
//                            BatchNorm+LeakyReLU prologue, dH blocks with the BN-backward transform of dY / H); group g takes
//                            task g and g + 6 of EVERY stage (so every group is at most one mbarrier phase behind), loads into
//                            registers (next task's loads in flight), waits for the stage, writes hi / lo, arrives on the stage barrier;
//   warp 4       issuer    : per stage 8 row groups × 3 MMAs (M = 128, N = 32 / 64), tcgen05.commit releases the stage;
//   warps 0..3   epilogue  : once per CTA, tcgen05.ld of dWᵀ and atomic adds into dW[slot][co][k].
// What bounds it: reading dY, H and X once from HBM (rows × (2·Cout + Ktot) × 4 bytes).
#include <algorithm>

#include "common.cuh"
#include "linear_args.cuh"
#include "umma.cuh"

namespace crf {
namespace lin3w {

using lin::WgradArgs;
using lin::lrelu;
using namespace umma;

constexpr int kEpiWarps = 4, kProdWarps = 12, kGroupWarps = 2, kGroups = kProdWarps / kGroupWarps;
constexpr int kThreads = (kEpiWarps + 1 + kProdWarps) * 32;      // 544
constexpr int RS = 64;                                           // rows per stage
constexpr int kBlockBytes = RS * 128;                            // one [64 rows × 32 channels] fp32 block
constexpr int kXBlocks = 4;                                      // M = 128 input channels (zero blocks beyond Ktot)

template <int BN>
struct Layout {
    static constexpr int NB = BN / 32;                                        // dH blocks
    static constexpr int kStageBytes = 2 * (kXBlocks + NB) * kBlockBytes;     // [X hi ×4][X lo ×4][dH hi ×NB][dH lo ×NB]
    static constexpr uint32_t kTmemCols = BN;
    static size_t bytes() { return (size_t)2 * kStageBytes + (size_t)(4 * BN + 2 * 128) * 4 + 8 * 8 + 16; }
};

template <int BN>
__global__ void __launch_bounds__(kThreads, 1) wgrad3_kernel(const WgradArgs a, const int ntiles) {
    using L = Layout<BN>;
    constexpr int NB = L::NB;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* stage0 = smem;                                                   // 2 stages
    float* s_par = reinterpret_cast<float*>(smem + 2 * L::kStageBytes);       // [4][BN]: sc, sh, pz, pw of the BN-backward transform
    float* s_sc = s_par + 4 * BN;                                             // [128] prologue scale per padded input column
    float* s_sh = s_sc + 128;
    uint64_t* full = reinterpret_cast<uint64_t*>(s_sh + 128);                 // [2] producers → issuer
    uint64_t* empty = full + 2;                                               // [2] issuer (commit) → producers
    uint64_t* done = empty + 2;                                               // accumulator final
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nch1 = (a.C1 + 31) / 32, nch2 = (a.C2 + 31) / 32, nchX = nch1 + nch2;
    const int C = a.Cout, Ktot = a.C1 + a.C2;
    const int T = 2 * (nchX + NB);                                            // tasks per stage
    const bool plain = a.bn.scale == nullptr;

    if (warp == 0) tmem_alloc(tmem_slot, L::kTmemCols);
    if (tid == kEpiWarps * 32) {
        for (int i = 0; i < 2; ++i) { mbar_init(full + i, (uint32_t)T); mbar_init(empty + i, 1); }
        mbar_init(done, 1);
        mbar_init_fence();
    }
    for (int k = tid; k < BN; k += kThreads) {
        const float4 p = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);
        s_par[k] = p.x; s_par[BN + k] = p.y; s_par[2 * BN + k] = p.z; s_par[3 * BN + k] = p.w;
    }
    for (int k = tid; k < 128; k += kThreads) {
        float sc = 1.f, sh = 0.f;
        if (a.scale1 && k < nch1 * 32 && k < a.C1) { sc = __ldg(a.scale1 + k); sh = __ldg(a.shift1 + k); }
        s_sc[k] = sc; s_sh[k] = sh;
    }
    // input-channel blocks beyond nchX are never written: they must read as zeros for the whole kernel
    for (int i = tid; i < 2 * L::kStageBytes / 16; i += kThreads) reinterpret_cast<float4*>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp > kEpiWarps) {
        // ===================================================================== producers
        const int g = (warp - (kEpiWarps + 1)) / kGroupWarps;
        const int t = tid - (kEpiWarps + 1) * 32 - g * (kGroupWarps * 32);
        const int c16 = t & 7, rb = t >> 3;                                   // 16-byte chunk of the 32-channel block; rows rb + 8 j
        const float slope1 = a.scale1 ? a.slope1 : 1.0f, slope = a.bn.slope;
        constexpr int NJ = 32 / (4 * kGroupWarps), RJ = 4 * kGroupWarps;      // rows per thread in a 32-row task, row step
        // raw loads of one task: X rows, or dY (+ H) rows
        auto load = [&](int ti, int task, float4 (&v)[NJ], float4 (&hh)[NJ]) {
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * RS;
            const int half = task & 1, blk = task >> 1, r0 = 32 * half + rb;
            if (blk < nchX) {
                const bool seg1 = blk < nch1;
                const float* X = seg1 ? a.X1 : a.X2;
                const int Cs = seg1 ? a.C1 : a.C2;
                const int col = (seg1 ? blk : blk - nch1) * 32 + 4 * c16;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int64_t m = m0 + r0 + RJ * j;
                    v[j] = (col < Cs && m < a.M) ? __ldg(reinterpret_cast<const float4*>(X + m * Cs + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            } else {
                const int col = 32 * (blk - nchX) + 4 * c16;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int64_t m = m0 + r0 + RJ * j;
                    const bool ok = col < C && m < a.M;
                    const int64_t off = ok ? m * C + col : 0;
                    v[j] = ok ? __ldg(reinterpret_cast<const float4*>(a.dY + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    hh[j] = (ok && !plain) ? __ldg(reinterpret_cast<const float4*>(a.H + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        };
        // transform in registers, wait for the stage, write hi / lo, publish.  No fence.proxy.async here (its MEMBAR would wait
        // for the loads of the next task that are already in flight): the issuer fences after acquiring the stage.
        auto publish = [&](int ti, int task, float4 (&v)[NJ], float4 (&hh)[NJ]) {
            const int st = ti & 1;
            const uint32_t use = (uint32_t)(ti >> 1);
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * RS;
            const int half = task & 1, blk = task >> 1, r0 = 32 * half + rb;
            uint8_t* sbase = stage0 + st * L::kStageBytes;
            uint8_t* dst_hi;
            int lo_off;
            if (blk < nchX) {
                if (blk < nch1 && a.scale1) {
                    const bool cok = blk * 32 + 4 * c16 < a.C1;
                    const float4 sc = *reinterpret_cast<const float4*>(s_sc + blk * 32 + 4 * c16);
                    const float4 sh = *reinterpret_cast<const float4*>(s_sh + blk * 32 + 4 * c16);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const bool ok = cok && (m0 + r0 + RJ * j < a.M);      // the prologue's shift must not leak into padding
                        v[j] = ok ? make_float4(lrelu(fmaf(v[j].x, sc.x, sh.x), slope1), lrelu(fmaf(v[j].y, sc.y, sh.y), slope1),
                                                lrelu(fmaf(v[j].z, sc.z, sh.z), slope1), lrelu(fmaf(v[j].w, sc.w, sh.w), slope1))
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                dst_hi = sbase + blk * kBlockBytes;                           // lo copy kXBlocks blocks further
                lo_off = kXBlocks * kBlockBytes;
            } else {
                const int b = blk - nchX, col = 32 * b + 4 * c16;
                if (!plain) {
                    const bool cok = col < C;
                    const float4 sc = *reinterpret_cast<const float4*>(s_par + col), sh = *reinterpret_cast<const float4*>(s_par + BN + col);
                    const float4 pz = *reinterpret_cast<const float4*>(s_par + 2 * BN + col), pw = *reinterpret_cast<const float4*>(s_par + 3 * BN + col);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const bool ok = cok && (m0 + r0 + RJ * j < a.M);
                        const float4 d = v[j], h = hh[j];
                        const float4 pre = make_float4(fmaf(h.x, sc.x, sh.x), fmaf(h.y, sc.y, sh.y), fmaf(h.z, sc.z, sh.z), fmaf(h.w, sc.w, sh.w));
                        float4 o;
                        o.x = fmaf(sc.x, pre.x > 0.f ? d.x : d.x * slope, fmaf(pz.x, h.x, pw.x));
                        o.y = fmaf(sc.y, pre.y > 0.f ? d.y : d.y * slope, fmaf(pz.y, h.y, pw.y));
                        o.z = fmaf(sc.z, pre.z > 0.f ? d.z : d.z * slope, fmaf(pz.z, h.z, pw.z));
                        o.w = fmaf(sc.w, pre.w > 0.f ? d.w : d.w * slope, fmaf(pz.w, h.w, pw.w));
                        v[j] = ok ? o : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                dst_hi = sbase + (2 * kXBlocks + b) * kBlockBytes;            // lo copy NB blocks further
                lo_off = NB * kBlockBytes;
            }
            // every group has a task in every stage, so it is at most one phase behind the stage barriers (parity is enough)
            mbar_wait_relaxed(empty + st, (use & 1) ^ 1);
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                float4 h, l;
                split_tf32(v[j].x, h.x, l.x); split_tf32(v[j].y, h.y, l.y); split_tf32(v[j].z, h.z, l.z); split_tf32(v[j].w, h.w, l.w);
                const uint32_t off = blk_off(r0 + RJ * j, c16);
                *reinterpret_cast<float4*>(dst_hi + off) = h;
                *reinterpret_cast<float4*>(dst_hi + lo_off + off) = l;
            }
            asm volatile("bar.sync %0, %1;" ::"r"(2 + g), "n"(kGroupWarps * 32) : "memory");
            if (t == 0) mbar_arrive(full + st);
        };
        // group g owns tasks g and g + kGroups of every stage; one task's loads are always in flight behind the other's conversion
        const int t0 = g, t1 = g + kGroups;
        float4 vA[NJ], hA[NJ], vB[NJ], hB[NJ];
        if (my_tiles > 0) {
            if (t0 < T) load(0, t0, vA, hA);
            if (t1 < T) load(0, t1, vB, hB);
        }
        for (int ti = 0; ti < my_tiles; ++ti) {
            if (t0 < T) publish(ti, t0, vA, hA);
            if (t0 < T && ti + 1 < my_tiles) load(ti + 1, t0, vA, hA);
            if (t1 < T) publish(ti, t1, vB, hB);
            if (t1 < T && ti + 1 < my_tiles) load(ti + 1, t1, vB, hB);
        }
    } else if (warp == kEpiWarps) {
        // ===================================================================== MMA issuer
        constexpr uint32_t idesc = idesc_tf32(128, BN) | (1u << 15) | (1u << 16);     // A and B MN-major
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int st = ti & 1;
            mbar_wait(full + st, (uint32_t)(ti >> 1) & 1);
            fence_async_smem();                                              // producers' generic-proxy stores → async proxy
            tc_fence_after();
            if (elect_one()) {
                const uint32_t sb = smem_u32(stage0 + st * L::kStageBytes);
                const uint64_t xh = desc_mn(sb, kBlockBytes), xl = desc_mn(sb + kXBlocks * kBlockBytes, kBlockBytes);
                const uint64_t dh = desc_mn(sb + 2 * kXBlocks * kBlockBytes, kBlockBytes), dl = desc_mn(sb + (2 * kXBlocks + NB) * kBlockBytes, kBlockBytes);
#pragma unroll
                for (int j = 0; j < RS / 8; ++j) {                            // 8 rows = 1024 bytes = 64 descriptor units per step
                    mma_tf32(tmem, xl + 64 * j, dh + 64 * j, idesc, (ti | j) != 0);
                    mma_tf32(tmem, xh + 64 * j, dl + 64 * j, idesc, 1);
                    mma_tf32(tmem, xh + 64 * j, dh + 64 * j, idesc, 1);
                }
                mma_commit(empty + st);
                if (ti == my_tiles - 1) mma_commit(done);
            }
            __syncwarp();
        }
    } else {
        // ===================================================================== epilogue: dWᵀ rows (input channel k) × columns (co)
        mbar_wait_relaxed(done, 0);
        tc_fence_after();
        const int kp = tid;                                                    // padded input-channel index = TMEM lane
        const int chunk = kp >> 5, kk = kp & 31;
        int col = -1;
        if (chunk < nch1) { if (chunk * 32 + kk < a.C1) col = chunk * 32 + kk; }
        else if (chunk < nchX && (chunk - nch1) * 32 + kk < a.C2) col = a.C1 + (chunk - nch1) * 32 + kk;
        float* dst = a.dW + a.slot_stride * (int64_t)(blockIdx.x % kGradSlots);
#pragma unroll
        for (int c0 = 0; c0 < BN; c0 += 16) {
            float v[16];
            tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
            if (col >= 0) {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (c0 + i < C) atomicAdd(dst + (int64_t)(c0 + i) * Ktot + col, v[i]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, L::kTmemCols);
}

}  // namespace lin3w

namespace lin {

int try_wgrad3(const WgradArgs& a, int precision, cudaStream_t st) {
    using namespace lin3w;
    if (precision != 0) return kDeclined;
    if (a.idx1 || a.dbias || a.bn.act_ref) return kDeclined;
    if (a.Cout > 64 || (a.Cout & 3) || (a.C1 & 3) || (a.C2 & 3) || a.C1 <= 0) return kDeclined;
    if ((a.C1 + 31) / 32 + (a.C2 + 31) / 32 > kXBlocks) return kDeclined;
    if (a.C1 + a.C2 <= 64) return kDeclined;    // narrow inputs: M is padded to 128 anyway and the mma.sync kernels are as fast (measured)
    if (!aligned16(a.dY) || !aligned16(a.X1) || (a.C2 && !aligned16(a.X2))) return kDeclined;
    if (a.bn.scale && !aligned16(a.H)) return kDeclined;
    const int ntiles = (int)ceil_div(a.M, RS);
    if (ntiles <= 0) return kDeclined;
    const dim3 grid(std::min(ntiles, kNumSMs));
    if (a.Cout > 32) return launch(wgrad3_kernel<64>, grid, dim3(kThreads), Layout<64>::bytes(), st, a, ntiles);
    return launch(wgrad3_kernel<32>, grid, dim3(kThreads), Layout<32>::bytes(), st, a, ntiles);
}

}  // namespace lin
}  // namespace crf
