// Input AND weight gradient of a Linear layer in one pass on the 5th-generation tensor cores (linear_args.cuh DgradArgs +
// WgradArgs, the contract of dgrad3_kernel + wgrad3_kernel):
//     dWᵀ[k, co] += Σ_rows Xin[r, k] · dH[r, co]        dXᵀ[k, r] = Σ_co W[co, k] · dH[r, co]
// (Xin = [lrelu(X1·scale1+shift1) | X2], dH = BatchNorm(+LeakyReLU)-backward transform of dY).  Both products are written with
// M = 128 = input channels, so dY, H, X1 and X2 are read from HBM once and dH is computed and split once:
//   weight gradient : A = Xin (MN-major SWIZZLE_128B_BASE32B blocks, K = rows), B = dH (same layout, N = Cout), D = dWᵀ in TMEM
//                     for all the CTA's tiles (exactly wgrad3_kernel);
//   input gradient  : A = Wᵀ (W is [Cout][Ktot]: channel-contiguous, stored as the same MN-major blocks with lines = Cout, split
//                     once per CTA, resident), B = dH with N = rows and K = Cout (K-major SWIZZLE_128B slabs: a second copy of the
//                     stage's dH), D = dXᵀ [128 channels × 32 rows], double-buffered in TMEM.
// The two B operands differ in their major-ness, so the producers store dH twice; the input-gradient MMA mixes an MN-major A with
// a K-major B (instruction-descriptor bit 15 only; validated in scripts/micro/umma_test.cu).  3xTF32 (hi·hi + hi·lo + lo·hi) in two
// MMAs per k-step: in both dH copies dH_lo lies behind dH_hi along N, so hi·[dH_hi | dH_lo] is ONE MMA with N doubled and lo·dH_hi
// accumulates onto its first half; the epilogue adds the two halves (operand fetch 56 + 88 KB per 32 rows instead of 72 + 120).
//
// Persistent CTA per SM, 32-row stages, two stages in shared memory (2 × 64 KB) beside the resident Wᵀ (64 KB):
//   warps 5..12  producers : warps 5..8 one X block each ([32 rows × 32 channels] with the prologue), warps 9..12 two per dH block
//                            ([32 rows × 32 output channels], BN-backward transform of dY / H); registers for two stages, so the loads
//                            of stage s + 1 are in flight while stage s is converted and stored;
//   warp 4       issuer    : per stage 4 × 2 weight-gradient MMAs (M = 128, N = 128 / 64) and 8 × 2 input-gradient MMAs (M = 128,
//                            N = 64 / 32), then commits the dXᵀ buffer and the stage;
//   warps 0..3   epilogue  : per stage tcgen05.ld 32x32b: thread k holds channel k of the 32 rows, each warp-wide store writes 32
//                            consecutive channels of one row (128 B, no staging); at the end dWᵀ goes to the partial slot.
// What bounds it: reading dY, H, X1, X2 and writing dX1, dX2 once (rows × (2·Cout + 2·Ktot) × 4 bytes).
#include <algorithm>

#include "common.cuh"
#include "linear_args.cuh"
#include "umma.cuh"

namespace crf {
namespace lin3b {

using lin::DgradArgs;
using lin::WgradArgs;
using lin::lrelu;
using namespace umma;

// 13 warps: 4 of them on one SM sub-partition leave 128 registers per thread (17 warps would leave 96, and the producers spill)
constexpr int kEpiWarps = 4, kProdWarps = 8;
constexpr int kThreads = (kEpiWarps + 1 + kProdWarps) * 32;      // 416
constexpr int RS = 32;                                           // rows per stage = N of the input-gradient MMA
constexpr int kBlockBytes = RS * 128;                            // one [32 rows × 32 channels] fp32 block / slab
constexpr int kXBlocks = 4;                                      // M = 128 input channels (zero blocks beyond Ktot)
constexpr int BN = 64, NB = BN / 32;                             // output channels padded to 64 (32 < Cout <= 64)
constexpr int kStages = 2;
// stage: [X hi ×4][X lo ×4][dH hi ×NB][dH lo ×NB] (MN-major, weight gradient) [dH hi, dH lo] × NB (K-major, input gradient).  In
// both dH copies the lo part lies behind the hi part along N, so that one MMA with N doubled computes hi·hi and hi·lo side by side.
constexpr int kStageBytes = 2 * (kXBlocks + 2 * NB) * kBlockBytes;
constexpr int kWBlockBytes = BN * 128;                           // one [64 output-channel lines × 32 input channels] block of Wᵀ
constexpr int kWBytes = 2 * kXBlocks * kWBlockBytes;             // hi, lo
// [dWᵀ: hi·hi + lo·hi | hi·lo][dXᵀ buffer 0: hi·hi + lo·hi | hi·lo][dXᵀ buffer 1: same]; the epilogue adds the two halves
constexpr uint32_t kTmemCols = 256;
static_assert(2 * BN + kStages * 2 * RS <= (int)kTmemCols, "TMEM columns");
constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + kWBytes + (size_t)(4 * BN + 2 * 128) * 4 + (2 * kStages + 2 * kStages) * 8 + 16;
static_assert(kSmemBytes <= 227 * 1024, "shared memory");

__global__ void __launch_bounds__(kThreads, 1) bwd3_kernel(const DgradArgs d, const WgradArgs a, const int ntiles) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* stage0 = smem;                                                   // kStages stages
    uint8_t* w_s = smem + kStages * kStageBytes;                              // [Wᵀ hi ×4][Wᵀ lo ×4]
    float* s_par = reinterpret_cast<float*>(w_s + kWBytes);                   // [4][BN]: sc, sh, pz, pw of the BN-backward transform
    float* s_sc = s_par + 4 * BN;                                             // [128] prologue scale per padded input column
    float* s_sh = s_sc + 128;
    uint64_t* full = reinterpret_cast<uint64_t*>(s_sh + 128);                 // [kStages] producers → issuer
    uint64_t* empty = full + kStages;                                         // [kStages] issuer (commit) → producers
    uint64_t* tfull = empty + kStages;                                        // [kStages] dXᵀ buffer ready → epilogue
    uint64_t* tempty = tfull + kStages;                                       // [kStages] epilogue → issuer
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + kStages);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nch1 = (a.C1 + 31) / 32, nch2 = (a.C2 + 31) / 32, nchX = nch1 + nch2;
    const int C = a.Cout, Ktot = a.C1 + a.C2;
    const int T = nchX + NB;                                                  // tasks per stage
    const bool plain = a.bn.scale == nullptr;

    if (warp == 0) tmem_alloc(tmem_slot, kTmemCols);
    if (tid == kEpiWarps * 32) {
        for (int i = 0; i < kStages; ++i) {
            mbar_init(full + i, (uint32_t)T); mbar_init(empty + i, 1);
            mbar_init(tfull + i, 1); mbar_init(tempty + i, kEpiWarps);
        }
        mbar_init_fence();
    }
    {   // Wᵀ: padded input channel p = 32·b + j on block b, line co; W is a parameter, read before the dependency wait
        constexpr int WPT = (kXBlocks * 32 * BN + kThreads - 1) / kThreads;
        float wv[WPT];
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * kThreads, co = e >> 7, p = e & 127, b = p >> 5, j = p & 31;
            int col = -1;                                                     // consecutive threads → consecutive columns of one W row
            if (b < nch1) { if (32 * b + j < a.C1) col = 32 * b + j; }
            else if (b < nchX && 32 * (b - nch1) + j < a.C2) col = a.C1 + 32 * (b - nch1) + j;
            wv[i] = (e < kXBlocks * 32 * BN && co < C && col >= 0) ? __ldg(d.W + (int64_t)co * Ktot + col) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * kThreads, co = e >> 7, p = e & 127, b = p >> 5, j = p & 31;
            if (e < kXBlocks * 32 * BN) {
                float hi, lo;
                split_tf32(wv[i], hi, lo);
                const uint32_t off = (uint32_t)(b * kWBlockBytes) + blk_off(co, j >> 2) + ((j & 3) << 2);
                *reinterpret_cast<float*>(w_s + off) = hi;
                *reinterpret_cast<float*>(w_s + kXBlocks * kWBlockBytes + off) = lo;
            }
        }
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
    for (int i = tid; i < kStages * kStageBytes / 16; i += kThreads) reinterpret_cast<float4*>(smem)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp > kEpiWarps) {
        // ===================================================================== producers
        // warps 5..8: one X block each (8 rows per thread); warps 9..12: two per dH block (4 rows of dY and H per thread).
        // Both keep 16 float4 in flight per thread: registers for two stages, so the loads of stage s + 1 are in flight while
        // stage s is converted and stored.  A unit has a task in every stage, so it is at most one phase behind the stage
        // barriers (parity is enough).  No fence.proxy.async here: the issuer fences after acquiring the stage.
        const int p = warp - (kEpiWarps + 1);
        const bool is_x = p < kXBlocks;
        const int blk = is_x ? p : (p - kXBlocks) / 2;                        // X block, or dH block
        const int t = is_x ? lane : tid - (kEpiWarps + 1 + kXBlocks + 2 * blk) * 32;
        const int c16 = t & 7, rb = t >> 3;                                   // 16-byte chunk of the 32-channel block; first row
        const int unit = is_x ? blk : kXBlocks + blk;                         // named barrier 2 + unit
        auto arrive = [&](int st, int nthreads) {
            asm volatile("bar.sync %0, %1;" ::"r"(2 + unit), "r"(nthreads) : "memory");
            if (t == 0) mbar_arrive(full + st);
        };
        auto row0 = [&](int ti) { return ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * RS; };
        if (is_x && blk < nchX) {
            constexpr int RJ = 4, NJ = RS / RJ;
            const bool seg1 = blk < nch1;
            const float* X = seg1 ? a.X1 : a.X2;
            const int Cs = seg1 ? a.C1 : a.C2;
            const int col = (seg1 ? blk : blk - nch1) * 32 + 4 * c16;
            const bool pro = seg1 && a.scale1 != nullptr;
            const float slope1 = a.scale1 ? a.slope1 : 1.0f;
            auto load = [&](int ti, float4 (&v)[NJ]) {
                const int64_t m0 = row0(ti);
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int64_t m = m0 + rb + RJ * j;
                    v[j] = (col < Cs && m < a.M) ? __ldg(reinterpret_cast<const float4*>(X + m * Cs + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            auto publish = [&](int ti, float4 (&v)[NJ]) {
                const int st = ti % kStages;
                const int64_t m0 = row0(ti);
                if (pro) {
                    const float4 sc = *reinterpret_cast<const float4*>(s_sc + blk * 32 + 4 * c16);
                    const float4 sh = *reinterpret_cast<const float4*>(s_sh + blk * 32 + 4 * c16);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const bool ok = col < Cs && (m0 + rb + RJ * j < a.M);   // the prologue's shift must not leak into padding
                        v[j] = ok ? make_float4(lrelu(fmaf(v[j].x, sc.x, sh.x), slope1), lrelu(fmaf(v[j].y, sc.y, sh.y), slope1),
                                                lrelu(fmaf(v[j].z, sc.z, sh.z), slope1), lrelu(fmaf(v[j].w, sc.w, sh.w), slope1))
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                mbar_wait_relaxed(empty + st, ((uint32_t)(ti / kStages) & 1) ^ 1);
                uint8_t* dst = stage0 + st * kStageBytes + blk * kBlockBytes;   // lo copy kXBlocks blocks further
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    float4 h, l;
                    split_tf32(v[j].x, h.x, l.x); split_tf32(v[j].y, h.y, l.y); split_tf32(v[j].z, h.z, l.z); split_tf32(v[j].w, h.w, l.w);
                    const uint32_t off = blk_off(rb + RJ * j, c16);
                    *reinterpret_cast<float4*>(dst + off) = h;
                    *reinterpret_cast<float4*>(dst + kXBlocks * kBlockBytes + off) = l;
                }
                arrive(st, 32);
            };
            float4 vA[NJ], vB[NJ];
            if (my_tiles > 0) load(0, vA);
            if (my_tiles > 1) load(1, vB);
            for (int ti = 0; ti < my_tiles; ti += 2) {
                publish(ti, vA);
                if (ti + 2 < my_tiles) load(ti + 2, vA);
                if (ti + 1 < my_tiles) {
                    publish(ti + 1, vB);
                    if (ti + 3 < my_tiles) load(ti + 3, vB);
                }
            }
        } else if (!is_x) {
            constexpr int RJ = 8, NJ = RS / RJ;
            const int col = 32 * blk + 4 * c16;
            const bool cok = col < C;
            const float slope = a.bn.slope;
            auto load = [&](int ti, float4 (&v)[NJ], float4 (&hh)[NJ]) {
                const int64_t m0 = row0(ti);
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int64_t m = m0 + rb + RJ * j;
                    const bool ok = cok && m < a.M;
                    const int64_t off = ok ? m * C + col : 0;
                    v[j] = ok ? __ldg(reinterpret_cast<const float4*>(a.dY + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    hh[j] = (ok && !plain) ? __ldg(reinterpret_cast<const float4*>(a.H + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            auto publish = [&](int ti, float4 (&v)[NJ], float4 (&hh)[NJ]) {
                const int st = ti % kStages;
                const int64_t m0 = row0(ti);
                if (!plain) {
                    const float4 sc = *reinterpret_cast<const float4*>(s_par + col), sh = *reinterpret_cast<const float4*>(s_par + BN + col);
                    const float4 pz = *reinterpret_cast<const float4*>(s_par + 2 * BN + col), pw = *reinterpret_cast<const float4*>(s_par + 3 * BN + col);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const bool ok = cok && (m0 + rb + RJ * j < a.M);      // the additive terms must not leak into padding
                        const float4 dy = v[j], h = hh[j];
                        const float4 pre = make_float4(fmaf(h.x, sc.x, sh.x), fmaf(h.y, sc.y, sh.y), fmaf(h.z, sc.z, sh.z), fmaf(h.w, sc.w, sh.w));
                        float4 o;
                        o.x = fmaf(sc.x, pre.x > 0.f ? dy.x : dy.x * slope, fmaf(pz.x, h.x, pw.x));
                        o.y = fmaf(sc.y, pre.y > 0.f ? dy.y : dy.y * slope, fmaf(pz.y, h.y, pw.y));
                        o.z = fmaf(sc.z, pre.z > 0.f ? dy.z : dy.z * slope, fmaf(pz.z, h.z, pw.z));
                        o.w = fmaf(sc.w, pre.w > 0.f ? dy.w : dy.w * slope, fmaf(pz.w, h.w, pw.w));
                        v[j] = ok ? o : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                mbar_wait_relaxed(empty + st, ((uint32_t)(ti / kStages) & 1) ^ 1);
                uint8_t* dmn = stage0 + st * kStageBytes + (2 * kXBlocks + blk) * kBlockBytes;          // MN-major copy; lo NB blocks further
                uint8_t* dk = stage0 + st * kStageBytes + (2 * kXBlocks + 2 * NB + 2 * blk) * kBlockBytes;  // K-major copy; lo one slab further
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    float4 h, l;
                    split_tf32(v[j].x, h.x, l.x); split_tf32(v[j].y, h.y, l.y); split_tf32(v[j].z, h.z, l.z); split_tf32(v[j].w, h.w, l.w);
                    const int r = rb + RJ * j;
                    const uint32_t om = blk_off(r, c16), okm = slab_chunk_off(r, c16);
                    *reinterpret_cast<float4*>(dmn + om) = h;
                    *reinterpret_cast<float4*>(dmn + NB * kBlockBytes + om) = l;
                    *reinterpret_cast<float4*>(dk + okm) = h;
                    *reinterpret_cast<float4*>(dk + kBlockBytes + okm) = l;
                }
                arrive(st, 64);
            };
            float4 vA[NJ], hA[NJ], vB[NJ], hB[NJ];
            if (my_tiles > 0) load(0, vA, hA);
            if (my_tiles > 1) load(1, vB, hB);
            for (int ti = 0; ti < my_tiles; ti += 2) {
                publish(ti, vA, hA);
                if (ti + 2 < my_tiles) load(ti + 2, vA, hA);
                if (ti + 1 < my_tiles) {
                    publish(ti + 1, vB, hB);
                    if (ti + 3 < my_tiles) load(ti + 3, vB, hB);
                }
            }
        }
    } else if (warp == kEpiWarps) {
        // ===================================================================== MMA issuer
        // hi·[hi | lo] as one MMA with N doubled, then lo·hi into the first half: 2 MMAs per k-step instead of 3 (operand fetch −22 %)
        constexpr uint32_t idesc_w2 = idesc_tf32(128, 2 * BN) | (1u << 15) | (1u << 16);   // A = Xin, B = dH: both MN-major
        constexpr uint32_t idesc_w = idesc_tf32(128, BN) | (1u << 15) | (1u << 16);
        constexpr uint32_t idesc_d2 = idesc_tf32(128, 2 * RS) | (1u << 15);                // A = Wᵀ MN-major, B = dH K-major
        constexpr uint32_t idesc_d = idesc_tf32(128, RS) | (1u << 15);
        const uint64_t wh = desc_mn(smem_u32(w_s), kWBlockBytes), wl = desc_mn(smem_u32(w_s + kXBlocks * kWBlockBytes), kWBlockBytes);
        const int nk8 = (C + 7) >> 3;
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int st = ti % kStages;
            const uint32_t par = (uint32_t)(ti / kStages) & 1;
            mbar_wait(full + st, par);
            mbar_wait(tempty + st, par ^ 1);
            fence_async_smem();                                              // producers' generic-proxy stores → async proxy
            tc_fence_after();
            if (elect_one()) {
                const uint32_t sb = smem_u32(stage0 + st * kStageBytes);
                const uint64_t xh = desc_mn(sb, kBlockBytes), xl = desc_mn(sb + kXBlocks * kBlockBytes, kBlockBytes);
                const uint64_t dh = desc_mn(sb + 2 * kXBlocks * kBlockBytes, kBlockBytes), dl = desc_mn(sb + (2 * kXBlocks + NB) * kBlockBytes, kBlockBytes);
#pragma unroll
                for (int j = 0; j < RS / 8; ++j) {                            // 8 rows = 1024 bytes = 64 descriptor units per step
                    mma_tf32(tmem, xh + 64 * j, dh + 64 * j, idesc_w2, (ti | j) != 0);     // N = [dH hi | dH lo]
                    mma_tf32(tmem, xl + 64 * j, dh + 64 * j, idesc_w, 1);
                }
                const uint32_t dx = tmem + (uint32_t)(2 * BN + st * 2 * RS);
                const uint64_t kh = smem_desc_k128(sb + (2 * kXBlocks + 2 * NB) * kBlockBytes);
#pragma unroll
                for (int k8 = 0; k8 < BN / 8; ++k8) {
                    if (k8 < nk8) {                                          // 8 output channels: 8 lines of Wᵀ, 32 bytes into a dH slab
                        const uint32_t bo = (uint32_t)((k8 >> 2) * (2 * kBlockBytes / 16) + 2 * (k8 & 3));
                        mma_tf32(dx, wh + 64 * k8, kh + bo, idesc_d2, k8 != 0);             // N = [32 rows hi | 32 rows lo]
                        mma_tf32(dx, wl + 64 * k8, kh + bo, idesc_d, 1);
                    }
                }
                mma_commit(tfull + st);
                mma_commit(empty + st);
            }
            __syncwarp();
        }
    } else {
        // ===================================================================== epilogue: TMEM lane = padded input channel
        float* dst = nullptr;
        int ld = 0, acc = 0, col = -1;
        if (warp < nch1) {
            const int c = 32 * warp + lane;
            if (c < a.C1) { col = c; if (d.dX1) { dst = d.dX1 + c; ld = a.C1; acc = d.acc1; } }
        } else if (warp < nchX) {
            const int c = 32 * (warp - nch1) + lane;
            if (c < a.C2) { col = a.C1 + c; if (d.dX2) { dst = d.dX2 + c; ld = a.C2; acc = d.acc2; } }
        }
        const uint32_t lanes = (uint32_t)(warp * 32) << 16;
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int st = ti % kStages;
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * RS;
            const int valid = (int)min((int64_t)RS, a.M - m0);
            mbar_wait_relaxed_nocall(tfull + st, (uint32_t)(ti / kStages) & 1);
            tc_fence_after();
            uint32_t v[RS / 16][16], u[RS / 16][16];
#pragma unroll
            for (int cb = 0; cb < RS / 16; ++cb) {
                tmem_ld16_issue(tmem + lanes + (uint32_t)(2 * BN + st * 2 * RS + 16 * cb), v[cb]);
                tmem_ld16_issue(tmem + lanes + (uint32_t)(2 * BN + st * 2 * RS + RS + 16 * cb), u[cb]);
            }
            tmem_ld_wait();
#pragma unroll
            for (int cb = 0; cb < RS / 16; ++cb)
#pragma unroll
                for (int i = 0; i < 16; ++i) v[cb][i] = __float_as_uint(__uint_as_float(v[cb][i]) + __uint_as_float(u[cb][i]));
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + st);
            if (dst) {
                float* p = dst + m0 * ld;
#pragma unroll
                for (int r0 = 0; r0 < RS; r0 += 8, p += 8 * ld) {            // 8 rows at a time: the += loads in flight together
                    float o[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) o[i] = __uint_as_float(v[(r0 + i) / 16][(r0 + i) % 16]);
                    if (acc) {
                        float old[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) old[i] = r0 + i < valid ? p[i * ld] : 0.f;
#pragma unroll
                        for (int i = 0; i < 8; ++i) o[i] += old[i];
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (r0 + i < valid) p[i * ld] = o[i];
                }
            }
        }
        // the last dXᵀ commit also covered every weight-gradient MMA: dWᵀ is final
        float* wdst = a.dW + a.slot_stride * (int64_t)(blockIdx.x % kGradSlots);
#pragma unroll
        for (int c0 = 0; c0 < BN; c0 += 16) {
            float w[16], wl[16];
            tmem_ld16(tmem + lanes + (uint32_t)c0, w);
            tmem_ld16(tmem + lanes + (uint32_t)(BN + c0), wl);
#pragma unroll
            for (int i = 0; i < 16; ++i) w[i] += wl[i];
            if (col >= 0) {
                float* q = wdst + (int64_t)c0 * Ktot + col;
#pragma unroll
                for (int i = 0; i < 16; ++i, q += Ktot)
                    if (c0 + i < C) atomicAdd(q, w[i]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

}  // namespace lin3b

namespace lin {

int try_bwd3(const DgradArgs& d, const WgradArgs& w, int precision, cudaStream_t st) {
    using namespace lin3b;
    if (precision != 0) return kDeclined;
    if (!w.dW || (!d.dX1 && !d.dX2)) return kDeclined;
    if (w.idx1 || w.dbias || w.bn.act_ref) return kDeclined;
    if (w.Cout <= 32 || w.Cout > BN || (w.Cout & 3) || (w.C1 & 3) || (w.C2 & 3) || w.C1 <= 0) return kDeclined;
    const int Ktot = w.C1 + w.C2;
    if (Ktot <= 64 || Ktot > 128 || (w.C1 + 31) / 32 + (w.C2 + 31) / 32 > kXBlocks) return kDeclined;
    if (!aligned16(w.dY) || !aligned16(w.X1) || (w.C2 && !aligned16(w.X2)) || (w.bn.scale && !aligned16(w.H))) return kDeclined;
    if ((d.dX1 && !aligned16(d.dX1)) || (d.dX2 && !aligned16(d.dX2))) return kDeclined;
    const int ntiles = (int)ceil_div(w.M, RS);
    if (ntiles <= 0) return kDeclined;
    return launch(bwd3_kernel, dim3(std::min(ntiles, kNumSMs)), dim3(kThreads), kSmemBytes, st, d, w, ntiles);
}

}  // namespace lin
}  // namespace crf
