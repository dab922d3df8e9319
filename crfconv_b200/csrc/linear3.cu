// Third-generation Linear forward for sm_100a: the contraction runs on the 5th-generation tensor cores (tcgen05.mma,
// kind::tf32, 128×N×8 per instruction) with the accumulator in TMEM.  Same contract as the other forward kernels
// (linear_args.cuh FwdArgs): Y = [ lrelu(X1·scale1+shift1) | X2 ] · Wᵀ (+bias), optional row gather on segment 1, BatchNorm
// Σ/Σ² partials in the epilogue.  fp32 parity comes from 3xTF32: every operand is split into tf32 hi + remainder lo and three
// MMAs accumulate hi·hi + hi·lo + lo·hi in fp32 (measured 1.7e-6 relative, scripts/micro/umma_test.cu).
//
// One persistent CTA per SM, 17 warps with fixed roles, rows streamed in 128-row tiles:
//   warps 5..16  producers : 3 groups of 4 warps; group g owns every 3rd [128 rows × 32 columns] slab and ring slot g: coalesced
//                            128-bit global loads into registers (double-buffered: the next slab's loads fly while this one is
//                            converted), BatchNorm+LeakyReLU prologue, hi/lo split, stores in the swizzled K-major operand layout,
//                            mbarrier arrive (release); the generic→async proxy fence is on the issuer's side;
//   warp 4       issuer    : one thread waits for a slab, issues its ≤12 MMAs against the CTA-resident split weights and
//                            tcgen05.commit's the slot back to the producers; after a tile's last slab it commits the accumulator;
//   warps 0..3   epilogue  : tcgen05.ld of the [128 × N] accumulator (one row per thread), bias, staging in shared memory,
//                            coalesced stores, per-column Σ/Σ² kept in registers across all the CTA's tiles.
// Two accumulator buffers in TMEM let tile i+1's MMAs overlap tile i's epilogue.  What bounds it: the activation read from
// HBM (rows × (Ktot + Cout) × 4 bytes); the MMAs of a tile take ≈0.8 us of the ≈1.9 us the tile's bytes need.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "linear_args.cuh"
#include "umma.cuh"

namespace crf {
namespace lin3 {

using lin::FwdArgs;
using namespace umma;

constexpr int kEpiWarps = 4, kProdWarps = 12;
constexpr int kThreads = (kEpiWarps + 1 + kProdWarps) * 32;      // 544
constexpr int kGroupWarps = 4;                                   // producer warps that share one slab
constexpr int kGroups = kProdWarps / kGroupWarps;                // = RING: group g owns ring slot g
constexpr int kRowsPerPass = kGroupWarps * 4;                    // a producer warp covers 4 rows × 128 B per load instruction
constexpr int kLoadsPerSlab = 128 / kRowsPerPass;                // float4 loads per producer thread and slab (8)
constexpr int BM = 128, BK = 32, RING = 3;
static_assert(kGroups == RING, "group g owns ring slot g: its uses of the slot barriers are consecutive phases");
constexpr int kSlabBytes = BM * 128;                             // one [128 × 32] fp32 slab
constexpr int kSlotBytes = 2 * kSlabBytes;                       // hi + lo

// Development aid (-DCRF_FWD3_TRACE): CTA 0 appends (event, index, clock) records; read back with crfconv_debug_fwd3_trace.
#ifdef CRF_FWD3_TRACE
__device__ long long g_trace[3 * 8192];
__device__ int g_trace_n;
__device__ __forceinline__ void trace(int ev, int idx) {      // fixed record slot per (event, index): plain stores, no atomics
    if (blockIdx.x != 0) return;
    const int i = ev <= 4 ? idx * 4 + (ev - 1) : (ev <= 6 ? 400 + idx * 2 + (ev - 5) : (ev <= 9 ? 700 + idx * 3 + (ev - 7) : 1000 + idx * 4 + (ev - 10)));
    if (i < 8192) { g_trace[3 * i] = ev; g_trace[3 * i + 1] = idx; g_trace[3 * i + 2] = clock64(); }
    g_trace_n = 1400;
}
#define CRF_TRACE(ev, idx) trace(ev, idx)
#else
#define CRF_TRACE(ev, idx)
#endif

template <int BN>
struct Layout {
    static constexpr int kStageLd = BN + 4;                      // padded staging rows: conflict-free row-per-thread float4 stores
    static constexpr uint32_t kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;
    static size_t bytes(int nch) {
        return (size_t)RING * kSlotBytes + (size_t)2 * nch * BN * 128 + (size_t)BM * kStageLd * 4 + (size_t)2 * nch * BK * 4 +
               (size_t)(2 * RING + 4) * 8 + 16;
    }
};

template <int BN>
__global__ void __launch_bounds__(kThreads, 1) fwd3_kernel(const FwdArgs a, const int ntiles) {
    using L = Layout<BN>;
    // Declared 1024-byte aligned (operand slabs need it for SWIZZLE_128B) and used through plain pointer arithmetic only: an
    // integer round-trip to align by hand makes the compiler lose the address space and emit generic ST.E/LD.E instead of STS/LDS.
    extern __shared__ __align__(1024) uint8_t smem[];
    const int nch1 = (a.C1 + BK - 1) / BK, nch2 = (a.C2 + BK - 1) / BK, nch = nch1 + nch2;
    const int Kpad = nch * BK, Ktot = a.C1 + a.C2;
    uint8_t* ring = smem;                                          // [RING][hi slab | lo slab]
    uint8_t* w_hi = ring + RING * kSlotBytes;                      // [nch][BN rows × 128 B]
    uint8_t* w_lo = w_hi + nch * BN * 128;
    float* stage = reinterpret_cast<float*>(w_lo + nch * BN * 128);   // [BM][BN + 4]
    float* s_sc = stage + BM * L::kStageLd;
    float* s_sh = s_sc + Kpad;
    uint64_t* full = reinterpret_cast<uint64_t*>(s_sh + Kpad);     // producers → issuer, per ring slot
    uint64_t* empty = full + RING;                                 // issuer (commit) → producers
    uint64_t* tfull = empty + RING;                                // issuer (commit) → epilogue, per accumulator buffer
    uint64_t* tempty = tfull + 2;                                  // epilogue → issuer
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(tmem_slot, L::kTmemCols);
    if (tid == kEpiWarps * 32) {
        for (int i = 0; i < RING; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, kEpiWarps); }
        mbar_init_fence();
    }
    // weights: split once per CTA, resident in the operand layout for the whole kernel.  All of a thread's loads are issued
    // before the first one is used (a dependent load per iteration made this prologue ≈6 us of a ≈60 us kernel).
    {
        constexpr int WPT = (BN * 128 + kThreads - 1) / kThreads;      // elements per thread at Kpad = 128
        float wv[WPT];
        const int total = BN * Kpad;
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * kThreads;
            float w = 0.f;
            if (e < total) {
                const int n = e / Kpad, k = e - n * Kpad, c = k / BK, kk = k % BK;
                int col = -1;
                if (c < nch1) { if (c * BK + kk < a.C1) col = c * BK + kk; }
                else if ((c - nch1) * BK + kk < a.C2) col = a.C1 + (c - nch1) * BK + kk;
                if (col >= 0 && n < a.Cout) w = __ldg(a.W + (int64_t)n * Ktot + col);
            }
            wv[i] = w;
        }
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
            const int e = tid + i * kThreads;
            if (e < total) {
                const int n = e / Kpad, k = e - n * Kpad, c = k / BK, kk = k % BK;
                float hi, lo;
                split_tf32(wv[i], hi, lo);
                const uint32_t off = (uint32_t)(c * BN * 128) + slab_chunk_off(n, kk >> 2) + ((kk & 3) << 2);
                *reinterpret_cast<float*>(w_hi + off) = hi;
                *reinterpret_cast<float*>(w_lo + off) = lo;
            }
        }
    }
    for (int k = tid; k < Kpad; k += kThreads) {
        float sc = 1.f, sh = 0.f;
        if (a.scale1 && k < nch1 * BK && k < a.C1) { sc = __ldg(a.scale1 + k); sh = __ldg(a.shift1 + k); }
        s_sc[k] = sc; s_sh[k] = sh;
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    if ((smem_u32(smem) & 1023u) != 0) __trap();                  // dynamic shared memory base not 1024-byte aligned
    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp > kEpiWarps) {
        // ===================================================================== producers
        // Slab q of this CTA's stream belongs to producer group q % kGroups, which also owns ring slot q % RING (kGroups == RING).
        // Two register sets per thread: the loads of the group's NEXT slab are in flight while the current one is converted, so
        // 6 slabs (96 KB) of HBM reads are outstanding per SM.  Producers do NOT execute fence.proxy.async: it compiles to
        // MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC, and the MEMBAR waits for every global load the thread has in flight, which serialised
        // each slab on a full HBM round trip (measured 1.4 us per slab).  The generic→async proxy fence is executed by the issuer
        // instead, after it has acquired the slab through the mbarrier and before it hands the shared-memory tile to the tensor core.
        const int g = (warp - (kEpiWarps + 1)) / kGroupWarps;
        const int t = tid - (kEpiWarps + 1) * 32 - g * (kGroupWarps * 32);
        const int c4 = t & 7, rb = t >> 3;                         // 16-byte column chunk; rows rb + kRowsPerPass·j
        const int Q = my_tiles * nch;
        uint8_t* hi_slab = ring + g * kSlotBytes;
        auto load = [&](int q, float4 (&buf)[kLoadsPerSlab]) {
            const int lt = q / nch, lc = q - lt * nch;
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)lt * gridDim.x) * BM;
            const bool seg1 = lc < nch1;
            const float* X = seg1 ? a.X1 : a.X2;
            const int C = seg1 ? a.C1 : a.C2;
            const int col = (seg1 ? lc : lc - nch1) * BK + 4 * c4;
            const float* base = X + (m0 + rb) * C + col;
            const int64_t left = a.M - m0 - rb;                    // rows of this thread's column that exist
#pragma unroll
            for (int j = 0; j < kLoadsPerSlab; ++j) {
                const bool ok = (kRowsPerPass * j < left) && (col < C);
                buf[j] = ok ? __ldg(reinterpret_cast<const float4*>(base + (int64_t)(kRowsPerPass * j) * C)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        auto publish = [&](int q, float4 (&buf)[kLoadsPerSlab]) {
            const int lt = q / nch, lc = q - lt * nch;
            const uint32_t use = (uint32_t)(q / RING);
            if (lc < nch1 && a.scale1) {                           // BatchNorm + LeakyReLU prologue (this is where the thread waits for its loads)
                const float4 sc = *reinterpret_cast<const float4*>(s_sc + lc * BK + 4 * c4);
                const float4 sh = *reinterpret_cast<const float4*>(s_sh + lc * BK + 4 * c4);
                const float sl = a.slope1;
#pragma unroll
                for (int j = 0; j < kLoadsPerSlab; ++j) {          // lrelu(v) = max(v, slope·v): slopes in [0, 1] only (checked by try_fwd3)
                    float4 v = buf[j];
                    v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y); v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
                    buf[j] = make_float4(fmaxf(v.x, v.x * sl), fmaxf(v.y, v.y * sl), fmaxf(v.z, v.z * sl), fmaxf(v.w, v.w * sl));
                }
            }
            mbar_wait_relaxed(empty + g, (use & 1) ^ 1);           // the tensor core has consumed this slot's previous slab
            if (t == 0) CRF_TRACE(2, q);
#pragma unroll
            for (int j = 0; j < kLoadsPerSlab; ++j) {
                const float4 v = buf[j];
                float4 h, l;
                split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
                const uint32_t off = slab_chunk_off(rb + kRowsPerPass * j, c4);
                *reinterpret_cast<float4*>(hi_slab + off) = h;
                *reinterpret_cast<float4*>(hi_slab + kSlabBytes + off) = l;
            }
            if (t == 0) CRF_TRACE(3, q);
            // all of the group's stores are ordered before the (release) arrive of its thread 0 by the named barrier
            asm volatile("bar.sync %0, %1;" ::"r"(2 + g), "n"(kGroupWarps * 32) : "memory");
            if (t == 0) mbar_arrive(full + g);
            if (t == 0) CRF_TRACE(4, q);
        };
        float4 bufA[kLoadsPerSlab], bufB[kLoadsPerSlab];
        if (g < Q) load(g, bufA);
        for (int q = g; q < Q; q += 2 * kGroups) {
            if (q + kGroups < Q) load(q + kGroups, bufB);
            publish(q, bufA);
            if (q + 2 * kGroups < Q) load(q + 2 * kGroups, bufA);
            if (q + kGroups < Q) publish(q + kGroups, bufB);
        }
    } else if (warp == kEpiWarps) {
        // ===================================================================== MMA issuer (whole warp waits, one elected lane issues)
        // The loop below is the kernel's critical path (one slab per iteration, ≈600 cycles of MMA issue): everything that
        // does not depend on the slot is hoisted, the chunk loop is unrolled so per-chunk constants sit in registers, and a full
        // chunk issues its 12 MMAs without predicates.
        constexpr uint32_t idesc = idesc_tf32(BM, BN);
        const uint64_t a_desc0 = smem_desc_k128(smem_u32(ring));          // + slot·(kSlotBytes/16), + kSlabBytes/16 for lo
        const uint64_t bh_desc0 = smem_desc_k128(smem_u32(w_hi));         // + c·(BN·128/16)
        const uint64_t bl_desc0 = smem_desc_k128(smem_u32(w_lo));
        int nk8[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int kvalid = c < nch1 ? min(BK, a.C1 - c * BK) : min(BK, a.C2 - (c - nch1) * BK);
            nk8[c] = c < nch ? (kvalid + 7) >> 3 : 0;
        }
        int slot = 0;
        uint32_t use = 0;
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int buf = ti & 1;
            mbar_wait(tempty + buf, ((uint32_t)(ti >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d = tmem + (uint32_t)(buf * BN);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c < nch) {
                    if (lane == 0) CRF_TRACE(10, ti * nch + c);      // loop top
                    mbar_wait(full + slot, use & 1);
                    fence_async_smem();                          // producers' generic-proxy stores (acquired above) → async proxy
                    tc_fence_after();
                    if (elect_one()) {
                        CRF_TRACE(5, ti * nch + c);                  // issuer saw the slab
                        const uint64_t ah0 = a_desc0 + (uint64_t)(slot * (kSlotBytes / 16)), al0 = ah0 + kSlabBytes / 16;
                        const uint64_t bh0 = bh_desc0 + (uint64_t)(c * (BN * 128 / 16)), bl0 = bl_desc0 + (uint64_t)(c * (BN * 128 / 16));
                        if (nk8[c] == 4) {
#pragma unroll
                            for (int k8 = 0; k8 < 4; ++k8) {           // 32 bytes along K = 2 descriptor units per step
                                mma_tf32(d, al0 + 2 * k8, bh0 + 2 * k8, idesc, (c | k8) != 0);
                                mma_tf32(d, ah0 + 2 * k8, bl0 + 2 * k8, idesc, 1);
                                mma_tf32(d, ah0 + 2 * k8, bh0 + 2 * k8, idesc, 1);
                            }
                        } else {
#pragma unroll
                            for (int k8 = 0; k8 < 3; ++k8) {
                                if (k8 < nk8[c]) {
                                    mma_tf32(d, al0 + 2 * k8, bh0 + 2 * k8, idesc, (c | k8) != 0);
                                    mma_tf32(d, ah0 + 2 * k8, bl0 + 2 * k8, idesc, 1);
                                    mma_tf32(d, ah0 + 2 * k8, bh0 + 2 * k8, idesc, 1);
                                }
                            }
                        }
                        CRF_TRACE(13, ti * nch + c);                 // MMAs issued, before the commits
                        mma_commit(empty + slot);                      // slot reusable once these MMAs have read it
                        if (c == nch - 1) mma_commit(tfull + buf);     // accumulator complete
                        CRF_TRACE(6, ti * nch + c);
                    }
                    if (++slot == RING) { slot = 0; ++use; }
                }
            }
        }
    } else {
        // ===================================================================== epilogue (warps 0..3, one accumulator row per thread)
        const int row = tid;                                       // TMEM lane == tile row
        constexpr int LD = L::kStageLd;
        const int scol = tid % BN, spart = tid / BN;               // statistics pass: BM / BN threads per column, BN rows each
        constexpr int CH = BN / 4;                                 // 16-byte chunks per output row
        const int ochunk = tid % CH, orow = tid / CH;
        constexpr int RPP = BM / CH;                               // rows written per pass by the 128 threads
        float ssum = 0.f, ssq = 0.f;
        for (int ti = 0; ti < my_tiles; ++ti) {
            const int buf = ti & 1;
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
            const int valid = (int)min((int64_t)BM, a.M - m0);
            mbar_wait_relaxed(tfull + buf, (uint32_t)(ti >> 1) & 1);
            tc_fence_after();
            if (tid == 0) CRF_TRACE(7, ti);                    // accumulator complete
            {
                uint32_t v[BN / 16][16];
#pragma unroll
                for (int cb = 0; cb < BN / 16; ++cb) tmem_ld16_issue(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * BN + cb * 16), v[cb]);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + buf);          // accumulator buffer free for tile ti + 2
#pragma unroll
                for (int cb = 0; cb < BN / 16; ++cb) {
#pragma unroll
                    for (int i = 0; i < 16; i += 4) {
                        float4 o = make_float4(__uint_as_float(v[cb][i]), __uint_as_float(v[cb][i + 1]), __uint_as_float(v[cb][i + 2]),
                                               __uint_as_float(v[cb][i + 3]));
                        if (a.bias) {
                            const int c = cb * 16 + i;
                            o.x += c < a.Cout ? __ldg(a.bias + c) : 0.f;         o.y += c + 1 < a.Cout ? __ldg(a.bias + c + 1) : 0.f;
                            o.z += c + 2 < a.Cout ? __ldg(a.bias + c + 2) : 0.f; o.w += c + 3 < a.Cout ? __ldg(a.bias + c + 3) : 0.f;
                        }
                        *reinterpret_cast<float4*>(stage + row * LD + cb * 16 + i) = o;
                    }
                }
            }
            if (tid == 0) CRF_TRACE(8, ti);                    // TMEM read out
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const bool colok = 4 * ochunk < a.Cout;
            if (valid == BM) {                                     // full tile: compile-time trip counts, loads batched ahead of their uses
                if (colok) {
                    float* yp = a.Y + (m0 + orow) * a.Cout + 4 * ochunk;
                    const float* sp = stage + orow * LD + 4 * ochunk;
#pragma unroll
                    for (int i0 = 0; i0 < CH; i0 += 8) {
                        float4 tmp[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            if (i0 + i < CH) tmp[i] = *reinterpret_cast<const float4*>(sp + (i0 + i) * RPP * LD);
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            if (i0 + i < CH) *reinterpret_cast<float4*>(yp + (int64_t)(i0 + i) * RPP * a.Cout) = tmp[i];
                    }
                }
                if (a.stats) {
                    const float* sp = stage + spart * BN * LD + scol;
                    float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
                    for (int r = 0; r < BN; r += 2) {
                        const float x0 = sp[r * LD], x1 = sp[(r + 1) * LD];
                        s0 += x0; s1 += x1;
                        q0 = fmaf(x0, x0, q0); q1 = fmaf(x1, x1, q1);
                    }
                    ssum += s0 + s1;
                    ssq += q0 + q1;
                }
            } else {
                if (colok) {
                    for (int r = orow; r < valid; r += RPP)
                        *reinterpret_cast<float4*>(a.Y + (m0 + r) * a.Cout + 4 * ochunk) = *reinterpret_cast<const float4*>(stage + r * LD + 4 * ochunk);
                }
                if (a.stats) {
                    const int r1 = min((spart + 1) * BN, valid);
                    for (int r = spart * BN; r < r1; ++r) {
                        const float x = stage[r * LD + scol];
                        ssum += x;
                        ssq = fmaf(x, x, ssq);
                    }
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (tid == 0) CRF_TRACE(9, ti);                    // tile stored
        }
        if (a.stats && scol < a.Cout) {
            float* st = a.stats + (size_t)(blockIdx.x % 16) * 2 * a.Cout;      // 16 of the kStatSlots rows: ≤ 10 CTAs per row, short fold
            atomicAdd(st + scol, ssum);
            atomicAdd(st + a.Cout + scol, ssq);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, L::kTmemCols);
    if (a.fin.part) {                                              // BatchNorm finalize by the last CTA (Cout == BN, checked by the launcher)
        constexpr int NT = (kThreads / (2 * BN)) * (2 * BN);
        __shared__ double s_red[NT];
        cl::fwd_fin_tail<BN, NT>(a.fin, 16, s_red);
    }
}

}  // namespace lin3

#ifdef CRF_FWD3_TRACE
extern "C" int crfconv_debug_fwd3_trace(long long* out, int max_records, int reset) {
    int n = 0;
    cudaMemcpyFromSymbol(&n, lin3::g_trace_n, sizeof(int));
    if (n > 8192) n = 8192;
    if (n > max_records) n = max_records;
    if (out && n > 0) cudaMemcpyFromSymbol(out, lin3::g_trace, (size_t)n * 3 * sizeof(long long));
    if (reset) { const int z = 0; cudaMemcpyToSymbol(lin3::g_trace_n, &z, sizeof(int)); }
    return n;
}
#endif

namespace lin {

// tcgen05 forward: fp32-grade precision only (3xTF32); shapes of the hot path (Cout <= 64, <= 4 slabs of 32 input channels)
int try_fwd3(const FwdArgs& a, int precision, cudaStream_t st) {
    using namespace lin3;
    if (precision != 0) return kDeclined;
    if (a.idx1 || (a.scale1 && !(a.slope1 >= 0.f && a.slope1 <= 1.f))) return kDeclined;   // gathered rows / expanding slopes: older kernels
    if (a.Cout > 64 || (a.Cout & 3) || (a.C1 & 3) || (a.C2 & 3) || a.C1 <= 0) return kDeclined;
    const int nch = (a.C1 + BK - 1) / BK + (a.C2 + BK - 1) / BK;
    if (nch > 4) return kDeclined;
    if (!aligned16(a.X1) || (a.C2 && !aligned16(a.X2)) || !aligned16(a.Y)) return kDeclined;
    const int ntiles = (int)ceil_div(a.M, BM);
    if (ntiles <= 0) return kDeclined;
    if (a.fin.part && (a.fin.part != a.stats || (a.Cout != 64 && a.Cout != 32 && a.Cout != 16))) return kDeclined;   // fused finalize: Cout == BN only
    const dim3 grid(std::min(ntiles, kNumSMs));
    if (a.Cout > 32) return launch(fwd3_kernel<64>, grid, dim3(kThreads), Layout<64>::bytes(nch), st, a, ntiles);
    if (a.Cout > 16) return launch(fwd3_kernel<32>, grid, dim3(kThreads), Layout<32>::bytes(nch), st, a, ntiles);
    return launch(fwd3_kernel<16>, grid, dim3(kThreads), Layout<16>::bytes(nch), st, a, ntiles);
}

}  // namespace lin
}  // namespace crf
