// Second-generation Linear kernels (see linear2.cuh for the design).  Entry points try_fwd2 / try_dgrad2 / try_wgrad2
// are called by the C-ABI functions in linear.cu and return false when a shape is outside the fast path, in which case
// the generic kernels run instead.
#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "linear2.cuh"
#include "linear_args.cuh"

namespace crf {
namespace lin2 {

using lin::BnBwd;
using lin::DgradArgs;
using lin::FwdArgs;
using lin::WgradArgs;
using lin::lrelu;

constexpr int BK = 32;     // reduction chunk (floats) per pipeline stage
constexpr int AS = 40;     // smem row stride (floats) of staged fp32 tiles: 40 ≡ 8 (mod 32) ⇒ conflict-free LDS.64 at (g, 2t)
constexpr int NST = 3;     // cp.async ring depth

// ===================================================================================================== forward
// Y[M, Cout] = [ lrelu(X1*scale+shift) | X2 ] · Wᵀ (+bias), Σ/Σ² epilogue, single bf16 pass.   BN = padded Cout tile (8..64).
template <int BN>
__global__ void __launch_bounds__(kThreads, 2) fwd2_kernel(const FwdArgs a, const int ntiles) {
    constexpr int BM = 128;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int nch1 = (a.C1 + BK - 1) / BK, nch2 = (a.C2 + BK - 1) / BK, nch = nch1 + nch2;
    const int Kpad = nch * BK, WS2 = (Kpad + 8) / 2;   // W smem row stride in 32-bit words (bf16 pairs)
    float* As = reinterpret_cast<float*>(smem_raw);                       // [NST][BM][AS]
    uint32_t* Wh = reinterpret_cast<uint32_t*>(As + NST * BM * AS);       // [BN][WS2]
    uint32_t* Wl = Wh + BN * WS2;
    float* s_sc = reinterpret_cast<float*>(Wl + BN * WS2);                // [Kpad]
    float* s_sh = s_sc + Kpad;
    float* s_sum = s_sh + Kpad;                                           // [BN]
    float* s_sq = s_sum + BN;

    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int Ktot = a.C1 + a.C2;

    // ---- one-time setup: split W into bf16 (hi, lo), padded-K layout; prologue parameters; CTA-level statistics
    for (int e = tid; e < BN * (Kpad / 2); e += kThreads) {
        const int n = e / (Kpad / 2), kp = 2 * (e % (Kpad / 2));
        float wv[2] = {0.f, 0.f};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int k = kp + u, c = k / BK, kk = k % BK;
            int col = -1;
            if (c < nch1) { if (c * BK + kk < a.C1) col = c * BK + kk; }
            else if ((c - nch1) * BK + kk < a.C2) col = a.C1 + (c - nch1) * BK + kk;
            if (col >= 0 && n < a.Cout) wv[u] = __ldg(a.W + (int64_t)n * Ktot + col);
        }
        uint32_t hi, lo;
        split2(wv[0], wv[1], hi, lo);
        Wh[n * WS2 + kp / 2] = hi;
        Wl[n * WS2 + kp / 2] = lo;
    }
    for (int k = tid; k < Kpad; k += kThreads) {
        float sc = 1.f, sh = 0.f;
        if (a.scale1 && k < nch1 * BK && k < a.C1) { sc = __ldg(a.scale1 + k); sh = __ldg(a.shift1 + k); }
        s_sc[k] = sc; s_sh[k] = sh;
    }
    if (tid < BN) { s_sum[tid] = 0.f; s_sq[tid] = 0.f; }

    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int Q = my_tiles * nch;
    const int c4 = tid & 7, r0 = tid >> 3;

    int iq_t = 0, iq_c = 0, iq_s = 0;          // next chunk to issue: (tile, chunk, stage) counters instead of div/mod
    auto issue = [&]() {
        const int ti = iq_t, c = iq_c;
        const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
        const bool seg1 = c < nch1;
        const float* X = seg1 ? a.X1 : a.X2;
        const int C = seg1 ? a.C1 : a.C2;
        const int col = (seg1 ? c : c - nch1) * BK + 4 * c4;
        float* dst = As + iq_s * BM * AS;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = r0 + 32 * j;
            const int64_t m = m0 + r;
            const bool ok = (m < a.M) && (col < C);
            int64_t srow = ok ? m : 0;
            if (ok && seg1 && a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
            cp_async16(dst + r * AS + 4 * c4, X + srow * C + (ok ? col : 0), ok);
        }
        if (++iq_c == nch) { iq_c = 0; ++iq_t; }
        if (++iq_s == NST) iq_s = 0;
    };

    for (int s = 0; s < NST - 1; ++s) {
        if (s < Q) issue();
        cp_async_commit();
    }

    float acc[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    int ti = 0, c = 0, cs = 0;
    for (int q = 0; q < Q; ++q) {
        cp_async_wait<NST - 2>();
        __syncthreads();
        if (q + NST - 1 < Q) issue();
        cp_async_commit();

        const float* At = As + cs * BM * AS;
        const bool seg1 = c < nch1;
        const int kvalid = seg1 ? min(BK, a.C1 - c * BK) : min(BK, a.C2 - (c - nch1) * BK);
        const float slope = (seg1 && a.scale1) ? a.slope1 : 1.0f;
#pragma unroll
        for (int ks = 0; ks < BK / 16; ++ks) {
            if (ks * 16 < kvalid) {
                const int kb = ks * 16, kp = c * BK + kb + 2 * t;
                uint32_t ah[4], al[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = 16 * w + g + ((i & 1) ? 8 : 0);
                    const int ko = (i & 2) ? 8 : 0;
                    float2 v = *reinterpret_cast<const float2*>(At + row * AS + kb + 2 * t + ko);
                    const float2 sc = *reinterpret_cast<const float2*>(s_sc + kp + ko);
                    const float2 sh = *reinterpret_cast<const float2*>(s_sh + kp + ko);
                    v.x = lrelu(fmaf(v.x, sc.x, sh.x), slope);
                    v.y = lrelu(fmaf(v.y, sc.y, sh.y), slope);
                    split2(v.x, v.y, ah[i], al[i]);
                }
                const int wb = (c * BK + kb) / 2 + t;
#pragma unroll
                for (int nt = 0; nt < BN / 8; ++nt) {
                    const int wi = (nt * 8 + g) * WS2 + wb;
                    mma3<false>(acc[nt], ah, al, Wh[wi], Wh[wi + 4], Wl[wi], Wl[wi + 4]);
                }
            }
        }
        if (c == nch - 1) {   // ---- tile epilogue
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
            const int64_t row_a = m0 + 16 * w + g, row_b = row_a + 8;
            const bool va = row_a < a.M, vb = row_b < a.M;
#pragma unroll
            for (int nt = 0; nt < BN / 8; ++nt) {
                const int col = nt * 8 + 2 * t;
                float c0 = acc[nt][0], c1 = acc[nt][1], c2 = acc[nt][2], c3 = acc[nt][3];
                acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
                const bool cv = col < a.Cout;   // Cout is a multiple of 4 on this path ⇒ col+1 is valid too
                if (cv) {
                    if (a.bias) { const float b0 = __ldg(a.bias + col), b1 = __ldg(a.bias + col + 1); c0 += b0; c1 += b1; c2 += b0; c3 += b1; }
                    if (va) *reinterpret_cast<float2*>(a.Y + row_a * a.Cout + col) = make_float2(c0, c1);
                    if (vb) *reinterpret_cast<float2*>(a.Y + row_b * a.Cout + col) = make_float2(c2, c3);
                }
                if (a.stats) {   // warp-uniform branch: the shuffles below are executed by all lanes
                    float s0 = (va ? c0 : 0.f) + (vb ? c2 : 0.f), s1 = (va ? c1 : 0.f) + (vb ? c3 : 0.f);
                    float q0 = (va ? c0 * c0 : 0.f) + (vb ? c2 * c2 : 0.f), q1 = (va ? c1 * c1 : 0.f) + (vb ? c3 * c3 : 0.f);
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                        q0 += __shfl_xor_sync(0xffffffffu, q0, o); q1 += __shfl_xor_sync(0xffffffffu, q1, o);
                    }
                    if (g == 0 && cv) {
                        atomicAdd(&s_sum[col], s0); atomicAdd(&s_sum[col + 1], s1);
                        atomicAdd(&s_sq[col], q0);  atomicAdd(&s_sq[col + 1], q1);
                    }
                }
            }
        }
        if (++c == nch) { c = 0; ++ti; }
        if (++cs == NST) cs = 0;
    }
    cp_async_wait<0>();
    if (a.stats) {
        __syncthreads();
        if (tid < BN && tid < a.Cout) {
            float* st = a.stats + (size_t)(blockIdx.x % kStatSlots) * 2 * a.Cout;
            atomicAdd(st + tid, s_sum[tid]);
            atomicAdd(st + a.Cout + tid, s_sq[tid]);
        }
    }
}

// ---- fp32-grade forward: same persistent / cp.async structure, contraction on m16n8k8 tf32 with 3xTF32 compensation.
// Forward pre-activations decide the LeakyReLU branch taken in backward; keeping them at ≈2^-21 makes kink flips as rare
// as between two fp32 implementations (DESIGN.md §precision).  Double-buffered (the tf32 (hi, lo) copy of W is twice the
// size of the bf16 one); row stride 36 ≡ 4 (mod 32) ⇒ conflict-free scalar fragment loads at (g, t).
constexpr int AST = 36;
template <int BN> struct FwdT { static constexpr int NS = BN <= 16 ? 3 : 4; static constexpr int CTAS = BN <= 16 ? 3 : 2; };   // ring depth, CTAs/SM

__device__ __forceinline__ uint32_t tf32_of(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
// (hi, lo) tf32 split by TRUNCATION: cvt.rna.tf32 costs ~4 integer instructions on this part (SASS: IMAD/LOP3 sequences), which
// made operand conversion — not the tensor pipe — the bound of the 3xTF32 forward (ncu: 14.6 issued instructions per mma).
// hi = top 19 bits, lo = top 19 bits of the exact remainder: |a − hi − lo| <= 2^-20 |a|, i.e. products good to ≈1e-6.
__device__ __forceinline__ void split_trunc(float v, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(v) & 0xffffe000u;
    lo = __float_as_uint(v - __uint_as_float(hi)) & 0xffffe000u;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int BN>
__global__ void __launch_bounds__(kThreads, FwdT<BN>::CTAS) fwd2t_kernel(const FwdArgs a, const int ntiles) {
    constexpr int BM = 128, NSTT = FwdT<BN>::NS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int nch1 = (a.C1 + BK - 1) / BK, nch2 = (a.C2 + BK - 1) / BK, nch = nch1 + nch2;
    const int Kpad = nch * BK, WS = Kpad + 4;
    float* As = reinterpret_cast<float*>(smem_raw);                       // [NSTT][BM][AST]
    float* Wf = As + NSTT * BM * AST;                                     // [BN][WS] fp32
    float* s_sc = Wf + BN * WS;
    float* s_sh = s_sc + Kpad;
    float* s_sum = s_sh + Kpad;
    float* s_sq = s_sum + BN;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int Ktot = a.C1 + a.C2;

    for (int e = tid; e < BN * Kpad; e += kThreads) {
        const int n = e / Kpad, k = e % Kpad, c = k / BK, kk = k % BK;
        int col = -1;
        if (c < nch1) { if (c * BK + kk < a.C1) col = c * BK + kk; }
        else if ((c - nch1) * BK + kk < a.C2) col = a.C1 + (c - nch1) * BK + kk;
        Wf[n * WS + k] = (col >= 0 && n < a.Cout) ? __ldg(a.W + (int64_t)n * Ktot + col) : 0.f;
    }
    for (int k = tid; k < Kpad; k += kThreads) {
        float sc = 1.f, sh = 0.f;
        if (a.scale1 && k < nch1 * BK && k < a.C1) { sc = __ldg(a.scale1 + k); sh = __ldg(a.shift1 + k); }
        s_sc[k] = sc; s_sh[k] = sh;
    }
    if (tid < BN) { s_sum[tid] = 0.f; s_sq[tid] = 0.f; }

    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int Q = my_tiles * nch;
    const int c4 = tid & 7, r0 = tid >> 3;
    int iq_t = 0, iq_c = 0, iq_s = 0;          // (tile, chunk, stage) of the next chunk to issue — counters, no div/mod in the loop
    auto issue = [&]() {
        const int ti = iq_t, c = iq_c;
        const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
        const bool seg1 = c < nch1;
        const float* X = seg1 ? a.X1 : a.X2;
        const int C = seg1 ? a.C1 : a.C2;
        const int col = (seg1 ? c : c - nch1) * BK + 4 * c4;
        float* dst = As + iq_s * BM * AST;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = r0 + 32 * j;
            const int64_t m = m0 + r;
            const bool ok = (m < a.M) && (col < C);
            int64_t srow = ok ? m : 0;
            if (ok && seg1 && a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
            cp_async16(dst + r * AST + 4 * c4, X + srow * C + (ok ? col : 0), ok);
        }
        if (++iq_c == nch) { iq_c = 0; ++iq_t; }
        if (++iq_s == NSTT) iq_s = 0;
    };
    for (int s = 0; s < NSTT - 1; ++s) {
        if (s < Q) issue();
        cp_async_commit();
    }

    float acc[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    int ti = 0, c = 0, cs = 0;                 // (tile, chunk, stage) being computed
    for (int q = 0; q < Q; ++q) {
        cp_async_wait<NSTT - 2>();
        __syncthreads();
        if (q + NSTT - 1 < Q) issue();
        cp_async_commit();
        const float* At = As + cs * BM * AST;
        const bool seg1 = c < nch1;
        const int kvalid = seg1 ? min(BK, a.C1 - c * BK) : min(BK, a.C2 - (c - nch1) * BK);
        const float slope = (seg1 && a.scale1) ? a.slope1 : 1.0f;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            if (ks * 8 < kvalid) {
                const int kb = ks * 8;
                uint32_t ah[4], al[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = 16 * w + g + ((i & 1) ? 8 : 0);
                    const int kk = kb + t + ((i & 2) ? 4 : 0);
                    float v = At[row * AST + kk];
                    v = lrelu(fmaf(v, s_sc[c * BK + kk], s_sh[c * BK + kk]), slope);
                    split_trunc(v, ah[i], al[i]);
                }
                const int wb = c * BK + kb + t;
#pragma unroll
                for (int nt = 0; nt < BN / 8; ++nt) {
                    const int wi = (nt * 8 + g) * WS + wb;
                    const float w0 = Wf[wi], w1 = Wf[wi + 4];
                    uint32_t bh0, bl0, bh1, bl1;
                    split_trunc(w0, bh0, bl0);
                    split_trunc(w1, bh1, bl1);
                    mma_tf32(acc[nt], al, bh0, bh1);
                    mma_tf32(acc[nt], ah, bl0, bl1);
                    mma_tf32(acc[nt], ah, bh0, bh1);
                }
            }
        }
        if (c == nch - 1) {
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
            const int64_t row_a = m0 + 16 * w + g, row_b = row_a + 8;
            const bool va = row_a < a.M, vb = row_b < a.M;
#pragma unroll
            for (int nt = 0; nt < BN / 8; ++nt) {
                const int col = nt * 8 + 2 * t;
                float c0 = acc[nt][0], c1 = acc[nt][1], c2 = acc[nt][2], c3 = acc[nt][3];
                acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
                const bool cv = col < a.Cout;
                if (cv) {
                    if (a.bias) { const float b0 = __ldg(a.bias + col), b1 = __ldg(a.bias + col + 1); c0 += b0; c1 += b1; c2 += b0; c3 += b1; }
                    if (va) *reinterpret_cast<float2*>(a.Y + row_a * a.Cout + col) = make_float2(c0, c1);
                    if (vb) *reinterpret_cast<float2*>(a.Y + row_b * a.Cout + col) = make_float2(c2, c3);
                }
                if (a.stats) {
                    float s0 = (va ? c0 : 0.f) + (vb ? c2 : 0.f), s1 = (va ? c1 : 0.f) + (vb ? c3 : 0.f);
                    float q0 = (va ? c0 * c0 : 0.f) + (vb ? c2 * c2 : 0.f), q1 = (va ? c1 * c1 : 0.f) + (vb ? c3 * c3 : 0.f);
#pragma unroll
                    for (int o = 4; o < 32; o <<= 1) {
                        s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                        q0 += __shfl_xor_sync(0xffffffffu, q0, o); q1 += __shfl_xor_sync(0xffffffffu, q1, o);
                    }
                    if (g == 0 && cv) {
                        atomicAdd(&s_sum[col], s0); atomicAdd(&s_sum[col + 1], s1);
                        atomicAdd(&s_sq[col], q0);  atomicAdd(&s_sq[col + 1], q1);
                    }
                }
            }
        }
        if (++c == nch) { c = 0; ++ti; }
        if (++cs == NSTT) cs = 0;
    }
    cp_async_wait<0>();
    if (a.stats) {
        __syncthreads();
        if (tid < BN && tid < a.Cout) {
            float* st = a.stats + (size_t)(blockIdx.x % kStatSlots) * 2 * a.Cout;
            atomicAdd(st + tid, s_sum[tid]);
            atomicAdd(st + a.Cout + tid, s_sq[tid]);
        }
    }
}

template <int BN>
size_t fwd2t_smem(int Kpad) {
    return (size_t)FwdT<BN>::NS * 128 * AST * 4 + (size_t)BN * (Kpad + 4) * 4 + (size_t)2 * Kpad * 4 + (size_t)2 * BN * 4;
}

template <int BN>
size_t fwd2_smem(int Kpad) {
    return (size_t)NST * 128 * AS * 4 + (size_t)2 * BN * ((Kpad + 8) / 2) * 4 + (size_t)2 * Kpad * 4 + (size_t)2 * BN * 4;
}

// ===================================================================================================== dgrad
// dX[M, Ktot] = dH[M, Cout] · W[Cout, Ktot];  dH from (dY, H[, act_ref]) on the fly.  BN = padded Ktot tile (16..128).
// Per-channel constants are pre-combined:  dH = sc·dV + p·h + q,  p = −sc·istd·k2,  q = −sc·k1 + sc·istd·k2·mean.
template <int BN, bool X3, bool REF>
__global__ void __launch_bounds__(kThreads, (BN >= 128 || REF) ? 1 : 2) dgrad2_kernel(const DgradArgs a, const int ntiles) {
    constexpr int WC = BN >= 64 ? 2 : 1, WR = 8 / WC, BM = 16 * WR, NT = BN / WC / 8;
    constexpr int NTILE = REF ? 3 : 2;                       // staged tiles per stage: dY, H (, act_ref)
    constexpr int NST = BN >= 64 ? 3 : 2;                    // shadows the file-level ring depth: 128-row tiles take 2 stages
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int C = a.Cout, nch = (C + BK - 1) / BK, Kpad = nch * BK, WS2 = (Kpad + 8) / 2, Ktot = a.C1 + a.C2;
    float* St = reinterpret_cast<float*>(smem_raw);                          // [NST][NTILE][BM][AS]
    uint32_t* Wh = reinterpret_cast<uint32_t*>(St + NST * NTILE * BM * AS);  // [BN][WS2]  Wt[n = cin][k = cout]
    uint32_t* Wl = Wh + BN * WS2;
    float4* s_par = reinterpret_cast<float4*>(Wl + BN * WS2);                // [Kpad]  (sc, sh, p, q)
    const bool plain = a.bn.scale == nullptr;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int wr = w % WR, wc = w / WR;

    for (int e = tid; e < BN * (Kpad / 2); e += kThreads) {
        const int n = e / (Kpad / 2), kp = 2 * (e % (Kpad / 2));
        float wv[2] = {0.f, 0.f};
#pragma unroll
        for (int u = 0; u < 2; ++u)
            if (kp + u < C && n < Ktot) wv[u] = __ldg(a.W + (int64_t)(kp + u) * Ktot + n);
        uint32_t hi, lo;
        split2(wv[0], wv[1], hi, lo);
        Wh[n * WS2 + kp / 2] = hi;
        Wl[n * WS2 + kp / 2] = lo;
    }
    for (int k = tid; k < Kpad; k += kThreads) s_par[k] = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);

    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int Q = my_tiles * nch;
    constexpr int RPP = kThreads / 8;                      // rows covered per pass of 256 threads (8 float4 per 32-float row)
    const int c4 = tid & 7, r0 = tid >> 3;

    int iq_t = 0, iq_c = 0, iq_s = 0;
    auto issue = [&]() {
        const int ti = iq_t, c = iq_c;
        const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
        const int col = c * BK + 4 * c4;
        float* dst = St + iq_s * NTILE * BM * AS;
#pragma unroll
        for (int j = 0; j < BM / RPP; ++j) {
            const int r = r0 + RPP * j;
            const int64_t m = m0 + r;
            const bool ok = (m < a.M) && (col < C);
            const int64_t off = ok ? m * C + col : 0;
            cp_async16(dst + r * AS + 4 * c4, a.dY + off, ok);
            if (!plain) cp_async16(dst + BM * AS + r * AS + 4 * c4, a.H + off, ok);
            if (REF) cp_async16(dst + 2 * BM * AS + r * AS + 4 * c4, a.bn.act_ref + off, ok);
        }
        if (++iq_c == nch) { iq_c = 0; ++iq_t; }
        if (++iq_s == NST) iq_s = 0;
    };
    for (int s = 0; s < NST - 1; ++s) {
        if (s < Q) issue();
        cp_async_commit();
    }
    float acc[NT][4];
#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const float slope = a.bn.slope;

    int ti = 0, c = 0, cs = 0;
    for (int q = 0; q < Q; ++q) {
        cp_async_wait<NST - 2>();
        __syncthreads();
        if (q + NST - 1 < Q) issue();
        cp_async_commit();
        const float* Dt = St + cs * NTILE * BM * AS;
        const float* Ht = Dt + BM * AS;
        const float* Rt = Dt + 2 * BM * AS;
        const int kvalid = min(BK, C - c * BK);
#pragma unroll
        for (int ks = 0; ks < BK / 16; ++ks) {
            if (ks * 16 < kvalid) {
                const int kb = ks * 16;
                uint32_t ah[4], al[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = 16 * wr + g + ((i & 1) ? 8 : 0);
                    const int kk = kb + 2 * t + ((i & 2) ? 8 : 0);
                    float2 d = *reinterpret_cast<const float2*>(Dt + row * AS + kk);
                    if (!plain) {
                        const float2 h = *reinterpret_cast<const float2*>(Ht + row * AS + kk);
                        const float4 p0 = s_par[c * BK + kk], p1 = s_par[c * BK + kk + 1];
                        float pre0, pre1;
                        if (REF) { const float2 r = *reinterpret_cast<const float2*>(Rt + row * AS + kk); pre0 = r.x; pre1 = r.y; }
                        else { pre0 = fmaf(h.x, p0.x, p0.y); pre1 = fmaf(h.y, p1.x, p1.y); }
                        const float dv0 = pre0 > 0.f ? d.x : d.x * slope, dv1 = pre1 > 0.f ? d.y : d.y * slope;
                        d.x = fmaf(p0.x, dv0, fmaf(p0.z, h.x, p0.w));
                        d.y = fmaf(p1.x, dv1, fmaf(p1.z, h.y, p1.w));
                    }
                    split2(d.x, d.y, ah[i], al[i]);
                }
                const int wb = (c * BK + kb) / 2 + t;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const int wi = (wc * NT * 8 + nt * 8 + g) * WS2 + wb;
                    mma3<X3>(acc[nt], ah, al, Wh[wi], Wh[wi + 4], Wl[wi], Wl[wi + 4]);
                }
            }
        }
        if (c == nch - 1) {
            const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * BM;
            const int64_t row_a = m0 + 16 * wr + g, row_b = row_a + 8;
            const bool va = row_a < a.M, vb = row_b < a.M;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int col = wc * NT * 8 + nt * 8 + 2 * t;     // even; C1 is a multiple of 4 ⇒ the pair stays in one segment
                const float c0 = acc[nt][0], c1 = acc[nt][1], c2 = acc[nt][2], c3 = acc[nt][3];
                acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
                if (col >= Ktot) continue;
                float* dst; int cc, ld, accm;
                if (col < a.C1) { dst = a.dX1; cc = col; ld = a.C1; accm = a.acc1; }
                else            { dst = a.dX2; cc = col - a.C1; ld = a.C2; accm = a.acc2; }
                if (!dst) continue;
                if (va) {
                    float2* p = reinterpret_cast<float2*>(dst + row_a * ld + cc);
                    float2 o = make_float2(c0, c1);
                    if (accm) { const float2 old = *p; o.x += old.x; o.y += old.y; }
                    *p = o;
                }
                if (vb) {
                    float2* p = reinterpret_cast<float2*>(dst + row_b * ld + cc);
                    float2 o = make_float2(c2, c3);
                    if (accm) { const float2 old = *p; o.x += old.x; o.y += old.y; }
                    *p = o;
                }
            }
        }
        if (++c == nch) { c = 0; ++ti; }
        if (++cs == NST) cs = 0;
    }
    cp_async_wait<0>();
}

template <int BN, bool REF>
size_t dgrad2_smem(int Kpad) {
    constexpr int WC = BN >= 64 ? 2 : 1, BM = 16 * (8 / WC), NTILE = REF ? 3 : 2, NSTD = BN >= 64 ? 3 : 2;
    return (size_t)NSTD * NTILE * BM * AS * 4 + (size_t)2 * BN * ((Kpad + 8) / 2) * 4 + (size_t)Kpad * 16;
}

// ===================================================================================================== wgrad
// dW[Cout, Ktot] += dHᵀ·[prologue(X1) | X2].  32-row tiles: cp.async raw tiles → transform pass (dH, activation, bf16 hi/lo
// split, transposed + XOR-swizzled so both the pass's stores and the fragment loads are bank-conflict free) → mma.
// CO = padded Cout (16/32/64), KP = padded Ktot (multiple of 16, <= 128).
constexpr int RT = 32;           // rows per tile
constexpr int TS = RT / 2 + 4;   // row stride (32-bit words = bf16 pairs along m) of transposed operands: 20 = 4·odd

template <int CO, int KP, bool X3, bool REF>
__global__ void __launch_bounds__(kThreads, 2) wgrad2_kernel(const WgradArgs a, const int ntiles) {
    constexpr int WCO = CO / 16, WCI = 8 / WCO, NT = KP / 8 / WCI;       // warp grid over the output, n-tiles per warp
    static_assert(NT >= 1, "output too narrow for the tensor-core wgrad");
    constexpr int DS = CO + 4, XS = KP + 4;                              // raw fp32 row strides
    constexpr int RAW = RT * DS * (REF ? 3 : 2) + RT * XS;               // floats per raw stage
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* raw = reinterpret_cast<float*>(smem_raw);                     // [2][RAW]
    uint32_t* DTh = reinterpret_cast<uint32_t*>(raw + 2 * RAW);          // [CO][TS]
    uint32_t* DTl = DTh + CO * TS;
    uint32_t* XTh = DTl + CO * TS;                                       // [KP][TS]
    uint32_t* XTl = XTh + KP * TS;
    float4* s_par = reinterpret_cast<float4*>(XTl + KP * TS);            // [CO] (sc, sh, p, q)
    float2* s_pro = reinterpret_cast<float2*>(s_par + CO);               // [KP] (scale1, shift1) of the X prologue

    const bool plain = a.bn.scale == nullptr;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int Ktot = a.C1 + a.C2, C = a.Cout;
    const int wco = w % WCO, wci = w / WCO;

    for (int k = tid; k < CO; k += kThreads) s_par[k] = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);
    for (int k = tid; k < KP; k += kThreads) {
        float2 pr = make_float2(1.f, 0.f);
        if (a.scale1 && k < a.C1) pr = make_float2(__ldg(a.scale1 + k), __ldg(a.shift1 + k));
        s_pro[k] = pr;
    }

    const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    auto issue = [&](int ti) {
        const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * RT;
        float* dst = raw + (ti & 1) * RAW;
        // dY / H / ref: RT rows × CO/4 float4
        for (int e = tid; e < RT * (CO / 4); e += kThreads) {
            const int r = e / (CO / 4), c = 4 * (e % (CO / 4));
            const int64_t m = m0 + r;
            const bool ok = (m < a.M) && (c < C);
            const int64_t off = ok ? m * C + c : 0;
            cp_async16(dst + r * DS + c, a.dY + off, ok);
            if (!plain) cp_async16(dst + RT * DS + r * DS + c, a.H + off, ok);
            if (REF) cp_async16(dst + 2 * RT * DS + r * DS + c, a.bn.act_ref + off, ok);
        }
        float* xd = dst + RT * DS * (REF ? 3 : 2);
        for (int e = tid; e < RT * (KP / 4); e += kThreads) {
            const int r = e / (KP / 4), c = 4 * (e % (KP / 4));
            const int64_t m = m0 + r;
            const bool in1 = c < a.C1;
            const bool ok = (m < a.M) && (c < Ktot);
            const float* src = a.X1;
            if (ok) {
                if (in1) {
                    int64_t srow = m;
                    if (a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
                    src = a.X1 + srow * a.C1 + c;
                } else {
                    src = a.X2 + m * a.C2 + (c - a.C1);
                }
            }
            cp_async16(xd + r * XS + c, src, ok);
        }
    };

    float acc[NT][4];
#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const float slope = a.bn.slope, slope1 = a.scale1 ? a.slope1 : 1.0f;

    if (my_tiles > 0) issue(0);
    cp_async_commit();
    for (int ti = 0; ti < my_tiles; ++ti) {
        cp_async_wait<0>();
        __syncthreads();                 // raw[ti&1] landed; previous MMA phase finished reading the transposed operands
        const int64_t m0 = ((int64_t)blockIdx.x + (int64_t)ti * gridDim.x) * RT;
        const float* Dr = raw + (ti & 1) * RAW;
        const float* Hr = Dr + RT * DS;
        const float* Rr = Dr + 2 * RT * DS;
        const float* Xr = Dr + RT * DS * (REF ? 3 : 2);
        if (ti + 1 < my_tiles) issue(ti + 1);
        cp_async_commit();
        // ---- transform pass: pairs of rows (2mp, 2mp+1) per channel → packed bf16 hi / lo, transposed, swizzled
        for (int e = tid; e < (RT / 2) * CO; e += kThreads) {
            const int c = e % CO, mp = e / CO;
            float v[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int r = 2 * mp + u;
                float d = Dr[r * DS + c];
                if (!plain) {
                    const float h = Hr[r * DS + c];
                    const float4 p = s_par[c];
                    const float pre = REF ? Rr[r * DS + c] : fmaf(h, p.x, p.y);
                    const float dv = pre > 0.f ? d : d * slope;
                    d = fmaf(p.x, dv, fmaf(p.z, h, p.w));
                }
                v[u] = (m0 + r < a.M && c < C) ? d : 0.f;
            }
            uint32_t hi, lo;
            split2(v[0], v[1], hi, lo);
            const int wi = c * TS + (mp ^ ((c >> 3) & 3));
            DTh[wi] = hi; DTl[wi] = lo;
        }
        for (int e = tid; e < (RT / 2) * KP; e += kThreads) {
            const int c = e % KP, mp = e / KP;
            const float2 pr = s_pro[c];
            const float sl = c < a.C1 ? slope1 : 1.0f;
            float v[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int r = 2 * mp + u;
                const float x = lrelu(fmaf(Xr[r * XS + c], pr.x, pr.y), sl);
                v[u] = (m0 + r < a.M && c < Ktot) ? x : 0.f;
            }
            uint32_t hi, lo;
            split2(v[0], v[1], hi, lo);
            const int wi = c * TS + (mp ^ ((c >> 3) & 3));
            XTh[wi] = hi; XTl[wi] = lo;
        }
        __syncthreads();
        // ---- tensor-core accumulation: D[co, k] += Σ_m dH[m, co] · X[m, k]
#pragma unroll
        for (int ks = 0; ks < RT / 16; ++ks) {
            uint32_t ah[4], al[4];
            {
                const int ca = wco * 16 + g, cb = ca + 8;
                const int fa = (ca >> 3) & 3, fb = (cb >> 3) & 3;
                const int w0 = ks * 8 + t, w1 = w0 + 4;
                ah[0] = DTh[ca * TS + (w0 ^ fa)]; al[0] = DTl[ca * TS + (w0 ^ fa)];
                ah[1] = DTh[cb * TS + (w0 ^ fb)]; al[1] = DTl[cb * TS + (w0 ^ fb)];
                ah[2] = DTh[ca * TS + (w1 ^ fa)]; al[2] = DTl[ca * TS + (w1 ^ fa)];
                ah[3] = DTh[cb * TS + (w1 ^ fb)]; al[3] = DTl[cb * TS + (w1 ^ fb)];
            }
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int cn = (wci * NT + nt) * 8 + g;
                const int f = (cn >> 3) & 3;
                const int w0 = ks * 8 + t, w1 = w0 + 4;
                mma3<X3>(acc[nt], ah, al, XTh[cn * TS + (w0 ^ f)], XTh[cn * TS + (w1 ^ f)], XTl[cn * TS + (w0 ^ f)], XTl[cn * TS + (w1 ^ f)]);
            }
        }
    }
    cp_async_wait<0>();
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int co = wco * 16 + g + (e >= 2 ? 8 : 0);
            const int k = (wci * NT + nt) * 8 + 2 * t + (e & 1);
            if (co < C && k < Ktot) atomicAdd(a.dW + a.slot_stride * (blockIdx.x % kGradSlots) + (int64_t)co * Ktot + k, acc[nt][e]);
        }
    }
}

template <int CO, int KP, bool REF>
size_t wgrad2_smem() {
    constexpr int DS = CO + 4, XS = KP + 4, RAW = RT * DS * (REF ? 3 : 2) + RT * XS;
    return (size_t)2 * RAW * 4 + (size_t)2 * (CO + KP) * TS * 4 + (size_t)CO * 16 + (size_t)KP * 8;
}

// ---- F×F weight gradients on CUDA cores (launched for F = 32; F = 8 / 16 are narrow_bwd's): dW[a][b] += Σ_m dH[m][a]·X[m][b].  Each thread owns a 4×4 block of the
// output; the (F/4)² block owners are replicated over 256/(F/4)² row groups that take interleaved rows of a 128-row tile.
template <int F, bool REF>
__global__ void __launch_bounds__(kThreads) wgrad_small_kernel(const WgradArgs a, const int ntiles) {
    constexpr int RTS = 128, Q4 = F / 4, OWN = Q4 * Q4, RG = kThreads / OWN;
    __shared__ __align__(16) float Ds[RTS][F];
    __shared__ __align__(16) float Xs[RTS][F];
    __shared__ float red[F * F];
    const bool plain = a.bn.scale == nullptr;
    const int tid = threadIdx.x;
    const int own = tid % OWN, rg = tid / OWN;
    const int a0 = 4 * (own / Q4), b0 = 4 * (own % Q4);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int i = tid; i < F * F; i += kThreads) red[i] = 0.f;
    const float slope = a.bn.slope, slope1 = a.scale1 ? a.slope1 : 1.0f;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t m0 = (int64_t)tile * RTS;
        __syncthreads();
        for (int e = tid; e < RTS * Q4; e += kThreads) {
            const int r = e / Q4, c = 4 * (e % Q4);
            const int64_t m = m0 + r;
            float4 d = make_float4(0.f, 0.f, 0.f, 0.f), x = d;
            if (m < a.M) {
                d = __ldg(reinterpret_cast<const float4*>(a.dY + m * F + c));
                if (!plain) {
                    const float4 h = __ldg(reinterpret_cast<const float4*>(a.H + m * F + c));
                    float4 rf = h;
                    if (REF) rf = __ldg(reinterpret_cast<const float4*>(a.bn.act_ref + m * F + c));
                    float* dp = &d.x; const float* hp = &h.x; const float* rp = &rf.x;
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float sc = __ldg(a.bn.scale + c + u), sh = __ldg(a.bn.shift + c + u), mu = __ldg(a.bn.mean + c + u);
                        const float is = __ldg(a.bn.invstd + c + u), k1 = __ldg(a.bn.k1 + c + u), k2 = __ldg(a.bn.k2 + c + u);
                        const float pre = REF ? rp[u] : fmaf(hp[u], sc, sh);
                        const float dv = pre > 0.f ? dp[u] : dp[u] * slope;
                        dp[u] = sc * (dv - k1 - (hp[u] - mu) * is * k2);
                    }
                }
                int64_t srow = m;
                if (a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
                x = __ldg(reinterpret_cast<const float4*>(a.X1 + srow * F + c));
                if (a.scale1) {
                    float* xp = &x.x;
#pragma unroll
                    for (int u = 0; u < 4; ++u) xp[u] = lrelu(fmaf(xp[u], __ldg(a.scale1 + c + u), __ldg(a.shift1 + c + u)), slope1);
                }
            }
            *reinterpret_cast<float4*>(&Ds[r][c]) = d;
            *reinterpret_cast<float4*>(&Xs[r][c]) = x;
        }
        __syncthreads();
#pragma unroll 4
        for (int r = rg; r < RTS; r += RG) {
            const float4 d = *reinterpret_cast<const float4*>(&Ds[r][a0]);
            const float4 x = *reinterpret_cast<const float4*>(&Xs[r][b0]);
            const float dv[4] = {d.x, d.y, d.z, d.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], xv[j], acc[i][j]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(&red[(a0 + i) * F + b0 + j], acc[i][j]);
    __syncthreads();
    for (int i = tid; i < F * F; i += kThreads) atomicAdd(a.dW + a.slot_stride * (blockIdx.x % kGradSlots) + i, red[i]);
}

}  // namespace lin2

namespace lin {

int try_fwd2(const FwdArgs& a, int precision, cudaStream_t st) {
    using namespace lin2;
    const int Ktot = a.C1 + a.C2;
    if (precision == 1) return kDeclined;                      // explicit TF32 request → generic kernels
    if (a.Cout > 64 || (a.Cout & 3) || Ktot > 128 || (a.C1 & 3) || (a.C2 & 3) || a.C1 == 0) return kDeclined;
    if (!aligned16(a.X1) || (a.C2 && !aligned16(a.X2)) || (reinterpret_cast<uintptr_t>(a.Y) & 7)) return kDeclined;
    const int nch = (a.C1 + BK - 1) / BK + (a.C2 + BK - 1) / BK, Kpad = nch * BK;
    if (Kpad > 160) return kDeclined;
    const int ntiles = (int)ceil_div(a.M, 128);
    auto go = [&](auto bnv) {
        constexpr int BN = decltype(bnv)::value;
        if (precision == 0)              // fp32-grade forward (3xTF32)
            return launch(fwd2t_kernel<BN>, dim3(std::min(ntiles, FwdT<BN>::CTAS * kNumSMs)), dim3(kThreads), fwd2t_smem<BN>(Kpad), st, a, ntiles);
        return launch(fwd2_kernel<BN>, dim3(std::min(ntiles, 2 * kNumSMs)), dim3(kThreads), fwd2_smem<BN>(Kpad), st, a, ntiles);
    };
    if (a.Cout > 32) return go(std::integral_constant<int, 64>{});
    if (a.Cout > 16) return go(std::integral_constant<int, 32>{});
    if (a.Cout > 8) return go(std::integral_constant<int, 16>{});
    return go(std::integral_constant<int, 8>{});
}

int try_dgrad2(const DgradArgs& a, int precision, cudaStream_t st) {
    using namespace lin2;
    const int Ktot = a.C1 + a.C2;
    if (precision == 1) return kDeclined;
    if (a.Cout > 64 || (a.Cout & 3) || Ktot > 128 || Ktot < 8 || (a.C1 & 3) || (a.C2 & 3)) return kDeclined;
    if (!aligned16(a.dY) || (a.bn.scale && !aligned16(a.H)) || (a.bn.act_ref && !aligned16(a.bn.act_ref))) return kDeclined;
    if ((a.dX1 && (reinterpret_cast<uintptr_t>(a.dX1) & 7)) || (a.dX2 && (reinterpret_cast<uintptr_t>(a.dX2) & 7))) return kDeclined;
    const int Kpad = (int)ceil_div(a.Cout, BK) * BK;
    const bool x3 = precision != 2, ref = a.bn.scale && a.bn.act_ref;
    auto go = [&](auto bnv) {
        constexpr int BN = decltype(bnv)::value;
        constexpr int BM = 16 * (8 / (BN >= 64 ? 2 : 1));
        const int ntiles = (int)ceil_div(a.M, BM);
        const dim3 grid(std::min(ntiles, 2 * kNumSMs));
        if (ref) return x3 ? launch(dgrad2_kernel<BN, true, true>, grid, dim3(kThreads), dgrad2_smem<BN, true>(Kpad), st, a, ntiles)
                           : launch(dgrad2_kernel<BN, false, true>, grid, dim3(kThreads), dgrad2_smem<BN, true>(Kpad), st, a, ntiles);
        return x3 ? launch(dgrad2_kernel<BN, true, false>, grid, dim3(kThreads), dgrad2_smem<BN, false>(Kpad), st, a, ntiles)
                  : launch(dgrad2_kernel<BN, false, false>, grid, dim3(kThreads), dgrad2_smem<BN, false>(Kpad), st, a, ntiles);
    };
    if (Ktot > 64) return go(std::integral_constant<int, 128>{});
    if (Ktot > 32) return go(std::integral_constant<int, 64>{});
    if (Ktot > 16) return go(std::integral_constant<int, 32>{});
    if (Ktot > 8) return go(std::integral_constant<int, 16>{});
    return go(std::integral_constant<int, 8>{});
}

int try_wgrad2(const WgradArgs& a, int precision, cudaStream_t st) {
    using namespace lin2;
    const int Ktot = a.C1 + a.C2;
    if (precision == 1 || a.dbias) return kDeclined;
    if (a.Cout > 64 || (a.Cout & 3) || Ktot > 128 || (a.C1 & 3) || (a.C2 & 3) || a.C1 == 0) return kDeclined;
    if (!aligned16(a.dY) || (a.bn.scale && !aligned16(a.H)) || !aligned16(a.X1) || (a.C2 && !aligned16(a.X2))) return kDeclined;
    if (a.bn.act_ref && !aligned16(a.bn.act_ref)) return kDeclined;
    const bool x3 = precision != 2, ref = a.bn.scale && a.bn.act_ref;
    // square hidden-width products (GC, GM, second MLP layers): CUDA-core kernel
    if (a.Cout == 32 && Ktot == 32 && a.C2 == 0) {
        const int ntiles = (int)ceil_div(a.M, 128);
        const dim3 grid(std::min(ntiles, 4 * kNumSMs));
        return ref ? launch(wgrad_small_kernel<32, true>, grid, dim3(kThreads), 0, st, a, ntiles)
                   : launch(wgrad_small_kernel<32, false>, grid, dim3(kThreads), 0, st, a, ntiles);
    }
    const int CO = a.Cout <= 16 ? 16 : (a.Cout <= 32 ? 32 : 64);
    const int KP = Ktot <= 16 ? 16 : (Ktot <= 32 ? 32 : (Ktot <= 64 ? 64 : 128));
    const int ntiles = (int)ceil_div(a.M, RT);
    const dim3 grid(std::min(ntiles, 2 * kNumSMs));
#define CRF_WG(co, kp)                                                                                                                       \
    if (CO == co && KP == kp) {                                                                                                              \
        if (ref) return x3 ? launch(wgrad2_kernel<co, kp, true, true>, grid, dim3(kThreads), wgrad2_smem<co, kp, true>(), st, a, ntiles)     \
                           : launch(wgrad2_kernel<co, kp, false, true>, grid, dim3(kThreads), wgrad2_smem<co, kp, true>(), st, a, ntiles);   \
        return x3 ? launch(wgrad2_kernel<co, kp, true, false>, grid, dim3(kThreads), wgrad2_smem<co, kp, false>(), st, a, ntiles)            \
                  : launch(wgrad2_kernel<co, kp, false, false>, grid, dim3(kThreads), wgrad2_smem<co, kp, false>(), st, a, ntiles);          \
    }
    CRF_WG(64, 128) CRF_WG(64, 64) CRF_WG(64, 32) CRF_WG(64, 16)
    CRF_WG(32, 128) CRF_WG(32, 64) CRF_WG(32, 32)
    CRF_WG(16, 128) CRF_WG(16, 64)
#undef CRF_WG
    return kDeclined;
}

}  // namespace lin
}  // namespace crf
