// Linear forward / input gradient for FEW rows and WIDE channels — the deep levels of PointConvResNet (models/point_conv_big.py:
// 116-128: 160-2,560 points per cloud, 128-512 channels).  The generic kernels (linear.cu) tile 128 rows per CTA and reload every
// 32-wide reduction chunk synchronously: a 960-row, 512→128 layer ran on 16 CTAs with 16 exposed global round trips each (80-90 us
// for 2.5 MB of data; 27 + 21 such launches were 1.8 ms of a 9.4 ms step).  Here the row tile is 32 (4× the CTAs), the next chunk's
// global loads are issued into registers before the current chunk's MMAs (one exposed round trip per CTA instead of one per
// chunk), and the BatchNorm-backward constants of the input gradient are folded once per CTA into shared memory.
// Same contracts as lin::fwd_kernel / lin::dgrad_kernel (linear_args.cuh); 3xTF32; channel counts must be multiples of 4.
#include <algorithm>
#include <cstdlib>

#include "../../include/crfconv_b200.h"
#include "common.cuh"
#include "linear_args.cuh"
#include "mma.cuh"

namespace crf {
namespace lin {
namespace sm {

constexpr int kThreads = 256;
constexpr int BM = 32, BK = 32, AS = BK + 4;

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// ------------------------------------------------------------------------------------------------------------------ forward
// CTA tile: 32 rows × BN output channels; warp w: rows 16·(w & 1).., channels (w >> 1)·(BN / 4)..
template <int BN>
__global__ void __launch_bounds__(kThreads) fwd_small_kernel(const FwdArgs a) {
    constexpr int NT = BN / 32;                                  // n-tiles (8 columns) per warp
    constexpr int WPT = BN * 8 / kThreads;                       // float4 of the weight chunk per thread
    __shared__ __align__(16) float As[BM][AS];
    __shared__ __align__(16) float Ws[BN][AS];
    __shared__ float s_part[2][2][BN];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int wr = (w & 1) * 16, wc = (w >> 1) * (BN / 4);
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int Ktot = a.C1 + a.C2;
    const int nch1 = (a.C1 + BK - 1) / BK, nch = nch1 + (a.C2 + BK - 1) / BK;
    const int c4 = tid & 7, r = tid >> 3;
    const int64_t m = m0 + r;
    int64_t srow1 = m;
    if (a.idx1 && m < a.M) srow1 = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);

    float acc[NT][4];
#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

    float4 ra, rw[WPT], rsc, rsh;
    bool rpro = false;
    auto gload = [&](int i) {
        const bool seg1 = i < nch1;
        const int kc = (seg1 ? i : i - nch1) * BK, C = seg1 ? a.C1 : a.C2, coloff = seg1 ? 0 : a.C1;
        const int k = kc + 4 * c4;
        ra = make_float4(0.f, 0.f, 0.f, 0.f);
        rpro = seg1 && a.scale1 != nullptr && k < C;
        if (m < a.M && k < C) ra = ldg4((seg1 ? a.X1 + srow1 * C : a.X2 + m * C) + k);
        if (rpro) { rsc = ldg4(a.scale1 + k); rsh = ldg4(a.shift1 + k); }
#pragma unroll
        for (int j = 0; j < WPT; ++j) {
            const int q = tid + j * kThreads, n = q >> 3, kk = 4 * (q & 7);
            rw[j] = (n0 + n < a.Cout && kc + kk < C) ? ldg4(a.W + (int64_t)(n0 + n) * Ktot + coloff + kc + kk) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto sstore = [&]() {
        float4 v = ra;
        if (rpro && m < a.M) {
            v.x = lrelu(fmaf(v.x, rsc.x, rsh.x), a.slope1); v.y = lrelu(fmaf(v.y, rsc.y, rsh.y), a.slope1);
            v.z = lrelu(fmaf(v.z, rsc.z, rsh.z), a.slope1); v.w = lrelu(fmaf(v.w, rsc.w, rsh.w), a.slope1);
        }
        *reinterpret_cast<float4*>(&As[r][4 * c4]) = v;
#pragma unroll
        for (int j = 0; j < WPT; ++j) {
            const int q = tid + j * kThreads;
            *reinterpret_cast<float4*>(&Ws[q >> 3][4 * (q & 7)]) = rw[j];
        }
    };
    gload(0);
    for (int i = 0; i < nch; ++i) {
        sstore();
        __syncthreads();
        if (i + 1 < nch) gload(i + 1);                           // in flight during this chunk's MMAs
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {                    // channels beyond the segment are zeros in both operands
            const float af[4] = {As[wr + g][ks * 8 + t], As[wr + g + 8][ks * 8 + t], As[wr + g][ks * 8 + t + 4], As[wr + g + 8][ks * 8 + t + 4]};
            FragA fa;
            make_frag_a<true>(fa, af);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                FragB fb;
                make_frag_b<true>(fb, Ws[wc + nt * 8 + g][ks * 8 + t], Ws[wc + nt * 8 + g][ks * 8 + t + 4]);
                mma_frag<true>(acc[nt], fa, fb);
            }
        }
        __syncthreads();
    }
    const int64_t row_a = m0 + wr + g, row_b = row_a + 8;
    const bool va = row_a < a.M, vb = row_b < a.M;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const int lc = wc + nt * 8 + 2 * t, col = n0 + lc;
        float c0 = acc[nt][0], c1 = acc[nt][1], c2 = acc[nt][2], c3 = acc[nt][3];
        if (a.bias) {
            const float b0 = col < a.Cout ? __ldg(a.bias + col) : 0.f, b1 = col + 1 < a.Cout ? __ldg(a.bias + col + 1) : 0.f;
            c0 += b0; c1 += b1; c2 += b0; c3 += b1;
        }
        if (col + 1 < a.Cout) {                                  // Cout % 4 == 0 ⇒ pairs never straddle the edge
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
            if (g == 0) {
                s_part[w & 1][0][lc] = s0; s_part[w & 1][0][lc + 1] = s1;
                s_part[w & 1][1][lc] = q0; s_part[w & 1][1][lc + 1] = q1;
            }
        }
    }
    if (a.stats) {
        __syncthreads();
        if (tid < BN && n0 + tid < a.Cout) {
            float* st = a.stats + (size_t)(blockIdx.x % kStatSlots) * 2 * a.Cout;
            atomicAdd(st + n0 + tid, s_part[0][0][tid] + s_part[1][0][tid]);
            atomicAdd(st + a.Cout + n0 + tid, s_part[0][1][tid] + s_part[1][1][tid]);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------- input gradient
// dX[m, n] (+)= Σ_c dH[m, c]·W[c, n];  CTA tile: 32 rows × BN input channels, contraction over the Cout channels in chunks of 32.
template <int BN, bool REF>
__global__ void __launch_bounds__(kThreads) dgrad_small_kernel(const DgradArgs a) {
    constexpr int NT = BN / 32, WPT = BN * 8 / kThreads, BS8 = 8;
    extern __shared__ __align__(16) float4 s_par[];              // [Cout] (sc, sh, −sc·istd·k2, −sc·k1 + sc·istd·k2·mu)
    __shared__ __align__(16) float As[BM][AS];
    __shared__ __align__(16) float Ws[BK][BN + BS8];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int wr = (w & 1) * 16, wc = (w >> 1) * (BN / 4);
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int Ktot = a.C1 + a.C2, C = a.Cout;
    const bool plain = a.bn.scale == nullptr;
    if (!plain)
        for (int k = tid; k < C; k += kThreads) s_par[k] = a.bn.coef(k);
    const int c4 = tid & 7, r = tid >> 3;
    const int64_t m = m0 + r;
    const int nch = (C + BK - 1) / BK;
    float acc[NT][4];
#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    float4 rd, rh, rr, rw[WPT];
    auto gload = [&](int i) {
        const int kc = i * BK, k = kc + 4 * c4;
        rd = rh = rr = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < a.M && k < C) {
            rd = ldg4(a.dY + m * C + k);
            if (!plain) rh = ldg4(a.H + m * C + k);
            if (REF) rr = ldg4(a.bn.act_ref + m * C + k);
        }
#pragma unroll
        for (int j = 0; j < WPT; ++j) {
            const int q = tid + j * kThreads, kk = q / (BN / 4), n = 4 * (q % (BN / 4));
            rw[j] = (kc + kk < C && n0 + n < Ktot) ? ldg4(a.W + (int64_t)(kc + kk) * Ktot + n0 + n) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto sstore = [&](int i) {
        float4 v = rd;
        const int k = i * BK + 4 * c4;
        if (!plain && m < a.M && k < C) {
            const float dy[4] = {rd.x, rd.y, rd.z, rd.w}, h[4] = {rh.x, rh.y, rh.z, rh.w}, rf[4] = {rr.x, rr.y, rr.z, rr.w};
            float o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float4 p = s_par[k + e];
                const float pre = REF ? rf[e] : fmaf(h[e], p.x, p.y);
                const float dv = pre > 0.f ? dy[e] : dy[e] * a.bn.slope;
                o[e] = fmaf(p.x, dv, fmaf(p.z, h[e], p.w));
            }
            v = make_float4(o[0], o[1], o[2], o[3]);
        }
        *reinterpret_cast<float4*>(&As[r][4 * c4]) = v;
#pragma unroll
        for (int j = 0; j < WPT; ++j) {
            const int q = tid + j * kThreads;
            *reinterpret_cast<float4*>(&Ws[q / (BN / 4)][4 * (q % (BN / 4))]) = rw[j];
        }
    };
    gload(0);
    __syncthreads();                                             // s_par visible
    for (int i = 0; i < nch; ++i) {
        sstore(i);
        __syncthreads();
        if (i + 1 < nch) gload(i + 1);
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            const float af[4] = {As[wr + g][ks * 8 + t], As[wr + g + 8][ks * 8 + t], As[wr + g][ks * 8 + t + 4], As[wr + g + 8][ks * 8 + t + 4]};
            FragA fa;
            make_frag_a<true>(fa, af);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                FragB fb;
                make_frag_b<true>(fb, Ws[ks * 8 + t][wc + nt * 8 + g], Ws[ks * 8 + t + 4][wc + nt * 8 + g]);
                mma_frag<true>(acc[nt], fa, fb);
            }
        }
        __syncthreads();
    }
    const int64_t row_a = m0 + wr + g, row_b = row_a + 8;
    const bool va = row_a < a.M, vb = row_b < a.M;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const int col = n0 + wc + nt * 8 + 2 * t;               // C1, C2 % 4 == 0 ⇒ the pair (col, col + 1) lies in one segment
        if (col >= Ktot) continue;
        float* dst; int cc, ld, accm;
        if (col < a.C1) { dst = a.dX1; cc = col; ld = a.C1; accm = a.acc1; }
        else            { dst = a.dX2; cc = col - a.C1; ld = a.C2; accm = a.acc2; }
        if (!dst) continue;
        if (va) {
            float2* p = reinterpret_cast<float2*>(dst + row_a * ld + cc);
            float2 o = make_float2(acc[nt][0], acc[nt][1]);
            if (accm) { const float2 old = *p; o.x += old.x; o.y += old.y; }
            *p = o;
        }
        if (vb) {
            float2* p = reinterpret_cast<float2*>(dst + row_b * ld + cc);
            float2 o = make_float2(acc[nt][2], acc[nt][3]);
            if (accm) { const float2 old = *p; o.x += old.x; o.y += old.y; }
            *p = o;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------- weight gradient
// dW[co, k] += Σ_m dH[m, co]·A[m, k] for few rows and a WIDE output (e.g. 512 × 256 at 960 rows): 64 × 64 output tile per CTA, the
// rows split over blockIdx.x in 32-row steps with the next step's dH / A float4s prefetched into registers (the generic kernel
// reloads 64-row tiles synchronously with scalar, per-element-guarded loads: 35-65 us for ≈4 MB).  Partial tiles meet in the
// kGradSlots slots (or directly in dW) through fp32 atomics, like lin::wgrad_kernel.
template <bool REF>
__global__ void __launch_bounds__(kThreads) wgrad_rows_kernel(const WgradArgs a) {
    constexpr int WS = 64 + 8;
    __shared__ __align__(16) float Ds[BM][WS];                   // dH rows   [m][co]
    __shared__ __align__(16) float Xs[BM][WS];                   // A rows    [m][k]
    __shared__ float4 s_par[64];
    __shared__ float2 s_pro[64];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int Ktot = a.C1 + a.C2, C = a.Cout;
    const int co0 = blockIdx.y * 64, k0 = blockIdx.z * 64;
    const int64_t mbeg = (int64_t)blockIdx.x * a.rows_per_cta, mend = min(a.M, mbeg + a.rows_per_cta);
    const bool plain = a.bn.scale == nullptr;
    if (tid < 64) {
        const int k = co0 + tid;
        s_par[tid] = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);
        float2 pp = make_float2(1.f, 0.f);
        const int kk = k0 + tid;
        if (a.scale1 && kk < a.C1) pp = make_float2(__ldg(a.scale1 + kk), __ldg(a.shift1 + kk));
        s_pro[tid] = pp;
    }
    const int wr = (w & 3) * 16, wc = (w >> 2) * 32;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) acc[i][jj] = 0.0f;
    const int c16 = tid & 15, rr = tid >> 4;                      // 16 float4 per 64-wide row, 16 rows per pass, 2 passes per step
    const int cD = co0 + 4 * c16, cX = k0 + 4 * c16;
    const bool okD = cD < C, okX = cX < Ktot, seg1 = cX < a.C1;
    float4 rd[2], rh[2], rf[2], rx[2];
    bool rok[2];
    auto gload = [&](int64_t mt) {
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
            const int64_t m = mt + rr + 16 * jj;
            rok[jj] = m < mend;
            rd[jj] = rh[jj] = rf[jj] = rx[jj] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (rok[jj] && okD) {
                rd[jj] = ldg4(a.dY + m * C + cD);
                if (!plain) rh[jj] = ldg4(a.H + m * C + cD);
                if (REF) rf[jj] = ldg4(a.bn.act_ref + m * C + cD);
            }
            if (rok[jj] && okX) {
                if (seg1) {
                    int64_t srow = m;
                    if (a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
                    rx[jj] = ldg4(a.X1 + srow * a.C1 + cX);
                } else {
                    rx[jj] = ldg4(a.X2 + m * a.C2 + (cX - a.C1));
                }
            }
        }
    };
    auto sstore = [&]() {
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
            const int r = rr + 16 * jj;
            float4 d = rd[jj];
            if (!plain && rok[jj] && okD) {
                const float dy[4] = {rd[jj].x, rd[jj].y, rd[jj].z, rd[jj].w}, h[4] = {rh[jj].x, rh[jj].y, rh[jj].z, rh[jj].w};
                const float ref[4] = {rf[jj].x, rf[jj].y, rf[jj].z, rf[jj].w};
                float o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 p = s_par[4 * c16 + e];
                    const float pre = REF ? ref[e] : fmaf(h[e], p.x, p.y);
                    const float dv = pre > 0.f ? dy[e] : dy[e] * a.bn.slope;
                    o[e] = fmaf(p.x, dv, fmaf(p.z, h[e], p.w));
                }
                d = make_float4(o[0], o[1], o[2], o[3]);
            }
            *reinterpret_cast<float4*>(&Ds[r][4 * c16]) = d;
            float4 x = rx[jj];
            if (a.scale1 && seg1 && rok[jj] && okX) {
                const float2 p0 = s_pro[4 * c16], p1 = s_pro[4 * c16 + 1], p2 = s_pro[4 * c16 + 2], p3 = s_pro[4 * c16 + 3];
                x = make_float4(lrelu(fmaf(x.x, p0.x, p0.y), a.slope1), lrelu(fmaf(x.y, p1.x, p1.y), a.slope1),
                                lrelu(fmaf(x.z, p2.x, p2.y), a.slope1), lrelu(fmaf(x.w, p3.x, p3.y), a.slope1));
            }
            *reinterpret_cast<float4*>(&Xs[r][4 * c16]) = x;
        }
    };
    gload(mbeg);
    __syncthreads();                                              // s_par / s_pro visible
    for (int64_t mt = mbeg; mt < mend; mt += BM) {
        sstore();
        __syncthreads();
        if (mt + BM < mend) gload(mt + BM);
#pragma unroll
        for (int ks = 0; ks < BM / 8; ++ks) {
            const float af[4] = {Ds[ks * 8 + t][wr + g], Ds[ks * 8 + t][wr + g + 8], Ds[ks * 8 + t + 4][wr + g], Ds[ks * 8 + t + 4][wr + g + 8]};
            FragA fa;
            make_frag_a<true>(fa, af);
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                FragB fb;
                make_frag_b<true>(fb, Xs[ks * 8 + t][wc + nt * 8 + g], Xs[ks * 8 + t + 4][wc + nt * 8 + g]);
                mma_frag<true>(acc[nt], fa, fb);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int co = co0 + wr + g + (e >= 2 ? 8 : 0), k = k0 + wc + nt * 8 + 2 * t + (e & 1);
            if (co < C && k < Ktot) atomicAdd(a.dW + a.slot_stride * (blockIdx.x % kGradSlots) + (int64_t)co * Ktot + k, acc[nt][e]);
        }
}

// rows at which the 128-row tiling of the generic kernels still fills the machine
inline bool few_rows(int64_t M, int ntiles_n) { return ceil_div(M, (int64_t)128) * ntiles_n < 2 * kNumSMs; }

}  // namespace sm

int try_fwd_small(const FwdArgs& a, cudaStream_t st) {
    using namespace sm;
    const int Ktot = a.C1 + a.C2;
    if (a.Cout < 32 || (a.Cout & 3) || (a.C1 & 3) || (a.C2 & 3) || a.C1 <= 0 || Ktot < 32) return kDeclined;
    if (!aligned16(a.X1) || (a.C2 && !aligned16(a.X2)) || !aligned16(a.W) || !aligned16(a.Y) ||
        (a.scale1 && (!aligned16(a.scale1) || !aligned16(a.shift1)))) return kDeclined;
    const int BN = a.Cout > 32 ? 64 : 32;
    const int tn = (int)ceil_div(a.Cout, BN);
    if (!few_rows(a.M, tn)) return kDeclined;
    const dim3 grid((unsigned)ceil_div(a.M, (int64_t)BM), (unsigned)tn);
    return launch(BN == 64 ? fwd_small_kernel<64> : fwd_small_kernel<32>, grid, dim3(kThreads), 0, st, a);
}

int try_dgrad_small(const DgradArgs& a, cudaStream_t st) {
    using namespace sm;
    const int Ktot = a.C1 + a.C2;
    if (Ktot < 32 || (a.Cout & 3) || (a.C1 & 3) || (a.C2 & 3) || a.Cout < 32 || a.Cout > 1024) return kDeclined;
    if (!aligned16(a.dY) || !aligned16(a.W) || (a.bn.scale && !aligned16(a.H)) || (a.bn.scale && a.bn.act_ref && !aligned16(a.bn.act_ref))) return kDeclined;
    if ((a.dX1 && (reinterpret_cast<uintptr_t>(a.dX1) & 7)) || (a.dX2 && (reinterpret_cast<uintptr_t>(a.dX2) & 7))) return kDeclined;
    const int BN = Ktot > 32 ? 64 : 32;
    const int tn = (int)ceil_div(Ktot, BN);
    if (!few_rows(a.M, tn)) return kDeclined;
    const dim3 grid((unsigned)ceil_div(a.M, (int64_t)BM), (unsigned)tn);
    const size_t smem = a.bn.scale ? (size_t)a.Cout * sizeof(float4) : 0;
    const bool ref = a.bn.scale && a.bn.act_ref;
    if (BN == 64) return launch(ref ? dgrad_small_kernel<64, true> : dgrad_small_kernel<64, false>, grid, dim3(kThreads), smem, st, a);
    return launch(ref ? dgrad_small_kernel<32, true> : dgrad_small_kernel<32, false>, grid, dim3(kThreads), smem, st, a);
}

int try_wgrad_rows(WgradArgs a, cudaStream_t st) {
    using namespace sm;
    const int Ktot = a.C1 + a.C2;
    if (a.dbias || (a.Cout & 3) || (a.C1 & 3) || (a.C2 & 3) || a.C1 <= 0 || a.Cout < 32 || Ktot < 32) return kDeclined;
    if (!aligned16(a.dY) || !aligned16(a.X1) || (a.C2 && !aligned16(a.X2)) || (a.bn.scale && !aligned16(a.H)) ||
        (a.bn.scale && a.bn.act_ref && !aligned16(a.bn.act_ref))) return kDeclined;
    const int ty = (int)ceil_div(a.Cout, 64), tz = (int)ceil_div(Ktot, 64);
    if (!few_rows(a.M, 1)) return kDeclined;
    int64_t splits = std::max<int64_t>(1, std::min<int64_t>(ceil_div(a.M, (int64_t)BM), (int64_t)(3 * kNumSMs) / (ty * tz) + 1));
    a.rows_per_cta = ceil_div(ceil_div(a.M, splits), (int64_t)BM) * BM;
    splits = ceil_div(a.M, a.rows_per_cta);
    const dim3 grid((unsigned)splits, (unsigned)ty, (unsigned)tz);
    return launch(a.bn.scale && a.bn.act_ref ? wgrad_rows_kernel<true> : wgrad_rows_kernel<false>, grid, dim3(kThreads), 0, st, a);
}

}  // namespace lin
}  // namespace crf
