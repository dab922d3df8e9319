// Weight gradients of NARROW layers over MANY rows:  dW[Cout, Ktot] += dHᵀ·[prologue(X1) | X2],  Cout·Ktot small, M large.
//
// The network's level-0 layers (245,760 points, models/point_conv_big.py:61-88,130-140) are Linear(6→8), (6→32), (8→32), (32→8),
// (32→16), (32→128), (128→13): their weight gradients read 40-160 floats per row and produce a few hundred numbers.  The tiled
// kernels (linear.cu wgrad_kernel: 64×64 output tile, unpipelined shared-memory staging; linear2.cu wgrad2_kernel: needs ≥ 8
// warps' worth of output) ran them at 0.3-1.3 TB/s — 125-250 us each, 1.7 ms of an 11 ms step.  Here nothing is staged: both MMA
// operands of the contraction over rows come straight from global memory in fragment order (4-byte "transposed" loads: the 8 lanes
// of a fragment column read one 32-byte sector, every element is fetched exactly once), the BatchNorm-backward transform
//     dH = sc·(dV − k1 − (H − mu)·istd·k2),   dV = dY·lrelu'(sc·H + sh)
// and the input prologue lrelu(x·s1 + t1) are applied in registers, and each warp owns whole 16-row tiles, so there is no
// CTA-wide barrier in the stream.  3xTF32 (fp32-grade).  Same scheme as cl::in16_wgrad_kernel (crf_fused.cu), for any
// Cout ≤ 128 (MB blocks of 16) and Ktot ≤ 128 (NB blocks of 8) with MB·NB ≤ 32 accumulator blocks.
#include <algorithm>
#include <cstdlib>

#include "../../include/crfconv_b200.h"
#include "common.cuh"
#include "fused_common.cuh"
#include "linear_args.cuh"

namespace crf {
namespace lin {
namespace dw {

constexpr int kThreads = 256, kWarps = 8;

template <int MB, int NB>
__global__ void __launch_bounds__(kThreads, MB * NB > 4 ? 1 : 2) wgrad_direct_kernel(const WgradArgs a) {
    constexpr int CO = 16 * MB, KP = 8 * NB;
    constexpr bool TWO = (8 * MB + 2 * NB) <= 40;              // both 8-row k-steps of a tile loaded before the first MMA
    constexpr int KSB = TWO ? 2 : 1;
    __shared__ float s_w[CO * KP];
    __shared__ float4 s_par[CO];                                // (sc, sh, −sc·istd·k2, −sc·k1 + sc·istd·k2·mu)
    __shared__ float2 s_pro[KP];
    __shared__ float s_b[CO];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int C = a.Cout, Ktot = a.C1 + a.C2;
    const bool plain = a.bn.scale == nullptr;
    for (int i = tid; i < CO * KP; i += kThreads) s_w[i] = 0.f;
    for (int k = tid; k < CO; k += kThreads) {
        s_par[k] = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);
        s_b[k] = 0.f;
    }
    for (int k = tid; k < KP; k += kThreads) {
        float2 pr = make_float2(1.f, 0.f);
        if (a.scale1 && k < a.C1) pr = make_float2(__ldg(a.scale1 + k), __ldg(a.shift1 + k));
        s_pro[k] = pr;
    }
    __syncthreads();
    const float slope = a.bn.slope, slope1 = a.scale1 ? a.slope1 : 1.0f;
    const bool pro = a.scale1 != nullptr;
    float acc[MB][NB][4];
    float bs[MB][2];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb) {
        bs[mb][0] = bs[mb][1] = 0.f;
#pragma unroll
        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[mb][nb][e] = 0.f;
    }
    const int64_t ntiles = (a.M + 15) >> 4;
    for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < ntiles; tile += (int64_t)gridDim.x * kWarps) {
#pragma unroll
        for (int k0 = 0; k0 < 2; k0 += KSB) {
            float tv[KSB][MB][4], th[KSB][MB][4], xa[KSB][NB], xb[KSB][NB];
            bool oka[KSB], okb[KSB];
#pragma unroll
            for (int kk = 0; kk < KSB; ++kk) {
                const int64_t ra = tile * 16 + 8 * (k0 + kk) + t, rb = ra + 4;
                oka[kk] = ra < a.M; okb[kk] = rb < a.M;
#pragma unroll
                for (int mb = 0; mb < MB; ++mb)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {                // fragment order: (co, ra), (co + 8, ra), (co, rb), (co + 8, rb)
                        const int co = 16 * mb + g + 8 * (q & 1);
                        const bool ok = ((q & 2) ? okb[kk] : oka[kk]) && co < C;
                        const int64_t off = ((q & 2) ? rb : ra) * C + co;
                        tv[kk][mb][q] = ok ? __ldg(a.dY + off) : 0.f;
                        th[kk][mb][q] = (ok && !plain) ? __ldg(a.H + off) : 0.f;
                    }
                int64_t sa = ra, sb = rb;
                if (a.idx1) {                                   // segment 1 rows gathered: src = (m / rows_dst)·rows_src + idx1[m]
                    if (oka[kk]) sa = (ra / a.rows_dst) * a.rows_src + __ldg(a.idx1 + ra);
                    if (okb[kk]) sb = (rb / a.rows_dst) * a.rows_src + __ldg(a.idx1 + rb);
                }
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) {
                    const int col = nb * 8 + g;
                    float va = 0.f, vb = 0.f;
                    if (col < a.C1) {
                        if (oka[kk]) va = __ldg(a.X1 + sa * a.C1 + col);
                        if (okb[kk]) vb = __ldg(a.X1 + sb * a.C1 + col);
                    } else if (col < Ktot) {
                        if (oka[kk]) va = __ldg(a.X2 + ra * a.C2 + (col - a.C1));
                        if (okb[kk]) vb = __ldg(a.X2 + rb * a.C2 + (col - a.C1));
                    }
                    xa[kk][nb] = va; xb[kk][nb] = vb;
                }
            }
#pragma unroll
            for (int kk = 0; kk < KSB; ++kk) {
                cl::FragB b[NB];
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) {
                    float va = xa[kk][nb], vb = xb[kk][nb];
                    if (pro) {
                        const int col = nb * 8 + g;
                        const float2 pr = s_pro[col];
                        const float sl = col < a.C1 ? slope1 : 1.0f;
                        va = (oka[kk] && col < Ktot) ? cl::lrelu(fmaf(va, pr.x, pr.y), sl) : 0.f;
                        vb = (okb[kk] && col < Ktot) ? cl::lrelu(fmaf(vb, pr.x, pr.y), sl) : 0.f;
                    }
                    cl::make_b(b[nb], va, vb);
                }
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) {
                    float av[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float d = tv[kk][mb][q];
                        if (!plain) {
                            const int co = 16 * mb + g + 8 * (q & 1);
                            const bool ok = ((q & 2) ? okb[kk] : oka[kk]) && co < C;
                            const float4 p = s_par[co];
                            const float h = th[kk][mb][q];
                            const float dv = fmaf(h, p.x, p.y) > 0.f ? d : d * slope;
                            d = ok ? fmaf(p.x, dv, fmaf(p.z, h, p.w)) : 0.f;
                        }
                        av[q] = d;
                    }
                    bs[mb][0] += av[0] + av[2];
                    bs[mb][1] += av[1] + av[3];
                    cl::FragA f;
                    cl::make_a(f, av[0], av[1], av[2], av[3]);
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) cl::mma3(acc[mb][nb], f, b[nb]);
                }
            }
        }
    }
#pragma unroll
    for (int mb = 0; mb < MB; ++mb) {
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
            float* w0 = &s_w[(16 * mb + g) * KP + nb * 8 + 2 * t];
            atomicAdd(w0, acc[mb][nb][0]);
            atomicAdd(w0 + 1, acc[mb][nb][1]);
            atomicAdd(w0 + 8 * KP, acc[mb][nb][2]);
            atomicAdd(w0 + 8 * KP + 1, acc[mb][nb][3]);
        }
        if (a.dbias) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                float v = bs[mb][e];
                v += __shfl_xor_sync(0xffffffffu, v, 1);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                if (t == 0) atomicAdd(&s_b[16 * mb + g + 8 * e], v);
            }
        }
    }
    __syncthreads();
    float* dst = a.dW + a.slot_stride * (int64_t)(blockIdx.x % kGradSlots);
    for (int i = tid; i < CO * KP; i += kThreads) {
        const int co = i / KP, k = i % KP;
        if (co < C && k < Ktot) atomicAdd(dst + (int64_t)co * Ktot + k, s_w[i]);
    }
    if (a.dbias)
        for (int i = tid; i < C; i += kThreads) atomicAdd(a.dbias + i, s_b[i]);
}

template <int MB, int NB>
inline int run(const WgradArgs& a, cudaStream_t st) {
    constexpr int per_sm = MB * NB > 4 ? 1 : 2;
    const int64_t tiles = ceil_div(a.M, 16);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(tiles, kWarps), (int64_t)kNumSMs * per_sm));
    return launch(wgrad_direct_kernel<MB, NB>, dim3(grid), dim3(kThreads), 0, st, a);
}

}  // namespace dw

int try_wgrad_direct(const WgradArgs& a, cudaStream_t st) {
    const int Ktot = a.C1 + a.C2;
    if (a.bn.scale && a.bn.act_ref) return kDeclined;           // saved-activation branch selection: tiled kernels
    if (a.Cout < 1 || a.Cout > 128 || Ktot < 1 || Ktot > 128 || a.C1 < 1 || a.M < 1) return kDeclined;
    const int mb = a.Cout <= 16 ? 1 : (a.Cout <= 32 ? 2 : (a.Cout <= 64 ? 4 : 8));
    const int nb = Ktot <= 8 ? 1 : (Ktot <= 16 ? 2 : (Ktot <= 32 ? 4 : (Ktot <= 64 ? 8 : 16)));
    if (mb * nb > 32) return kDeclined;
#define CRF_DW(m, n) \
    if (mb == m && nb == n) return dw::run<m, n>(a, st);
    CRF_DW(1, 1) CRF_DW(1, 2) CRF_DW(1, 4) CRF_DW(1, 8) CRF_DW(1, 16)
    CRF_DW(2, 1) CRF_DW(2, 2) CRF_DW(2, 4) CRF_DW(2, 8) CRF_DW(2, 16)
    CRF_DW(4, 1) CRF_DW(4, 2) CRF_DW(4, 4) CRF_DW(4, 8)
    CRF_DW(8, 1) CRF_DW(8, 2) CRF_DW(8, 4)
#undef CRF_DW
    return kDeclined;
}

}  // namespace lin
}  // namespace crf

// =====================================================================================================================================
// "Up-projection" passes:  Y[M, N] = act(A[M, K])·B,  K <= 32 narrow, N = 32 / 64 / 128 wide, M large — the pass is a pure stream of
// its OUTPUT (classifier MLP(32→128) forward: 31 MB in, 126 MB out; the 13-class head's input gradient dX = dY[M,13]·W[13,128]).
// Same scheme as cl::up16_fwd_kernel (K = 16 → 64): A fragments straight from global memory (natural m16n8k8 layout, 4-byte loads: A is
// the small operand), pre-split B fragments in shared memory with the output columns permuted (phys_col) so that a lane owns 4
// consecutive channels of a row ⇒ 128-bit stores, Σ / Σ² per column kept in registers over all the warp's tiles.  3xTF32.
namespace crf {
namespace lin {
namespace up {

constexpr int kThreads = 256, kWarps = 8;

__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 fma4(float4 a, float4 b, float4 c) {
    return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
}
__device__ __forceinline__ float group8_sum(float v) {          // sum over the 8 lanes that share lane & 3
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return v;
}

struct UpArgs {
    const float* A; int K; int lda;                           // [M, K] rows lda floats apart
    const float* ps; const float* pt; float pslope;           // optional prologue lrelu(a·ps[k] + pt[k]) (null = identity)
    const float* B; int sbn, sbk;                             // B(k, n) = B[n·sbn + k·sbk]   (forward: W[n][k]; input gradient: W[k][n])
    const float* bias;                                        // [N] or null
    float* Y; int N;                                          // [M, N]
    float* stats;                                             // [kStatSlots][2N] or null
    int64_t M;
};

template <int KP, int NP>
__global__ void __launch_bounds__(kThreads, NP > 64 ? 1 : 2) upproj_kernel(const UpArgs a) {
    constexpr int KS = KP / 8, NB = NP / 8, NQ = NP / 16;
    __shared__ float2 Bh[KS * NB * 32], Bl[KS * NB * 32];     // [k8 step][n block][lane]
    __shared__ float s_part[2 * NP];
    __shared__ float s_ps[KP], s_pt[KP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    for (int i = tid; i < KS * NB * 32; i += kThreads) {
        const int s = i / (NB * 32), nb = (i / 32) % NB, gg = (i & 31) >> 2, tt = i & 3;
        const int k0 = 8 * s + tt, k1 = k0 + 4, n = cl::phys_col(nb, gg);
        const float w0 = (k0 < a.K && n < a.N) ? __ldg(a.B + (int64_t)n * a.sbn + (int64_t)k0 * a.sbk) : 0.f;
        const float w1 = (k1 < a.K && n < a.N) ? __ldg(a.B + (int64_t)n * a.sbn + (int64_t)k1 * a.sbk) : 0.f;
        cl::store_split(Bh, Bl, i, w0, w1);
    }
    for (int i = tid; i < 2 * NP; i += kThreads) s_part[i] = 0.f;
    for (int i = tid; i < KP; i += kThreads) {
        s_ps[i] = (a.ps && i < a.K) ? __ldg(a.ps + i) : 1.f;
        s_pt[i] = (a.ps && i < a.K) ? __ldg(a.pt + i) : 0.f;
    }
    __syncthreads();
    const bool pro = a.ps != nullptr;
    float4 ssum[NQ], ssq[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) { ssum[q] = zero4(); ssq[q] = zero4(); }
    const int64_t ntiles = (a.M + 15) >> 4;
    const int64_t stride = (int64_t)gridDim.x * kWarps;
    auto load = [&](int64_t tl, float (&v)[KS][4]) {
        const int64_t r0 = tl * 16 + g, r1 = r0 + 8;
        const bool k0 = r0 < a.M, k1 = r1 < a.M;
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            const int ca = 8 * s + t, cb = ca + 4;
            v[s][0] = (k0 && ca < a.K) ? __ldg(a.A + r0 * a.lda + ca) : 0.f;
            v[s][1] = (k1 && ca < a.K) ? __ldg(a.A + r1 * a.lda + ca) : 0.f;
            v[s][2] = (k0 && cb < a.K) ? __ldg(a.A + r0 * a.lda + cb) : 0.f;
            v[s][3] = (k1 && cb < a.K) ? __ldg(a.A + r1 * a.lda + cb) : 0.f;
        }
    };
    float cur[KS][4];
    int64_t tile = (int64_t)blockIdx.x * kWarps + warp;
    load(tile, cur);
    for (; tile < ntiles; tile += stride) {
        const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.M, ok1 = r1 < a.M;
        float nxt[KS][4];
        load(tile + stride, nxt);                              // rows beyond M come back as zeros
        cl::FragA f[KS];
#pragma unroll
        for (int s = 0; s < KS; ++s) {
            float v0 = cur[s][0], v1 = cur[s][1], v2 = cur[s][2], v3 = cur[s][3];
            if (pro) {
                const int ca = 8 * s + t, cb = ca + 4;
                v0 = (ok0 && ca < a.K) ? cl::lrelu(fmaf(v0, s_ps[ca], s_pt[ca]), a.pslope) : 0.f;
                v1 = (ok1 && ca < a.K) ? cl::lrelu(fmaf(v1, s_ps[ca], s_pt[ca]), a.pslope) : 0.f;
                v2 = (ok0 && cb < a.K) ? cl::lrelu(fmaf(v2, s_ps[cb], s_pt[cb]), a.pslope) : 0.f;
                v3 = (ok1 && cb < a.K) ? cl::lrelu(fmaf(v3, s_ps[cb], s_pt[cb]), a.pslope) : 0.f;
            }
            cl::make_a(f[s], v0, v1, v2, v3);
        }
        float* p0 = a.Y + r0 * a.N + 4 * t;
        float* p1 = a.Y + r1 * a.N + 4 * t;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int nb = 2 * q + e;
#pragma unroll
                for (int s = 0; s < KS; ++s) cl::mma3(acc[e], f[s], Bh[(s * NB + nb) * 32 + lane], Bl[(s * NB + nb) * 32 + lane]);
            }
            float4 o0 = make_float4(acc[0][0], acc[0][1], acc[1][0], acc[1][1]);
            float4 o1 = make_float4(acc[0][2], acc[0][3], acc[1][2], acc[1][3]);
            const int c = 16 * q + 4 * t;
            if (a.bias && c < a.N) {
                const float4 b = cl::ldg4(a.bias + c);
                o0 = add4(o0, b); o1 = add4(o1, b);
            }
            if (c < a.N) {                                     // N % 4 == 0
                if (ok0) *reinterpret_cast<float4*>(p0 + 16 * q) = o0;
                if (ok1) *reinterpret_cast<float4*>(p1 + 16 * q) = o1;
            }
            if (a.stats) {
                if (!ok0) o0 = zero4();
                if (!ok1) o1 = zero4();
                ssum[q] = add4(ssum[q], add4(o0, o1));
                ssq[q] = fma4(o0, o0, fma4(o1, o1, ssq[q]));
            }
        }
#pragma unroll
        for (int s = 0; s < KS; ++s)
#pragma unroll
            for (int e = 0; e < 4; ++e) cur[s][e] = nxt[s][e];
    }
    if (!a.stats) return;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const float v1[4] = {ssum[q].x, ssum[q].y, ssum[q].z, ssum[q].w}, v2[4] = {ssq[q].x, ssq[q].y, ssq[q].z, ssq[q].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float x1 = group8_sum(v1[e]), x2 = group8_sum(v2[e]);
            if (g == 0) { atomicAdd(&s_part[16 * q + 4 * t + e], x1); atomicAdd(&s_part[NP + 16 * q + 4 * t + e], x2); }
        }
    }
    __syncthreads();
    float* st = a.stats + (size_t)(blockIdx.x % kStatSlots) * 2 * a.N;
    for (int i = tid; i < NP; i += kThreads)
        if (i < a.N) { atomicAdd(st + i, s_part[i]); atomicAdd(st + a.N + i, s_part[NP + i]); }
}

template <int KP, int NP>
inline int run(const UpArgs& a, cudaStream_t st) {
    const int64_t tiles = ceil_div(a.M, (int64_t)16);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(tiles, (int64_t)kWarps), (int64_t)kNumSMs * (NP > 64 ? 1 : 2)));
    return launch(upproj_kernel<KP, NP>, dim3(grid), dim3(kThreads), 0, st, a);
}

inline int dispatch(const UpArgs& a, cudaStream_t st) {
    const int kp = a.K <= 8 ? 8 : (a.K <= 16 ? 16 : 32);
    const int np = a.N <= 32 ? 32 : (a.N <= 64 ? 64 : 128);
#define CRF_UP(k, n) \
    if (kp == k && np == n) return run<k, n>(a, st);
    CRF_UP(8, 32) CRF_UP(8, 64) CRF_UP(8, 128) CRF_UP(16, 32) CRF_UP(16, 64) CRF_UP(16, 128) CRF_UP(32, 64) CRF_UP(32, 128)
#undef CRF_UP
    return kDeclined;
}

}  // namespace up

// forward: wide output, narrow plain input
int try_upproj_fwd(const FwdArgs& a, cudaStream_t st) {
    if (a.idx1 || a.C2 != 0 || a.C1 < 1 || a.C1 > 32 || a.Cout < 32 || a.Cout > 128 || (a.Cout & 3) || a.M < 8192) return kDeclined;
    if (a.Cout <= 2 * a.C1) return kDeclined;                  // only when the output dominates the traffic
    if (!aligned16(a.Y) || (a.bias && !aligned16(a.bias))) return kDeclined;
    up::UpArgs u{a.X1, a.C1, a.C1, a.scale1, a.shift1, a.slope1, a.W, a.C1, 1, a.bias, a.Y, a.Cout, a.stats, a.M};
    return up::dispatch(u, st);
}

// input gradient of a plain Linear with few outputs: dX[M, Ktot] = dY[M, Cout]·W[Cout, Ktot]   (the 13-class head)
int try_upproj_dgrad(const DgradArgs& a, cudaStream_t st) {
    const int Ktot = a.C1 + a.C2;
    if (a.bn.scale || a.C2 != 0 || !a.dX1 || a.acc1 || a.Cout < 1 || a.Cout > 32 || Ktot < 32 || Ktot > 128 || (Ktot & 3) || a.M < 8192) return kDeclined;
    if (Ktot <= 2 * a.Cout) return kDeclined;
    if (!aligned16(a.dX1)) return kDeclined;
    up::UpArgs u{a.dY, a.Cout, a.Cout, nullptr, nullptr, 1.f, a.W, 1, Ktot, nullptr, a.dX1, Ktot, nullptr, a.M};
    return up::dispatch(u, st);
}

}  // namespace lin
}  // namespace crf
