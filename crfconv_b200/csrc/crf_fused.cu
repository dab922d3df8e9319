// Layer-specialised kernels of the dense ContinuousGaussianCRFConv (reference: models/continuous_crf_conv_big.py:7-78) for the
// hidden width the hot path uses (F = out_channels / 4 = 16).  The generic Linear kernels treat every MLP of the layer as an
// independent GEMM + three bookkeeping launches; here each BatchNorm boundary of the layer is ONE streaming pass:
//
//   forward   lin16_fwd<CIN>      X[M,CIN] → H[M,16] = act(X)·Wᵀ, Σ/Σ² of H, BatchNorm finalize by the last CTA
//                                 (CIN = 64/128: unary_nn[0] / pairwise_nn[0] (:20-27);  CIN = 16 with the previous layer's
//                                 BN + LeakyReLU applied on the fly: unary_nn[1] / pairwise_nn[1])
//   backward  out_bwd             dO[M,64], H3[M,64], x[M,16] → t = W3ᵀ·diag(γ·istd)·dv3, Σdv3, Σdv3·Ĥ3, Σdv3ᵀx, Σx, Σxxᵀ; the last
//                                 CTA turns them into k1/k2, dγ/dβ, dW3 and the 16×16 matrix Q / vector a0 with which the
//                                 BatchNorm-backward of out_nn (:74) collapses to  g_i = t_i − a0 − Q·x_i  (applied in the
//                                 mean-field backward's prologue): out_nn's backward is one pass over dO instead of three.
//             step_bwd            mean-field backward (:68-72, SURVEY Appendix B) with GC = Σ mᵀh, GM = Σ vᵀg accumulated on the
//                                 tensor cores inside the kernel (no m/v/h tensors, no extra GEMM launches) and the BatchNorm
//                                 backward sums of pairwise_nn[1] emitted per edge (Σ_rows Gy = 0, Σ_rows Gy·Ĥ = −istd·Σ_e 2Ga·df·dfH).
//             upsample_bwd        Gu[up(i)] += Gz_i + g0_i plus the BN-backward sums of unary_nn[1] (Σ v_i, Σ v_i·Ĥ[up(i)]).
//             mid16_bwd           16→16 layer: dH2 on the fly, dV1 = (dH2·W2)⊙lrelu'(·), dW2, and the NEXT BatchNorm's
//                                 backward sums (Σ dV1, Σ dV1·Ĥ1) in the same pass.
//             in16_dgrad/wgrad    first layers: dX (+)= dH1·W1 and dW1 = dH1ᵀ·X.
//
// All contractions are warp-level mma.sync m16n8k8 3xTF32 (fp32-grade, these GEMMs have K or N = 16 and are HBM-bound by a wide
// margin); activations go from global memory straight into MMA fragments: a thread's float4 of 4 consecutive channels feeds two
// k-steps through a channel permutation that is folded into the (shared-memory resident, pre-split) weight fragments, so there
// is no shared-memory staging, no shuffle and no bank conflict on the activation path.  Contractions over ROWS (weight
// gradients) read their operands a second time with 4-byte "transposed" loads (8 lanes = one 32-byte sector, L1 hits).
#include <algorithm>
#include <type_traits>

#include "../../include/crfconv_b200.h"
#include "common.cuh"
#include "fused_common.cuh"

namespace crf {
namespace cl {

constexpr int kThreads = 256, kWarps = 8;
constexpr int kFinSlots = 16;             // statistics slots used by kernels that finalize in their own tail (<= kStatSlots; the rest stay zero)
constexpr int kGradSlotsF = kGradSlots;   // weight-gradient partial slots shared with the generic kernels (folded by grad_slots_reduce)

__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 sub4(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 fma4(float4 a, float4 b, float4 c) {
    return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
}
__device__ __forceinline__ float4 lrelu4(float4 v, float s) { return make_float4(lrelu(v.x, s), lrelu(v.y, s), lrelu(v.z, s), lrelu(v.w, s)); }
// dv = pre > 0 ? d : d·slope   (LeakyReLU backward selected by the pre-activation)
__device__ __forceinline__ float4 mask4(float4 d, float4 pre, float s) {
    return make_float4(pre.x > 0.f ? d.x : d.x * s, pre.y > 0.f ? d.y : d.y * s, pre.z > 0.f ? d.z : d.z * s, pre.w > 0.f ? d.w : d.w * s);
}
__device__ __forceinline__ float group8_sum(float v) {          // sum over the 8 lanes that share lane & 3
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return v;
}

// BatchNorm-backward constants of one layer for the on-the-fly transform  dH = sc·(dV − k1 − (H − mu)·c2),  c2 = istd·k2
struct BnB {
    const float* sc; const float* mu; const float* is; const float* k1; const float* k2;
};

// =========================================================================================== forward: X[M,CIN] → H[M,16]
struct LinFwdArgs {
    const float* X;                                           // [M, CIN]
    const float* W;                                           // [16, CIN]
    const float* pscale; const float* pshift; float pslope;   // PRO: X ← lrelu(X·pscale + pshift)
    float* Y;                                                 // [M, 16]
    int64_t M;
    FwdFin fin;
};

template <int CIN, bool PRO>
__global__ void __launch_bounds__(kThreads, CIN > 64 ? 1 : 2) lin16_fwd_kernel(const LinFwdArgs a) {
    constexpr int NS = CIN / 8, NJ = CIN / 16;
    __shared__ float2 Bh[NS * 2 * 32], Bl[NS * 2 * 32];        // [k8 step][n block][lane]
    __shared__ __align__(16) float s_sc[CIN], s_sh[CIN];
    __shared__ float s_part[kWarps][32];
    __shared__ double s_red[kThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    // k-step s = 2j + h covers the physical columns {16j + 4t' + 2h, +1 : t' = 0..3}: fragment index k = t' ↔ column 16j+4t'+2h,
    // k = t'+4 ↔ the next column — exactly the (x,y) / (z,w) halves of the float4 a thread loads.
    for (int i = tid; i < NS * 2 * 32; i += kThreads) {
        const int s = i >> 6, nb = (i >> 5) & 1, gg = (i & 31) >> 2, tt = i & 3;
        const int col = 16 * (s >> 1) + 4 * tt + 2 * (s & 1), n = nb * 8 + gg;
        store_split(Bh, Bl, i, __ldg(a.W + n * CIN + col), __ldg(a.W + n * CIN + col + 1));
    }
    if (PRO) {
        for (int i = tid; i < CIN; i += kThreads) { s_sc[i] = a.pscale[i]; s_sh[i] = a.pshift[i]; }
    }
    __syncthreads();

    const int64_t ntiles = (a.M + 15) >> 4;
    const int64_t stride = (int64_t)gridDim.x * kWarps;
    float ssum[2][2] = {{0.f, 0.f}, {0.f, 0.f}}, ssq[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    float4 c0[NJ], c1[NJ];
    auto load = [&](int64_t tl, float4 (&v0)[NJ], float4 (&v1)[NJ]) {
        const int64_t r0 = tl * 16 + g, r1 = r0 + 8;
        const bool k0 = r0 < a.M, k1 = r1 < a.M;               // tl >= ntiles ⇒ both false
        const float* p0 = a.X + r0 * CIN + 4 * t;
        const float* p1 = a.X + r1 * CIN + 4 * t;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            v0[j] = k0 ? ldg4(p0 + 16 * j) : zero4();
            v1[j] = k1 ? ldg4(p1 + 16 * j) : zero4();
        }
    };
    int64_t tile = (int64_t)blockIdx.x * kWarps + warp;
    load(tile, c0, c1);
    for (; tile < ntiles; tile += stride) {
        float4 n0[NJ], n1[NJ];
        load(tile + stride, n0, n1);                           // next tile's loads fly while this one is contracted
        const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.M, ok1 = r1 < a.M;
        float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            float4 x0 = c0[j], x1 = c1[j];
            if (PRO) {
                const float4 sc = *reinterpret_cast<const float4*>(s_sc + 16 * j + 4 * t);
                const float4 sh = *reinterpret_cast<const float4*>(s_sh + 16 * j + 4 * t);
                x0 = ok0 ? lrelu4(fma4(x0, sc, sh), a.pslope) : zero4();
                x1 = ok1 ? lrelu4(fma4(x1, sc, sh), a.pslope) : zero4();
            }
            FragA f;
            make_a(f, x0.x, x1.x, x0.y, x1.y);
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) mma3(acc[nb], f, Bh[((2 * j) * 2 + nb) * 32 + lane], Bl[((2 * j) * 2 + nb) * 32 + lane]);
            make_a(f, x0.z, x1.z, x0.w, x1.w);
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) mma3(acc[nb], f, Bh[((2 * j + 1) * 2 + nb) * 32 + lane], Bl[((2 * j + 1) * 2 + nb) * 32 + lane]);
        }
#pragma unroll
        for (int nb = 0; nb < 2; ++nb) {
            if (ok0) *reinterpret_cast<float2*>(a.Y + r0 * 16 + nb * 8 + 2 * t) = make_float2(acc[nb][0], acc[nb][1]);
            if (ok1) *reinterpret_cast<float2*>(a.Y + r1 * 16 + nb * 8 + 2 * t) = make_float2(acc[nb][2], acc[nb][3]);
            ssum[nb][0] += acc[nb][0] + acc[nb][2];            // rows beyond M are exact zeros
            ssum[nb][1] += acc[nb][1] + acc[nb][3];
            ssq[nb][0] = fmaf(acc[nb][0], acc[nb][0], fmaf(acc[nb][2], acc[nb][2], ssq[nb][0]));
            ssq[nb][1] = fmaf(acc[nb][1], acc[nb][1], fmaf(acc[nb][3], acc[nb][3], ssq[nb][1]));
        }
#pragma unroll
        for (int j = 0; j < NJ; ++j) { c0[j] = n0[j]; c1[j] = n1[j]; }
    }
    // per-CTA Σ / Σ² in a fixed order (lanes → warps), one plain store per column: reproducible statistics
#pragma unroll
    for (int nb = 0; nb < 2; ++nb)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const float s = group8_sum(ssum[nb][e]), q = group8_sum(ssq[nb][e]);
            if (g == 0) { s_part[warp][nb * 8 + 2 * t + e] = s; s_part[warp][16 + nb * 8 + 2 * t + e] = q; }
        }
    __syncthreads();
    if (tid < 32) {
        float tot = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) tot += s_part[w][tid];
        a.fin.part[(size_t)blockIdx.x * 32 + tid] = tot;
    }
    if (grid_reduce_rows<32, kThreads>(a.fin.part, part_group_rows(a.fin.part), a.fin.counter, s_red) && tid < 16)
        bn_fwd_finalize(a.fin, s_red[tid], s_red[16 + tid], tid);
}

// =========================================================================================== forward: X[M,16] → H[M,COUT]
// out_nn's Linear (16 → 64, continuous_crf_conv_big.py:28,74): K = 16, so the pass is a pure stream of the 64-wide output.  Same
// fragment scheme as in16_dgrad (output columns permuted so that a thread owns 4 consecutive ones ⇒ 128-bit stores); Σ/Σ² go to
// kStatSlots zeroed slots with one atomic per CTA and column, and the last CTA finalizes the BatchNorm.
struct Up16FwdArgs {
    const float* X;                                           // [M, 16]
    const float* W;                                           // [COUT, 16]
    float* Y;                                                 // [M, COUT]
    int64_t M;
    FwdFin fin;                                               // fin.part = statistics slots [kStatSlots][2·COUT], zeroed
};

template <int COUT>
__global__ void __launch_bounds__(kThreads, 2) up16_fwd_kernel(const Up16FwdArgs a) {
    constexpr int NB = COUT / 8, NQ = COUT / 16;
    __shared__ float2 Bh[2 * NB * 32], Bl[2 * NB * 32];        // [k8 step][n block][lane]
    __shared__ float s_part[2 * COUT];
    __shared__ double s_red[kThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    for (int i = tid; i < 2 * NB * 32; i += kThreads) {
        const int s = i / (NB * 32), nb = (i / 32) % NB, gg = (i & 31) >> 2, tt = i & 3;
        const int in = 4 * tt + 2 * s, out = phys_col(nb, gg);
        store_split(Bh, Bl, i, __ldg(a.W + out * 16 + in), __ldg(a.W + out * 16 + in + 1));
    }
    for (int i = tid; i < 2 * COUT; i += kThreads) s_part[i] = 0.f;
    __syncthreads();
    float4 ssum[NQ], ssq[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) { ssum[q] = zero4(); ssq[q] = zero4(); }
    const int64_t ntiles = (a.M + 15) >> 4;
    const int64_t stride = (int64_t)gridDim.x * kWarps;
    int64_t tile = (int64_t)blockIdx.x * kWarps + warp;
    auto load = [&](int64_t tl, float4& v0, float4& v1) {
        const int64_t r0 = tl * 16 + g, r1 = r0 + 8;
        v0 = r0 < a.M ? ldg4(a.X + r0 * 16 + 4 * t) : zero4();
        v1 = r1 < a.M ? ldg4(a.X + r1 * 16 + 4 * t) : zero4();
    };
    float4 c0, c1;
    load(tile, c0, c1);
    for (; tile < ntiles; tile += stride) {
        const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.M, ok1 = r1 < a.M;
        float4 n0, n1;
        load(tile + stride, n0, n1);
        FragA f0, f1;
        make_a(f0, c0.x, c1.x, c0.y, c1.y);
        make_a(f1, c0.z, c1.z, c0.w, c1.w);
        float* p0 = a.Y + r0 * COUT + 4 * t;
        float* p1 = a.Y + r1 * COUT + 4 * t;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int nb = 2 * q + e;
                mma3(acc[e], f0, Bh[(0 * NB + nb) * 32 + lane], Bl[(0 * NB + nb) * 32 + lane]);
                mma3(acc[e], f1, Bh[(1 * NB + nb) * 32 + lane], Bl[(1 * NB + nb) * 32 + lane]);
            }
            const float4 o0 = make_float4(acc[0][0], acc[0][1], acc[1][0], acc[1][1]);
            const float4 o1 = make_float4(acc[0][2], acc[0][3], acc[1][2], acc[1][3]);
            if (ok0) *reinterpret_cast<float4*>(p0 + 16 * q) = o0;
            if (ok1) *reinterpret_cast<float4*>(p1 + 16 * q) = o1;
            ssum[q] = add4(ssum[q], add4(o0, o1));             // rows beyond M are exact zeros
            ssq[q] = fma4(o0, o0, fma4(o1, o1, ssq[q]));
        }
        c0 = n0; c1 = n1;
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        const float v1[4] = {ssum[q].x, ssum[q].y, ssum[q].z, ssum[q].w}, v2[4] = {ssq[q].x, ssq[q].y, ssq[q].z, ssq[q].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float x1 = group8_sum(v1[e]), x2 = group8_sum(v2[e]);
            if (g == 0) { atomicAdd(&s_part[16 * q + 4 * t + e], x1); atomicAdd(&s_part[COUT + 16 * q + 4 * t + e], x2); }
        }
    }
    __syncthreads();
    if (tid < 2 * COUT) atomicAdd(a.fin.part + (size_t)(blockIdx.x % kFinSlots) * 2 * COUT + tid, s_part[tid]);
    fwd_fin_tail<COUT, kThreads>(a.fin, kFinSlots, s_red);
}

// =========================================================================================== backward of a 16→16 layer
// Layer 2 of unary_nn / pairwise_nn:  y = BN2(H2), H2 = A1·W2ᵀ, A1 = lrelu(BN1(H1)).  Given dY = dL/dy:
//   dH2 = sc2·(dY − k1 − (H2−mu2)·c2)            (BN2 backward, k1/k2 finalized by the kernel that produced dY)
//   dV1 = (dH2·W2) ⊙ lrelu'(BN1(H1))  → written;  Σ dV1, Σ dV1·Ĥ1 → BN1 backward constants (last CTA)
//   dW2 += dH2ᵀ·A1
struct Mid16BwdArgs {
    const float* dY; const float* H2; BnB b2;
    const float* H1; const float* sc1; const float* sh1; const float* mu1; const float* is1; float slope1;
    const float* W2;                                          // [16 out, 16 in]
    float* dV1;                                               // [M, 16]
    float* dW2; int64_t slot_stride;                          // partial slots: dW2 + slot·slot_stride
    int64_t M;
    BwdFin fin;
};

__global__ void __launch_bounds__(kThreads, 2) mid16_bwd_kernel(const Mid16BwdArgs a) {
    __shared__ float2 Bh[2 * 2 * 32], Bl[2 * 2 * 32];
    __shared__ float s_part[kWarps][32];
    __shared__ float s_w[256];
    __shared__ double s_red[kThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    // dgrad: contraction over the OUTPUT channel o of layer 2 (k-step s: k = t' ↔ o = 4t'+2s, k = t'+4 ↔ o = 4t'+2s+1), result
    // column n of block nb ↔ input channel phys_col(nb, n) ⇒ a thread ends up with input channels 4t..4t+3 of rows g, g+8.
    for (int i = tid; i < 2 * 2 * 32; i += kThreads) {
        const int s = i >> 6, nb = (i >> 5) & 1, gg = (i & 31) >> 2, tt = i & 3;
        const int o = 4 * tt + 2 * s, in = phys_col(nb, gg);
        store_split(Bh, Bl, i, __ldg(a.W2 + o * 16 + in), __ldg(a.W2 + (o + 1) * 16 + in));
    }
    s_w[tid] = 0.f;
    __syncthreads();
    // row-major constants (channels 4t..4t+3)
    const float4 sc2 = ldg4(a.b2.sc + 4 * t), mu2 = ldg4(a.b2.mu + 4 * t), k12 = ldg4(a.b2.k1 + 4 * t);
    const float4 c22 = mul4(ldg4(a.b2.is + 4 * t), ldg4(a.b2.k2 + 4 * t));
    const float4 sc1 = ldg4(a.sc1 + 4 * t), sh1 = ldg4(a.sh1 + 4 * t), mu1 = ldg4(a.mu1 + 4 * t), is1 = ldg4(a.is1 + 4 * t);
    // transposed constants (channels g and g+8)
    float tsc2[2], tmu2[2], tk1[2], tc2[2], tsc1[2], tsh1[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int c = g + 8 * e;
        tsc2[e] = __ldg(a.b2.sc + c); tmu2[e] = __ldg(a.b2.mu + c); tk1[e] = __ldg(a.b2.k1 + c);
        tc2[e] = __ldg(a.b2.is + c) * __ldg(a.b2.k2 + c);
        tsc1[e] = __ldg(a.sc1 + c); tsh1[e] = __ldg(a.sh1 + c);
    }
    auto dh4 = [&](float4 dy, float4 h) {                     // sc·(dy − k1 − (h − mu)·c2)
        return make_float4(sc2.x * (dy.x - k12.x - (h.x - mu2.x) * c22.x), sc2.y * (dy.y - k12.y - (h.y - mu2.y) * c22.y),
                           sc2.z * (dy.z - k12.z - (h.z - mu2.z) * c22.z), sc2.w * (dy.w - k12.w - (h.w - mu2.w) * c22.w));
    };
    float accW[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    float4 s1 = zero4(), s2 = zero4();
    const int64_t ntiles = (a.M + 15) >> 4;
    for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < ntiles; tile += (int64_t)gridDim.x * kWarps) {
        const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.M, ok1 = r1 < a.M;
        // ---- all loads of the tile first
        const float4 dy0 = ok0 ? ldg4(a.dY + r0 * 16 + 4 * t) : zero4(), dy1 = ok1 ? ldg4(a.dY + r1 * 16 + 4 * t) : zero4();
        const float4 h20 = ok0 ? ldg4(a.H2 + r0 * 16 + 4 * t) : zero4(), h21 = ok1 ? ldg4(a.H2 + r1 * 16 + 4 * t) : zero4();
        const float4 h10 = ok0 ? ldg4(a.H1 + r0 * 16 + 4 * t) : zero4(), h11 = ok1 ? ldg4(a.H1 + r1 * 16 + 4 * t) : zero4();
        float tdy[2][4], th2[2][4], th1[2][4];                 // [k8 step][ (ra,g) (ra,g+8) (rb,g) (rb,g+8) ]
        bool tok[2][2];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const int64_t ra = tile * 16 + 8 * ks + t, rb = ra + 4;
            tok[ks][0] = ra < a.M; tok[ks][1] = rb < a.M;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int64_t r = (q & 2) ? rb : ra;
                const bool ok = (q & 2) ? tok[ks][1] : tok[ks][0];
                const int64_t off = r * 16 + g + 8 * (q & 1);
                tdy[ks][q] = ok ? __ldg(a.dY + off) : 0.f;
                th2[ks][q] = ok ? __ldg(a.H2 + off) : 0.f;
                th1[ks][q] = ok ? __ldg(a.H1 + off) : 0.f;
            }
        }
        // ---- dgrad + activation backward + next BatchNorm's sums
        float4 dh0 = dh4(dy0, h20), dh1 = dh4(dy1, h21);
        if (!ok0) dh0 = zero4();
        if (!ok1) dh1 = zero4();
        float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
        FragA f;
        make_a(f, dh0.x, dh1.x, dh0.y, dh1.y);
#pragma unroll
        for (int nb = 0; nb < 2; ++nb) mma3(acc[nb], f, Bh[(0 * 2 + nb) * 32 + lane], Bl[(0 * 2 + nb) * 32 + lane]);
        make_a(f, dh0.z, dh1.z, dh0.w, dh1.w);
#pragma unroll
        for (int nb = 0; nb < 2; ++nb) mma3(acc[nb], f, Bh[(1 * 2 + nb) * 32 + lane], Bl[(1 * 2 + nb) * 32 + lane]);
        const float4 da0 = make_float4(acc[0][0], acc[0][1], acc[1][0], acc[1][1]);
        const float4 da1 = make_float4(acc[0][2], acc[0][3], acc[1][2], acc[1][3]);
        const float4 dv0 = mask4(da0, fma4(h10, sc1, sh1), a.slope1), dv1 = mask4(da1, fma4(h11, sc1, sh1), a.slope1);
        if (ok0) *reinterpret_cast<float4*>(a.dV1 + r0 * 16 + 4 * t) = dv0;
        if (ok1) *reinterpret_cast<float4*>(a.dV1 + r1 * 16 + 4 * t) = dv1;
        s1 = add4(s1, add4(dv0, dv1));                         // rows beyond M: dh = 0 ⇒ dv = 0
        s2 = fma4(dv0, mul4(sub4(h10, mu1), is1), s2);
        s2 = fma4(dv1, mul4(sub4(h11, mu1), is1), s2);
        // ---- wgrad: dW2[o][i] += Σ_rows dH2[row][o]·A1[row][i]   (m = o, n = i, k = rows)
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            float av[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = q & 1;
                const bool ok = (q & 2) ? tok[ks][1] : tok[ks][0];
                av[q] = ok ? tsc2[e] * (tdy[ks][q] - tk1[e] - (th2[ks][q] - tmu2[e]) * tc2[e]) : 0.f;
            }
            make_a(f, av[0], av[1], av[2], av[3]);
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) {                  // B: b0 = A1[ra][nb*8+g], b1 = A1[rb][nb*8+g]
                FragB b;
                make_b(b, lrelu(fmaf(th1[ks][nb], tsc1[nb], tsh1[nb]), a.slope1), lrelu(fmaf(th1[ks][2 + nb], tsc1[nb], tsh1[nb]), a.slope1));
                mma3(accW[nb], f, b);
            }
        }
    }
    // ---- CTA reductions
#pragma unroll
    for (int nb = 0; nb < 2; ++nb) {
        atomicAdd(&s_w[g * 16 + nb * 8 + 2 * t], accW[nb][0]);
        atomicAdd(&s_w[g * 16 + nb * 8 + 2 * t + 1], accW[nb][1]);
        atomicAdd(&s_w[(g + 8) * 16 + nb * 8 + 2 * t], accW[nb][2]);
        atomicAdd(&s_w[(g + 8) * 16 + nb * 8 + 2 * t + 1], accW[nb][3]);
    }
    {
        const float v1[4] = {s1.x, s1.y, s1.z, s1.w}, v2[4] = {s2.x, s2.y, s2.z, s2.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float x1 = group8_sum(v1[e]), x2 = group8_sum(v2[e]);
            if (g == 0) { s_part[warp][4 * t + e] = x1; s_part[warp][16 + 4 * t + e] = x2; }
        }
    }
    __syncthreads();
    atomicAdd(a.dW2 + a.slot_stride * (int64_t)(blockIdx.x % kGradSlotsF) + tid, s_w[tid]);
    if (tid < 32) {
        float tot = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) tot += s_part[w][tid];
        a.fin.part[(size_t)blockIdx.x * 32 + tid] = tot;
    }
    if (grid_reduce_rows<32, kThreads>(a.fin.part, part_group_rows(a.fin.part), a.fin.counter, s_red) && tid < 16)
        bn_bwd_finalize(a.fin, s_red[tid], s_red[16 + tid], tid);
}

// =========================================================================================== first layers: dX (+)= dH1·W1
struct In16DgradArgs {
    const float* dV1; const float* H1; BnB b1;
    const float* W1;                                          // [16, CIN]
    float* dX;                                                // [M, CIN]
    int64_t M;
};

template <int CIN, bool ACC>
__global__ void __launch_bounds__(kThreads, CIN > 64 ? 1 : 2) in16_dgrad_kernel(const In16DgradArgs a) {
    constexpr int NB = CIN / 8, NQ = CIN / 16;
    __shared__ float2 Bh[2 * NB * 32], Bl[2 * NB * 32];        // [k8 step][n block][lane]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    for (int i = tid; i < 2 * NB * 32; i += kThreads) {
        const int s = i / (NB * 32), nb = (i / 32) % NB, gg = (i & 31) >> 2, tt = i & 3;
        const int o = 4 * tt + 2 * s, in = phys_col(nb, gg);
        store_split(Bh, Bl, i, __ldg(a.W1 + o * CIN + in), __ldg(a.W1 + (o + 1) * CIN + in));
    }
    __syncthreads();
    const float4 sc = ldg4(a.b1.sc + 4 * t), mu = ldg4(a.b1.mu + 4 * t), k1 = ldg4(a.b1.k1 + 4 * t);
    const float4 c2 = mul4(ldg4(a.b1.is + 4 * t), ldg4(a.b1.k2 + 4 * t));
    auto dh4 = [&](float4 dv, float4 h) {
        return make_float4(sc.x * (dv.x - k1.x - (h.x - mu.x) * c2.x), sc.y * (dv.y - k1.y - (h.y - mu.y) * c2.y),
                           sc.z * (dv.z - k1.z - (h.z - mu.z) * c2.z), sc.w * (dv.w - k1.w - (h.w - mu.w) * c2.w));
    };
    const int64_t ntiles = (a.M + 15) >> 4;
    const int64_t stride = (int64_t)gridDim.x * kWarps;
    int64_t tile = (int64_t)blockIdx.x * kWarps + warp;
    float4 cv0, cv1, ch0, ch1;
    auto load = [&](int64_t tl, float4& v0, float4& v1, float4& h0, float4& h1) {
        const int64_t r0 = tl * 16 + g, r1 = r0 + 8;
        const bool k0 = r0 < a.M, k1_ = r1 < a.M;
        v0 = k0 ? ldg4(a.dV1 + r0 * 16 + 4 * t) : zero4(); h0 = k0 ? ldg4(a.H1 + r0 * 16 + 4 * t) : zero4();
        v1 = k1_ ? ldg4(a.dV1 + r1 * 16 + 4 * t) : zero4(); h1 = k1_ ? ldg4(a.H1 + r1 * 16 + 4 * t) : zero4();
    };
    load(tile, cv0, cv1, ch0, ch1);
    for (; tile < ntiles; tile += stride) {
        const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.M, ok1 = r1 < a.M;
        float* p0 = a.dX + r0 * CIN + 4 * t;
        float* p1 = a.dX + r1 * CIN + 4 * t;
        float4 old0[ACC ? NQ : 1], old1[ACC ? NQ : 1];
        if (ACC) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                old0[q] = ok0 ? *reinterpret_cast<const float4*>(p0 + 16 * q) : zero4();
                old1[q] = ok1 ? *reinterpret_cast<const float4*>(p1 + 16 * q) : zero4();
            }
        }
        float4 nv0, nv1, nh0, nh1;
        load(tile + stride, nv0, nv1, nh0, nh1);
        const float4 dh0 = dh4(cv0, ch0), dh1 = dh4(cv1, ch1);   // rows beyond M are never stored
        FragA f0, f1;
        make_a(f0, dh0.x, dh1.x, dh0.y, dh1.y);
        make_a(f1, dh0.z, dh1.z, dh0.w, dh1.w);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int nb = 2 * q + e;
                mma3(acc[e], f0, Bh[(0 * NB + nb) * 32 + lane], Bl[(0 * NB + nb) * 32 + lane]);
                mma3(acc[e], f1, Bh[(1 * NB + nb) * 32 + lane], Bl[(1 * NB + nb) * 32 + lane]);
            }
            float4 o0 = make_float4(acc[0][0], acc[0][1], acc[1][0], acc[1][1]);
            float4 o1 = make_float4(acc[0][2], acc[0][3], acc[1][2], acc[1][3]);
            if (ACC) { o0 = add4(o0, old0[q]); o1 = add4(o1, old1[q]); }
            if (ok0) *reinterpret_cast<float4*>(p0 + 16 * q) = o0;
            if (ok1) *reinterpret_cast<float4*>(p1 + 16 * q) = o1;
        }
        cv0 = nv0; cv1 = nv1; ch0 = nh0; ch1 = nh1;
    }
}

// =========================================================================================== first layers: dW1 += dH1ᵀ·X
struct In16WgradArgs {
    const float* dV1; const float* H1; BnB b1;
    const float* X;                                           // [M, CIN]
    float* dW; int64_t slot_stride;                           // [16, CIN] partial slots
    int64_t M;
};

template <int CIN>
__global__ void __launch_bounds__(kThreads, CIN > 64 ? 1 : 2) in16_wgrad_kernel(const In16WgradArgs a) {
    constexpr int NB = CIN / 8;
    __shared__ float s_w[16 * CIN];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    for (int i = tid; i < 16 * CIN; i += kThreads) s_w[i] = 0.f;
    __syncthreads();
    float tsc[2], tmu[2], tk1[2], tc2[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int c = g + 8 * e;
        tsc[e] = __ldg(a.b1.sc + c); tmu[e] = __ldg(a.b1.mu + c); tk1[e] = __ldg(a.b1.k1 + c);
        tc2[e] = __ldg(a.b1.is + c) * __ldg(a.b1.k2 + c);
    }
    float accW[NB][4];
#pragma unroll
    for (int nb = 0; nb < NB; ++nb)
#pragma unroll
        for (int e = 0; e < 4; ++e) accW[nb][e] = 0.f;
    const int64_t ntiles = (a.M + 15) >> 4;                    // 16-row tiles = two 8-row k-steps whose loads are all issued first
    for (int64_t tile = (int64_t)blockIdx.x * kWarps + warp; tile < ntiles; tile += (int64_t)gridDim.x * kWarps) {
        float tv[2][4], th[2][4], xa[2][NB], xb[2][NB];
        bool oka[2], okb[2];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const int64_t ra = tile * 16 + 8 * ks + t, rb = ra + 4;
            oka[ks] = ra < a.M; okb[ks] = rb < a.M;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const bool ok = (q & 2) ? okb[ks] : oka[ks];
                const int64_t off = ((q & 2) ? rb : ra) * 16 + g + 8 * (q & 1);
                tv[ks][q] = ok ? __ldg(a.dV1 + off) : 0.f;
                th[ks][q] = ok ? __ldg(a.H1 + off) : 0.f;
            }
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
                xa[ks][nb] = oka[ks] ? __ldg(a.X + ra * CIN + nb * 8 + g) : 0.f;
                xb[ks][nb] = okb[ks] ? __ldg(a.X + rb * CIN + nb * 8 + g) : 0.f;
            }
        }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            float av[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = q & 1;
                const bool ok = (q & 2) ? okb[ks] : oka[ks];
                av[q] = ok ? tsc[e] * (tv[ks][q] - tk1[e] - (th[ks][q] - tmu[e]) * tc2[e]) : 0.f;
            }
            FragA f;
            make_a(f, av[0], av[1], av[2], av[3]);
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
                FragB b;
                make_b(b, xa[ks][nb], xb[ks][nb]);
                mma3(accW[nb], f, b);
            }
        }
    }
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) {
        atomicAdd(&s_w[g * CIN + nb * 8 + 2 * t], accW[nb][0]);
        atomicAdd(&s_w[g * CIN + nb * 8 + 2 * t + 1], accW[nb][1]);
        atomicAdd(&s_w[(g + 8) * CIN + nb * 8 + 2 * t], accW[nb][2]);
        atomicAdd(&s_w[(g + 8) * CIN + nb * 8 + 2 * t + 1], accW[nb][3]);
    }
    __syncthreads();
    float* dst = a.dW + a.slot_stride * (int64_t)(blockIdx.x % kGradSlotsF);
    for (int i = tid; i < 16 * CIN; i += kThreads) atomicAdd(dst + i, s_w[i]);
}

// =========================================================================================== out_nn backward (16 → 64 layer)
// o = lrelu(BN3(H3)), H3 = x·W3ᵀ.  Given dO = dL/do (from the fusion layer's input gradient):
//   dv3 = dO ⊙ lrelu'(BN3(H3));  t_i = W3ᵀ·(sc3 ⊙ dv3_i)  → T[M,16]
//   sums over rows: s1 = Σdv3, s2 = Σdv3·Ĥ3, S = Σ dv3_iᵀ x_i [64×16], Sx = Σx_i, Sxx = Σ x_i x_iᵀ
// The last CTA derives (k1 = s1/M, k2 = s2/M, c2 = istd3·k2):
//   dγ3 += s2, dβ3 += s1
//   Q  = W3ᵀ·diag(sc3·c2)·W3 ,  a0 = W3ᵀ·(sc3 ⊙ (k1 − c2·mu3))        ⇒  dL/dx_i = t_i − a0 − Q·x_i
//   dW3[ch][a] += sc3[ch]·( S[ch][a] − k1[ch]·Sx[a] − c2[ch]·( (W3·Sxx)[ch][a] − mu3[ch]·Sx[a] ) )
constexpr int kOutSlots = 8;
constexpr int kOutPart = 64 + 64 + 16 + 256 + 1024;            // s1 | s2 | Sx | Sxx | S

struct OutBwdArgs {
    const float* dO; const float* H3;                         // [M, 64]
    const float* sc3; const float* sh3; const float* mu3; const float* is3; float slope3;
    const float* X;                                           // [M, 16]
    const float* W3;                                          // [64, 16]
    float* T;                                                 // [M, 16]
    float* part;                                              // [kOutSlots][kOutPart], zero on entry
    unsigned int* counter;
    double count;
    float* k1; float* k2; float* dgamma; float* dbeta;        // [64]
    float* dW3;                                               // [64, 16]  +=
    float* Q; float* a0;                                      // [16,16], [16]
    int64_t M;
};

// Each warp streams its 16-row tiles of dO and H3 through a private double-buffered cp.async ring (the next tile's 8 KB are in
// flight while this one is contracted; no register staging, no CTA-wide barrier).  The row-major pass turns the dO tile into dv3
// IN PLACE in shared memory; the contraction over rows (S = dv3ᵀ·x) then reads it back transposed, conflict-free (row pitch 72).
// Σ dv3·Ĥ3 is not accumulated per row: H3 = x·W3ᵀ, so Σ_r dv3[r,c]·H3[r,c] = Σ_a W3[c,a]·S[c,a] — the finalize derives it from S.
constexpr int kOutPitch = 72;                                   // floats per staged row (64 + 8: bank = 8·row + col)
constexpr int kOutStage = 2 * 16 * kOutPitch;                   // floats per stage: dO tile | H3 tile
constexpr size_t kOutSmem = (size_t)kWarps * 2 * kOutStage * sizeof(float);

__global__ void __launch_bounds__(kThreads, 1) out_bwd_kernel(const OutBwdArgs a) {
    extern __shared__ __align__(16) float ring[];               // [warp][stage][dO | H3][16][72]
    __shared__ float2 Bh[8 * 2 * 32], Bl[8 * 2 * 32];          // t-GEMM: [k8 step over the 64 channels][n block][lane]
    __shared__ __align__(16) float s_sc[64], s_sh[64], s_mu[64], s_is[64];
    __shared__ float s_acc[kOutPart];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    if (tid < 64) { s_sc[tid] = a.sc3[tid]; s_sh[tid] = a.sh3[tid]; s_mu[tid] = a.mu3[tid]; s_is[tid] = a.is3[tid]; }
    for (int i = tid; i < kOutPart; i += kThreads) s_acc[i] = 0.f;
    // B[k = channel][n ↔ x-channel phys_col(nb, n)] = sc3[ch]·W3[ch][x-channel];  k-step s = 2j+h: k = t' ↔ ch = 16j+4t'+2h, +1
    for (int i = tid; i < 8 * 2 * 32; i += kThreads) {
        const int s = i >> 6, nb = (i >> 5) & 1, gg = (i & 31) >> 2, tt = i & 3;
        const int ch = 16 * (s >> 1) + 4 * tt + 2 * (s & 1), xc = phys_col(nb, gg);
        store_split(Bh, Bl, i, __ldg(a.sc3 + ch) * __ldg(a.W3 + ch * 16 + xc), __ldg(a.sc3 + ch + 1) * __ldg(a.W3 + (ch + 1) * 16 + xc));
    }
    __syncthreads();

    float4 s1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) s1[j] = zero4();
    float accS[4][2][4], accXX[2][4], sx[2] = {0.f, 0.f};
#pragma unroll
    for (int mb = 0; mb < 4; ++mb)
#pragma unroll
        for (int nb = 0; nb < 2; ++nb)
#pragma unroll
            for (int e = 0; e < 4; ++e) accS[mb][nb][e] = 0.f;
#pragma unroll
    for (int nb = 0; nb < 2; ++nb)
#pragma unroll
        for (int e = 0; e < 4; ++e) accXX[nb][e] = 0.f;

    float* wring = ring + (size_t)warp * 2 * kOutStage;
    const int64_t ntiles = (a.M + 15) >> 4;
    const int64_t stride = (int64_t)gridDim.x * kWarps;
    auto issue = [&](int64_t tl, int st) {                     // 16 rows x 256 B of dO and of H3 → stage st (rows beyond M: zeros)
        float* dst = wring + st * kOutStage;
        if (tl < ntiles) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int c = lane + 32 * i, row = c >> 4, cc = c & 15;
                const int64_t r = tl * 16 + row;
                const bool ok = r < a.M;
                const int64_t off = (ok ? r : 0) * 64 + 4 * cc;
                cp_async16(dst + row * kOutPitch + 4 * cc, a.dO + off, ok);
                cp_async16(dst + 16 * kOutPitch + row * kOutPitch + 4 * cc, a.H3 + off, ok);
            }
        }
        cp_async_commit();
    };
    int64_t tile = (int64_t)blockIdx.x * kWarps + warp;
    int st = 0;
    issue(tile, 0);
    for (; tile < ntiles; tile += stride, st ^= 1) {
        issue(tile + stride, st ^ 1);
        const int64_t r0 = tile * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.M, ok1 = r1 < a.M;
        // x values for the transposed pass (global, 4-byte loads: 8 lanes = one sector) — issued before the wait
        float xv[2][4];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const int64_t ra = tile * 16 + 8 * ks + t, rb = ra + 4;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int64_t r = (q & 2) ? rb : ra;
                xv[ks][q] = r < a.M ? __ldg(a.X + r * 16 + g + 8 * (q & 1)) : 0.f;     // x[ra][g], x[ra][g+8], x[rb][g], x[rb][g+8]
            }
        }
        cp_async_wait<1>();                                    // this tile has landed (the newest group may still be in flight)
        __syncwarp();
        float* dOs = wring + st * kOutStage;
        const float* H3s = dOs + 16 * kOutPitch;
        // ---- row-major pass: dv3 (written back in place), column sums, t = dv3·(sc3 ⊙ W3)
        float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float* q0 = dOs + g * kOutPitch + 16 * j + 4 * t;
            float* q1 = q0 + 8 * kOutPitch;
            const float4 d0 = *reinterpret_cast<const float4*>(q0), d1 = *reinterpret_cast<const float4*>(q1);
            const float4 h0 = *reinterpret_cast<const float4*>(H3s + g * kOutPitch + 16 * j + 4 * t);
            const float4 h1 = *reinterpret_cast<const float4*>(H3s + (g + 8) * kOutPitch + 16 * j + 4 * t);
            const float4 sc = *reinterpret_cast<const float4*>(s_sc + 16 * j + 4 * t), sh = *reinterpret_cast<const float4*>(s_sh + 16 * j + 4 * t);
            const float4 v0 = mask4(d0, fma4(h0, sc, sh), a.slope3), v1 = mask4(d1, fma4(h1, sc, sh), a.slope3);   // zero rows stay zero
            *reinterpret_cast<float4*>(q0) = v0;
            *reinterpret_cast<float4*>(q1) = v1;
            s1[j] = add4(s1[j], add4(v0, v1));
            FragA f;
            make_a(f, v0.x, v1.x, v0.y, v1.y);
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) mma3(acc[nb], f, Bh[((2 * j) * 2 + nb) * 32 + lane], Bl[((2 * j) * 2 + nb) * 32 + lane]);
            make_a(f, v0.z, v1.z, v0.w, v1.w);
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) mma3(acc[nb], f, Bh[((2 * j + 1) * 2 + nb) * 32 + lane], Bl[((2 * j + 1) * 2 + nb) * 32 + lane]);
        }
        if (ok0) *reinterpret_cast<float4*>(a.T + r0 * 16 + 4 * t) = make_float4(acc[0][0], acc[0][1], acc[1][0], acc[1][1]);
        if (ok1) *reinterpret_cast<float4*>(a.T + r1 * 16 + 4 * t) = make_float4(acc[0][2], acc[0][3], acc[1][2], acc[1][3]);
        __syncwarp();                                          // dv3 tile complete
        // ---- transposed pass (k = rows): S += dv3ᵀ·x, Sxx += xᵀ·x, Sx += x
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            sx[0] += xv[ks][0] + xv[ks][2];
            sx[1] += xv[ks][1] + xv[ks][3];
            FragB xb[2];
            make_b(xb[0], xv[ks][0], xv[ks][2]);               // n block 0: x-channel g      (b0 = row ra, b1 = row rb)
            make_b(xb[1], xv[ks][1], xv[ks][3]);               // n block 1: x-channel g + 8
            FragA fx;
            make_a(fx, xv[ks][0], xv[ks][1], xv[ks][2], xv[ks][3]);   // A = xᵀ: (m = g, k = ra) (m = g+8, k = ra) (g, rb) (g+8, rb)
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) mma3(accXX[nb], fx, xb[nb]);
            const float* ra_ = dOs + (8 * ks + t) * kOutPitch + g;
            const float* rb_ = ra_ + 4 * kOutPitch;
#pragma unroll
            for (int mb = 0; mb < 4; ++mb) {
                FragA f;                                       // A = dv3ᵀ: (ch = 16mb+g, ra) (ch+8, ra) (ch, rb) (ch+8, rb)
                make_a(f, ra_[16 * mb], ra_[16 * mb + 8], rb_[16 * mb], rb_[16 * mb + 8]);
#pragma unroll
                for (int nb = 0; nb < 2; ++nb) mma3(accS[mb][nb], f, xb[nb]);
            }
        }
        __syncwarp();                                          // stage free for the copy issued two iterations from now
    }
    cp_async_wait<0>();
    // ---- CTA reduction in shared memory, then one atomic per value into a slot
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float v1[4] = {s1[j].x, s1[j].y, s1[j].z, s1[j].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float x1 = group8_sum(v1[e]);
            if (g == 0) atomicAdd(&s_acc[16 * j + 4 * t + e], x1);
        }
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        float v = sx[e];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if (t == 0) atomicAdd(&s_acc[128 + g + 8 * e], v);
    }
#pragma unroll
    for (int nb = 0; nb < 2; ++nb) {
        float* xx = s_acc + 144;
        atomicAdd(&xx[g * 16 + nb * 8 + 2 * t], accXX[nb][0]);
        atomicAdd(&xx[g * 16 + nb * 8 + 2 * t + 1], accXX[nb][1]);
        atomicAdd(&xx[(g + 8) * 16 + nb * 8 + 2 * t], accXX[nb][2]);
        atomicAdd(&xx[(g + 8) * 16 + nb * 8 + 2 * t + 1], accXX[nb][3]);
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) {
            float* ss = s_acc + 400 + mb * 16 * 16;
            atomicAdd(&ss[g * 16 + nb * 8 + 2 * t], accS[mb][nb][0]);
            atomicAdd(&ss[g * 16 + nb * 8 + 2 * t + 1], accS[mb][nb][1]);
            atomicAdd(&ss[(g + 8) * 16 + nb * 8 + 2 * t], accS[mb][nb][2]);
            atomicAdd(&ss[(g + 8) * 16 + nb * 8 + 2 * t + 1], accS[mb][nb][3]);
        }
    }
    __syncthreads();
    {
        float* dst = a.part + (size_t)(blockIdx.x % kOutSlots) * kOutPart;
        for (int i = tid; i < kOutPart; i += kThreads)
            if (i < 64 || i >= 128) atomicAdd(dst + i, s_acc[i]);      // [64, 128) (Σ dv3·Ĥ3) is derived in the finalize
    }
    if (!arrive_is_last(a.counter)) return;
    // ---- finalize (one CTA): fold the slots, then the small algebra above
    for (int i = tid; i < kOutPart; i += kThreads) {
        float x[kOutSlots];
#pragma unroll
        for (int p = 0; p < kOutSlots; ++p) x[p] = __ldcg(a.part + (size_t)p * kOutPart + i);
        float tot = 0.f;
#pragma unroll
        for (int p = 0; p < kOutSlots; ++p) tot += x[p];
        s_acc[i] = tot;
    }
    __syncthreads();
    const float* S1 = s_acc; float* S2 = s_acc + 64; const float* Sx = s_acc + 128; const float* Sxx = s_acc + 144; const float* S = s_acc + 400;
    __shared__ float f_k1[64], f_c2[64];
    if (tid < 64) {
        float hs = 0.f;                                        // Σ_rows dv3·H3 for channel tid
#pragma unroll
        for (int b = 0; b < 16; ++b) hs = fmaf(__ldg(a.W3 + tid * 16 + b), S[tid * 16 + b], hs);
        const float s2 = s_is[tid] * (hs - s_mu[tid] * S1[tid]);
        S2[tid] = s2;
        const float k1 = (float)((double)S1[tid] / a.count), k2 = (float)((double)s2 / a.count);
        a.k1[tid] = k1; a.k2[tid] = k2;
        if (a.dgamma) a.dgamma[tid] += s2;
        if (a.dbeta) a.dbeta[tid] += S1[tid];
        f_k1[tid] = k1; f_c2[tid] = s_is[tid] * k2;
    }
    __syncthreads();
    {   // Q[a][b] (thread = one entry), a0[a]
        const int qa = tid >> 4, qb = tid & 15;
        float q = 0.f;
        for (int ch = 0; ch < 64; ++ch) q = fmaf(__ldg(a.W3 + ch * 16 + qa) * s_sc[ch] * f_c2[ch], __ldg(a.W3 + ch * 16 + qb), q);
        a.Q[tid] = q;
        if (tid < 16) {
            float v = 0.f;
            for (int ch = 0; ch < 64; ++ch) v = fmaf(__ldg(a.W3 + ch * 16 + tid) * s_sc[ch], f_k1[ch] - f_c2[ch] * s_mu[ch], v);
            a.a0[tid] = v;
        }
    }
    for (int i = tid; i < 1024; i += kThreads) {
        const int ch = i >> 4, xc = i & 15;
        float wxx = 0.f;
#pragma unroll
        for (int b = 0; b < 16; ++b) wxx = fmaf(__ldg(a.W3 + ch * 16 + b), Sxx[b * 16 + xc], wxx);
        a.dW3[i] += s_sc[ch] * (S[i] - f_k1[ch] * Sx[xc] - f_c2[ch] * (wxx - s_mu[ch] * Sx[xc]));
    }
}

// =========================================================================================== mean-field backward, fused
__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float quad_sum(float v) {              // the 4 lanes of a point
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
// all-gather of the float4 slices of the 4 lanes of a point → full[16]
__device__ __forceinline__ void gather16(float4 v, float (&full)[16], int lane) {
    const int gb = lane & ~3;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        full[4 * s + 0] = __shfl_sync(0xffffffffu, v.x, gb + s);
        full[4 * s + 1] = __shfl_sync(0xffffffffu, v.y, gb + s);
        full[4 * s + 2] = __shfl_sync(0xffffffffu, v.z, gb + s);
        full[4 * s + 3] = __shfl_sync(0xffffffffu, v.w, gb + s);
    }
}
// out[c0..c0+3] = Σ_k full[k]·Mat[k][c0+e]   (Mat row-major [16][16] in shared memory)
__device__ __forceinline__ float4 rowvec_mat16(const float (&full)[16], const float* Mat, int c0) {
    float4 o = zero4();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const float4 m = *reinterpret_cast<const float4*>(Mat + k * 16 + c0);
        o.x = fmaf(full[k], m.x, o.x); o.y = fmaf(full[k], m.y, o.y); o.z = fmaf(full[k], m.z, o.z); o.w = fmaf(full[k], m.w, o.w);
    }
    return o;
}

constexpr int kStepSlots = 8;
struct StepBwdArgs {
    const float* Hy; const float* sc_y;                       // pre-BN pairwise embedding [M,16], γ·istd of its BatchNorm
    const float* z; const float* xprev; const int64_t* nbr;   // [M,16], [M,16], [M,16] (column 0 = self, skipped)
    const float* Cm; const float* Minv;                       // [16,16]
    const float* g;                                           // [M,16]  dL/dx^t  (t_i of out_bwd when Q != null)
    const float* xT; const float* Q; const float* a0;         // out_nn BatchNorm-backward correction: g_i ← g_i − a0 − Q·xT_i
    float* Gz; int gz_acc;                                    // owner rows: h_i (= or +=)
    float* gprev; float* Gy;                                  // scatter targets, zero-initialised
    float* GC; float* GM; int64_t slot_stride;                // [16,16] partial slots (kGradSlots), +=
    float* ysum;                                              // [kStepSlots][16] partial Σ_edges 2Ga·df², zero-initialised
    int64_t total, N;
    // last launch of the backward loop: fold ysum into the BatchNorm-backward constants of the y layer (pairwise_nn[1]; gamma_y = its weight)
    int finalize; unsigned int* counter; double count; const float* gamma_y;
    // Always 0: the three `sched_mask` tests in the kernel never fire.  Without them nvcc schedules the gather / reduction loop
    // differently and the kernel measured 6.5 % slower (147.9 -> 157.6 us at the S1 shape, B200 at 1,000 W).
    int sched_mask;
    float* k1; float* k2; float* dgamma; float* dbeta;
};

constexpr int KN = 15;
__global__ void __launch_bounds__(128, 3) step_bwd_kernel(const StepBwdArgs a) {
    __shared__ __align__(16) float4 fCT[128], fMT[128], fC[128], fQ[128];   // pre-split MMA fragments of Cᵀ, Minvᵀ, C, Q (rows8_mat16)
    __shared__ __align__(16) float stage[4][4][8][24];           // per warp: m, h, v, g rows of its 8 points (MMA operand staging)
    __shared__ __align__(16) float s_gc[4][32][20];              // per warp and lane: its 16 running GC | GM fragment values (pitch 20: conflict-free 128-bit RMW)
    __shared__ float s_y[16];
    __shared__ __align__(16) long long s_idx[4][2][8][16];          // per warp: double-buffered neighbour-index rows of its next group (cp.async)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    stage_mat16(fC, [&](int k, int n) { return a.Cm[k * 16 + n]; }, tid, 128);
    stage_mat16(fCT, [&](int k, int n) { return a.Cm[n * 16 + k]; }, tid, 128);
    stage_mat16(fMT, [&](int k, int n) { return a.Minv[n * 16 + k]; }, tid, 128);
    stage_mat16(fQ, [&](int k, int n) { return a.Q ? a.Q[k * 16 + n] : 0.f; }, tid, 128);
    for (int i = tid; i < 4 * 32 * 20; i += 128) (&s_gc[0][0][0])[i] = 0.f;
    if (tid < 16) s_y[tid] = 0.f;
    __syncthreads();
    const int sub = lane & 3, c0 = 4 * sub, pt = lane >> 2, gfr = lane >> 2, tfr = lane & 3;
    const float4 sc = ldg4(a.sc_y + c0);
    float4 ey = zero4();                                       // Σ_edges 2Ga·df·dfH for channels c0..c0+3
    float (*st)[8][24] = stage[warp];
    float4* wacc = reinterpret_cast<float4*>(&s_gc[warp][lane][0]);   // [accC nb0 | accC nb1 | accM nb0 | accM nb1]
    const int64_t ngroups = (a.total + 7) >> 3;
    const int64_t gstride = (int64_t)gridDim.x * 4;
    // The gathers of a group cannot be issued before its neighbour indices have arrived: that dependent round trip (≈1 us, with only
    // 8 warps per SM to hide it) is taken off the critical path by prefetching the NEXT group's 8 index rows (1 KB) into shared memory.
    auto prefetch_idx = [&](int64_t g_, int buf) {
        if (g_ < ngroups) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int c = lane + 32 * i, row = c >> 3, ch = c & 7;       // 8 rows x 8 chunks of 16 B
                const int64_t pp = min(g_ * 8 + row, a.total - 1);
                cp_async16(&s_idx[warp][buf][row][2 * ch], a.nbr + pp * 16 + 2 * ch, true);
            }
        }
        cp_async_commit();
    };
    int ibuf = 0;
    prefetch_idx((int64_t)blockIdx.x * 4 + warp, 0);
    for (int64_t grp = (int64_t)blockIdx.x * 4 + warp; grp < ngroups; grp += gstride, ibuf ^= 1) {
        prefetch_idx(grp + gstride, ibuf ^ 1);
        int64_t p = grp * 8 + pt;
        const bool valid = p < a.total;
        if (!valid) p = a.total - 1;
        const int64_t base = (p / a.N) * a.N;
        int rj[KN];
        {   // the 16 int64 neighbour indices of a point are one 128-byte row: two 128-bit loads per lane, shared by shuffle
            cp_async_wait<1>();                                // this group's rows have landed (the next group's may be in flight)
            __syncwarp();
            const longlong2 ia = *reinterpret_cast<const longlong2*>(&s_idx[warp][ibuf][pt][2 * sub]);
            const longlong2 ib = *reinterpret_cast<const longlong2*>(&s_idx[warp][ibuf][pt][8 + 2 * sub]);
            const int r0 = (int)ia.x, r1 = (int)ia.y, r2 = (int)ib.x, r3 = (int)ib.y;   // indices 2s, 2s+1, 8+2s, 8+2s+1
            const int gb = lane & ~3;
#pragma unroll
            for (int k = 1; k < 16; ++k) {                    // index k lives in lane (k & 7) >> 1 of the group, register (k>>3)*2 + (k&1)
                const int v = (k & 8) ? ((k & 1) ? r3 : r2) : ((k & 1) ? r1 : r0);
                rj[k - 1] = __shfl_sync(0xffffffffu, v, gb + ((k & 7) >> 1));
            }
        }
        const float4 hyi = ldg4(a.Hy + p * 16 + c0);
        const float4 gi_raw = ldg4(a.g + p * 16 + c0);
        const float4 xt_raw = a.Q ? ldg4(a.xT + p * 16 + c0) : zero4();
        // the point-local algebra (h = g·Minvᵀ, q = h·Cᵀ; tensor cores, chained through registers)
        float4 q;
        {
            float4 gi = gi_raw;
            if (a.Q) {
                const float4 qx = rows8_mat16(xt_raw, fQ, lane);
                const float4 a0v = ldg4(a.a0 + c0);
                gi = make_float4(gi.x - a0v.x - qx.x, gi.y - a0v.y - qx.y, gi.z - a0v.z - qx.z, gi.w - a0v.w - qx.w);
            }
            const float4 h = rows8_mat16(gi, fMT, lane);       // h = g·Minvᵀ
            q = rows8_mat16(h, fCT, lane);                     // q = h·Cᵀ
            if (valid) {
                float* gz = a.Gz + p * 16 + c0;
                float4 o = h;
                if (a.gz_acc) o = add4(o, *reinterpret_cast<const float4*>(gz));
                *reinterpret_cast<float4*>(gz) = o;
            }
            *reinterpret_cast<float4*>(&st[1][pt][c0]) = valid ? h : zero4();
            *reinterpret_cast<float4*>(&st[3][pt][c0]) = valid ? gi : zero4();
        }
        float4 dfj[KN];
        float dj[KN], gsj[KN];
        float mx = -INFINITY;
        float l = 0.f, tacc = 0.f;
        float4 acc = zero4();
        // x_j rows are consumed as they arrive (online softmax) instead of all being gathered first: 60 fewer live registers, 3 CTAs per SM
#pragma unroll
        for (int k = 0; k < KN; ++k) {
            const int64_t row = base + rj[k];
            const float4 hj = ldg4(a.Hy + row * 16 + c0), x = ldg4(a.xprev + row * 16 + c0);
            dfj[k] = mul4(sub4(hyi, hj), sc);                  // df = sc ⊙ (Hy_i − Hy_j) = y_i − y_j
            const float al = -quad_sum(dot4(dfj[k], dfj[k]));
            gsj[k] = quad_sum(dot4(q, x));
            const float nm = fmaxf(mx, al);
            const float corr = __expf(mx - nm), pj = __expf(al - nm);
            l = fmaf(l, corr, pj);
            tacc = fmaf(tacc, corr, pj * gsj[k]);
            acc.x = fmaf(acc.x, corr, pj * x.x); acc.y = fmaf(acc.y, corr, pj * x.y);
            acc.z = fmaf(acc.z, corr, pj * x.z); acc.w = fmaf(acc.w, corr, pj * x.w);
            dj[k] = al;
            mx = nm;
        }
#pragma unroll
        for (int k = 0; k < KN; ++k) dj[k] = __expf(dj[k] - mx);
        const float inv_l = 1.0f / l;
        const float sdot = tacc * inv_l;
        {
            const float4 msg = make_float4(acc.x * inv_l, acc.y * inv_l, acc.z * inv_l, acc.w * inv_l);
            float4 v = rows8_mat16(msg, fC, lane);             // v = z + m·C
            v = add4(v, ldg4(a.z + p * 16 + c0));
            *reinterpret_cast<float4*>(&st[0][pt][c0]) = valid ? msg : zero4();
            *reinterpret_cast<float4*>(&st[2][pt][c0]) = valid ? v : zero4();
        }
        float4 gyi = zero4();
#pragma unroll
        for (int k = 0; k < KN; ++k) {
            const float s_ = dj[k] * inv_l;
            const float ga2 = valid ? 2.0f * s_ * (gsj[k] - sdot) : 0.f;
            const float4 df = dfj[k];
            const float4 gd = make_float4(ga2 * df.x, ga2 * df.y, ga2 * df.z, ga2 * df.w);
            gyi = sub4(gyi, gd);
            ey = fma4(gd, df, ey);                             // Σ 2Ga·df² (divided by sc at the end: df·dfH = df²/sc)
            if (valid) {
                // the index is re-read from the (still intact) shared-memory row instead of staying live in a register
                const int64_t row = base + (int)s_idx[warp][ibuf][pt][k + 1];
                if (!(a.sched_mask & 1)) red_add_v4(a.Gy + row * 16 + c0, gd);
                if (!(a.sched_mask & 2)) red_add_v4(a.gprev + row * 16 + c0, make_float4(s_ * q.x, s_ * q.y, s_ * q.z, s_ * q.w));
            }
        }
        if (valid) red_add_v4(a.Gy + p * 16 + c0, gyi);
        // ---- GC += mᵀ·h, GM += vᵀ·g over the warp's 8 points on the tensor cores (k = point)
        __syncwarp();
        if (!(a.sched_mask & 4)) {
            FragA fm, fv;
            make_a(fm, st[0][tfr][gfr], st[0][tfr][gfr + 8], st[0][tfr + 4][gfr], st[0][tfr + 4][gfr + 8]);
            make_a(fv, st[2][tfr][gfr], st[2][tfr][gfr + 8], st[2][tfr + 4][gfr], st[2][tfr + 4][gfr + 8]);
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) {
                FragB bh_, bg_;
                make_b(bh_, st[1][tfr][nb * 8 + gfr], st[1][tfr + 4][nb * 8 + gfr]);
                make_b(bg_, st[3][tfr][nb * 8 + gfr], st[3][tfr + 4][nb * 8 + gfr]);
                const float4 c4 = wacc[nb], m4 = wacc[2 + nb];
                float cC[4] = {c4.x, c4.y, c4.z, c4.w}, cM[4] = {m4.x, m4.y, m4.z, m4.w};
                mma3(cC, fm, bh_);
                mma3(cM, fv, bg_);
                wacc[nb] = make_float4(cC[0], cC[1], cC[2], cC[3]);
                wacc[2 + nb] = make_float4(cM[0], cM[1], cM[2], cM[3]);
            }
        }
        __syncwarp();
    }
    // ---- CTA reduction: GC | GM (512 values, 4 warps) and the y-layer sum (16 values)
    {
        const float v[4] = {ey.x, ey.y, ey.z, ey.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float x = group8_sum(v[e]);
            if (pt == 0) atomicAdd(&s_y[c0 + e], x);
        }
    }
    __syncthreads();
    {
        const int64_t slot = blockIdx.x % kGradSlotsF;
        // fragment value k of lane l: matrix k >> 3 (GC / GM), block nb = (k >> 2) & 1, element e = k & 3 ↔ (row g (+8 if e >= 2), col 8nb + 2t + (e & 1))
        for (int i = tid; i < 512; i += 128) {
            const int l = i >> 4, k = i & 15, gg = l >> 2, tt = l & 3, e = k & 3;
            const int row = gg + ((e & 2) ? 8 : 0), col = ((k >> 2) & 1) * 8 + 2 * tt + (e & 1);
            const float v = s_gc[0][l][k] + s_gc[1][l][k] + s_gc[2][l][k] + s_gc[3][l][k];
            atomicAdd(((k >> 3) ? a.GM : a.GC) + a.slot_stride * slot + row * 16 + col, v);
        }
        if (tid < 16) atomicAdd(a.ysum + (blockIdx.x % kStepSlots) * 16 + tid, s_y[tid]);
    }
    if (!a.finalize) return;
    if (!arrive_is_last(a.counter)) return;
    if (tid < 16) {
        float e = 0.f;
#pragma unroll
        for (int p = 0; p < kStepSlots; ++p) e += __ldcg(a.ysum + p * 16 + tid);
        // Σ_rows Gy·Ĥ = Σ_edges 2Ga·df·(Ĥ_j − Ĥ_i) = −istd·Σ_edges 2Ga·df·dfH = −Σ_edges 2Ga·df² / γ   (df = γ·istd·dfH);
        // Σ_rows Gy = 0 identically (every edge adds +gd to one row and −gd to another)
        const float gm = a.gamma_y[tid];
        const double s2 = gm != 0.f ? -(double)e / (double)gm : 0.0;
        a.k1[tid] = 0.f;
        a.k2[tid] = (float)(s2 / a.count);
        if (a.dgamma) a.dgamma[tid] += (float)s2;
        (void)a.dbeta;                                         // dβ += 0
    }
}

// =========================================================================================== upsample backward + BN sums
// v_i = Gz_i (+ G0_i);  Gu[b·Nc + up(i)] += v_i;  s1 = Σ_i v_i,  s2 = Σ_i v_i ⊙ Ĥu[up(i)]   (= Σ_rows Gu, Σ_rows Gu·Ĥu)
struct UpBwdArgs {
    const float* Gz; const float* G0; const int64_t* up;
    const float* Hu; const float* mu; const float* is;        // unary_nn[1]: pre-BN output [B·Nc,16] and its batch statistics
    float* Gu;                                                // [B·Nc,16], zero-initialised
    int64_t total, N, Nc;
    BwdFin fin;
};

__global__ void __launch_bounds__(kThreads, 4) upsample_bwd_kernel(const UpBwdArgs a) {
    __shared__ float s_part[kWarps][32];
    __shared__ double s_red[kThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, sub = lane & 3, c0 = 4 * sub;
    const float4 mu = ldg4(a.mu + c0), is = ldg4(a.is + c0);
    float4 s1 = zero4(), s2 = zero4();
    const int64_t nthr = (int64_t)gridDim.x * kThreads;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + tid; i < a.total * 4; i += nthr) {
        const int64_t m = i >> 2;
        const int64_t dst = (m / a.N) * a.Nc + __ldg(a.up + m);
        float4 v = ldg4(a.Gz + m * 16 + c0);
        if (a.G0) v = add4(v, ldg4(a.G0 + m * 16 + c0));
        const float4 hu = ldg4(a.Hu + dst * 16 + c0);
        red_add_v4(a.Gu + dst * 16 + c0, v);
        s1 = add4(s1, v);
        s2 = fma4(v, mul4(sub4(hu, mu), is), s2);
    }
    const float v1[4] = {s1.x, s1.y, s1.z, s1.w}, v2[4] = {s2.x, s2.y, s2.z, s2.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const float x1 = group8_sum(v1[e]), x2 = group8_sum(v2[e]);
        if ((lane >> 2) == 0) { s_part[warp][c0 + e] = x1; s_part[warp][16 + c0 + e] = x2; }
    }
    __syncthreads();
    if (tid < 32) {
        float tot = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) tot += s_part[w][tid];
        a.fin.part[(size_t)blockIdx.x * 32 + tid] = tot;
    }
    if (grid_reduce_rows<32, kThreads>(a.fin.part, part_group_rows(a.fin.part), a.fin.counter, s_red) && tid < 16)
        bn_bwd_finalize(a.fin, s_red[tid], s_red[16 + tid], tid);
}

inline int grid_for(int64_t units, int per_cta, int ctas_per_sm) {
    const int64_t want = ceil_div(units, per_cta);
    return (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)kNumSMs * ctas_per_sm));
}
inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace cl
}  // namespace crf

using namespace crf;
using namespace crf::cl;

extern "C" {

int crfconv_fused_max_parts(void) { return kMaxTicketGrid; }
int crfconv_fused_part_floats(void) { return kPartFloats; }
int crfconv_fused_counter_ints(void) { return kTicketInts; }

// H[M,16] = act(X[M,Cin])·Wᵀ with the BatchNorm statistics of H finalized in the same launch.  Cin ∈ {16, 64, 128}; pscale/pshift
// (BN affine of the previous layer, applied with LeakyReLU(pslope) while loading X) are required for Cin = 16 and must be NULL otherwise.
// part: scratch of crfconv_fused_max_parts()·32 floats; counter: one zeroed uint32 (left zero).  Outputs scale/shift/mean/invstd [16].
int crfconv_lin16_fwd(const float* X, int Cin, const float* W, const float* pscale, const float* pshift, float pslope, float* Y, int64_t M,
                      float* part, unsigned int* counter, const float* gamma, const float* beta, float* running_mean,
                      float* running_var, float eps, float momentum, float* scale, float* shift, float* mean, float* invstd, void* stream) {
    if (!X || !W || !Y || !part || !counter || !scale || !shift || M <= 0 || !al16(X) || !al16(Y)) return CRF_ERR_INVALID_ARG;
    LinFwdArgs a{};
    a.X = X; a.W = W; a.pscale = pscale; a.pshift = pshift; a.pslope = pslope; a.Y = Y; a.M = M;
    a.fin = FwdFin{part, counter, gamma, beta, running_mean, running_var, eps, momentum, (double)M, scale, shift, mean, invstd};
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t tiles = ceil_div(M, 16);
    if (Cin == 16) {
        if (!pscale || !pshift) return CRF_ERR_INVALID_ARG;
        lin16_fwd_kernel<16, true><<<grid_for(tiles, kWarps * 4, 2), kThreads, 0, st>>>(a);
    } else if (Cin == 64 && !pscale) {
        lin16_fwd_kernel<64, false><<<grid_for(tiles, kWarps * 2, 2), kThreads, 0, st>>>(a);
    } else if (Cin == 128 && !pscale) {
        lin16_fwd_kernel<128, false><<<grid_for(tiles, kWarps * 2, 1), kThreads, 0, st>>>(a);
    } else {
        return CRF_ERR_UNSUPPORTED;
    }
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// H[M,64] = X[M,16]·Wᵀ + BatchNorm finalize of H (out_nn's Linear).  stats: [CRFCONV_STAT_SLOTS][128] zeroed floats.
int crfconv_up16_fwd(const float* X, const float* W, int Cout, float* Y, int64_t M, float* stats, unsigned int* counter, const float* gamma,
                     const float* beta, float* running_mean, float* running_var, float eps, float momentum, float* scale, float* shift,
                     float* mean, float* invstd, void* stream) {
    if (!X || !W || !Y || !stats || !counter || !scale || !shift || M <= 0 || !al16(X) || !al16(Y)) return CRF_ERR_INVALID_ARG;
    if (Cout != 64) return CRF_ERR_UNSUPPORTED;
    Up16FwdArgs a{};
    a.X = X; a.W = W; a.Y = Y; a.M = M;
    a.fin = FwdFin{stats, counter, gamma, beta, running_mean, running_var, eps, momentum, (double)M, scale, shift, mean, invstd};
    up16_fwd_kernel<64><<<grid_for(ceil_div(M, 16), kWarps * 2, 2), kThreads, 0, (cudaStream_t)stream>>>(a);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// Backward of a 16→16 layer that follows a BN+LeakyReLU'd 16-channel layer (see mid16_bwd_kernel).  dW2 points at the first partial
// slot (CRFCONV_GRAD_SLOTS slots, slot_stride floats apart, zero-initialised, folded by crfconv_grad_slots_reduce).
int crfconv_mid16_bwd(const float* dY, const float* H2, const float* sc2, const float* mu2, const float* is2, const float* k1_2,
                      const float* k2_2, const float* H1, const float* sc1, const float* sh1, const float* mu1, const float* is1,
                      float slope1, const float* W2, float* dV1, float* dW2, int64_t slot_stride, int64_t M, float* part,
                      unsigned int* counter, float* k1_1, float* k2_1, float* dgamma1, float* dbeta1, void* stream) {
    if (!dY || !H2 || !H1 || !W2 || !dV1 || !dW2 || !part || !counter || !k1_1 || !k2_1 || M <= 0) return CRF_ERR_INVALID_ARG;
    Mid16BwdArgs a{};
    a.dY = dY; a.H2 = H2; a.b2 = BnB{sc2, mu2, is2, k1_2, k2_2};
    a.H1 = H1; a.sc1 = sc1; a.sh1 = sh1; a.mu1 = mu1; a.is1 = is1; a.slope1 = slope1;
    a.W2 = W2; a.dV1 = dV1; a.dW2 = dW2; a.slot_stride = slot_stride; a.M = M;
    a.fin = BwdFin{part, counter, (double)M, k1_1, k2_1, dgamma1, dbeta1};
    mid16_bwd_kernel<<<grid_for(ceil_div(M, 16), kWarps * 4, 2), kThreads, 0, (cudaStream_t)stream>>>(a);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// dX[M,Cin] (= or +=) dH1·W1 with dH1 the BatchNorm backward of (dV1, H1).  Cin ∈ {64, 128}.
int crfconv_in16_dgrad(const float* dV1, const float* H1, const float* sc1, const float* mu1, const float* is1, const float* k1,
                       const float* k2, const float* W1, int Cin, float* dX, int accumulate, int64_t M, void* stream) {
    if (!dV1 || !H1 || !W1 || !dX || M <= 0 || !al16(dX)) return CRF_ERR_INVALID_ARG;
    In16DgradArgs a{dV1, H1, BnB{sc1, mu1, is1, k1, k2}, W1, dX, M};
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t tiles = ceil_div(M, 16);
    if (Cin == 64) {
        if (accumulate) in16_dgrad_kernel<64, true><<<grid_for(tiles, kWarps * 2, 2), kThreads, 0, st>>>(a);
        else in16_dgrad_kernel<64, false><<<grid_for(tiles, kWarps * 2, 2), kThreads, 0, st>>>(a);
    } else if (Cin == 128) {
        if (accumulate) in16_dgrad_kernel<128, true><<<grid_for(tiles, kWarps * 2, 1), kThreads, 0, st>>>(a);
        else in16_dgrad_kernel<128, false><<<grid_for(tiles, kWarps * 2, 1), kThreads, 0, st>>>(a);
    } else {
        return CRF_ERR_UNSUPPORTED;
    }
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// dW1[16,Cin] partial slots += dH1ᵀ·X.  Cin ∈ {64, 128}.
int crfconv_in16_wgrad(const float* dV1, const float* H1, const float* sc1, const float* mu1, const float* is1, const float* k1,
                       const float* k2, const float* X, int Cin, float* dW, int64_t slot_stride, int64_t M, void* stream) {
    if (!dV1 || !H1 || !X || !dW || M <= 0) return CRF_ERR_INVALID_ARG;
    In16WgradArgs a{dV1, H1, BnB{sc1, mu1, is1, k1, k2}, X, dW, slot_stride, M};
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t steps = ceil_div(M, 16);
    if (Cin == 64) in16_wgrad_kernel<64><<<grid_for(steps, kWarps * 2, 2), kThreads, 0, st>>>(a);
    else if (Cin == 128) in16_wgrad_kernel<128><<<grid_for(steps, kWarps * 2, 1), kThreads, 0, st>>>(a);
    else return CRF_ERR_UNSUPPORTED;
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

int crfconv_out_bwd_part_floats(void) { return kOutSlots * kOutPart; }

// out_nn (16 → 64, BN, LeakyReLU) backward in one pass over dO (see out_bwd_kernel).  part: crfconv_out_bwd_part_floats() zeroed floats.
int crfconv_out16_bwd(const float* dO, const float* H3, const float* sc3, const float* sh3, const float* mu3, const float* is3,
                      float slope3, const float* X, const float* W3, float* T, int64_t M, float* part, unsigned int* counter,
                      float* k1, float* k2, float* dgamma, float* dbeta, float* dW3, float* Q, float* a0, void* stream) {
    if (!dO || !H3 || !X || !W3 || !T || !part || !counter || !k1 || !k2 || !dW3 || !Q || !a0 || M <= 0) return CRF_ERR_INVALID_ARG;
    OutBwdArgs a{};
    a.dO = dO; a.H3 = H3; a.sc3 = sc3; a.sh3 = sh3; a.mu3 = mu3; a.is3 = is3; a.slope3 = slope3;
    a.X = X; a.W3 = W3; a.T = T; a.part = part; a.counter = counter; a.count = (double)M;
    a.k1 = k1; a.k2 = k2; a.dgamma = dgamma; a.dbeta = dbeta; a.dW3 = dW3; a.Q = Q; a.a0 = a0; a.M = M;
    static bool attr_set = false;
    if (!attr_set) {
        CRF_CUDA(cudaFuncSetAttribute(out_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kOutSmem));
        attr_set = true;
    }
    out_bwd_kernel<<<grid_for(ceil_div(M, 16), kWarps * 2, 1), kThreads, kOutSmem, (cudaStream_t)stream>>>(a);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// Mean-field backward of one step, F = 16, K = 16 (see step_bwd_kernel).  Q/a0/xT may be NULL (no out_nn correction).
// ysum: 8·16 zeroed floats shared by all steps of one backward; finalize != 0 on the last launch (t = 1).
int crfconv_crf_step_bwd_fused(const float* Hy, const float* sc_y, const float* z, const float* xprev, const int64_t* neighbor_idx,
                               const float* Cm, const float* Minv, const float* g, const float* xT, const float* Q, const float* a0,
                               float* Gz, int gz_acc, float* gprev, float* Gy, float* GC, float* GM, int64_t slot_stride,
                               float* ysum, int64_t B, int64_t N, int K, int F, int finalize, unsigned int* counter,
                               const float* gamma_y, float* k1, float* k2, float* dgamma, float* dbeta, void* stream) {
    if (F != 16 || K != 16) return CRF_ERR_UNSUPPORTED;
    if (!Hy || !sc_y || !z || !xprev || !neighbor_idx || !Cm || !Minv || !g || !Gz || !gprev || !Gy || !GC || !GM || !ysum || B <= 0 || N <= 0)
        return CRF_ERR_INVALID_ARG;
    if (Q && (!xT || !a0)) return CRF_ERR_INVALID_ARG;
    if (finalize && (!counter || !gamma_y || !k1 || !k2)) return CRF_ERR_INVALID_ARG;
    StepBwdArgs a{};
    a.Hy = Hy; a.sc_y = sc_y; a.z = z; a.xprev = xprev; a.nbr = neighbor_idx; a.Cm = Cm; a.Minv = Minv; a.g = g;
    a.xT = xT; a.Q = Q; a.a0 = a0; a.Gz = Gz; a.gz_acc = gz_acc; a.gprev = gprev; a.Gy = Gy; a.GC = GC; a.GM = GM;
    a.slot_stride = slot_stride; a.ysum = ysum; a.total = B * N; a.N = N;
    a.finalize = finalize; a.counter = counter; a.count = (double)(B * N); a.gamma_y = gamma_y; a.k1 = k1; a.k2 = k2; a.dgamma = dgamma; a.dbeta = dbeta;
    step_bwd_kernel<<<grid_for(ceil_div(a.total, 8), 4 * 4, 3), 128, 0, (cudaStream_t)stream>>>(a);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// Gu[B·Nc,16] += (Gz + G0)[·] through up_idx, and the BatchNorm-backward constants of unary_nn[1] (count = B·Nc rows).
int crfconv_crf_upsample_bwd_fused(const float* Gz, const float* G0, const int64_t* up_idx, const float* Hu, const float* mu,
                                   const float* is, float* Gu, int64_t B, int64_t N, int64_t Nc, float* part, unsigned int* counter,
                                   float* k1, float* k2, float* dgamma, float* dbeta, void* stream) {
    if (!Gz || !up_idx || !Hu || !mu || !is || !Gu || !part || !counter || !k1 || !k2 || B <= 0 || N <= 0 || Nc <= 0) return CRF_ERR_INVALID_ARG;
    UpBwdArgs a{};
    a.Gz = Gz; a.G0 = G0; a.up = up_idx; a.Hu = Hu; a.mu = mu; a.is = is; a.Gu = Gu; a.total = B * N; a.N = N; a.Nc = Nc;
    a.fin = BwdFin{part, counter, (double)(B * Nc), k1, k2, dgamma, dbeta};
    upsample_bwd_kernel<<<grid_for(a.total * 4, kThreads * 4, 3), kThreads, 0, (cudaStream_t)stream>>>(a);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

}  // extern "C"
