// Linear (+ training-mode BatchNorm + LeakyReLU) chains of the hot path on sm_100a tensor cores.
//
// Every dense contraction of the reference goes through models/common.py:26-40
//     MLP = nn.Linear(bias = not bn) → FastBatchNorm1d (statistics over all B·N rows) → activation
// The rows (M = B·N points or B·N·K edges) outnumber the channels by 10^3-10^5, so these GEMMs are A-streaming
// (HBM/L2-bound) and the BatchNorm forces a grid-wide statistics barrier between a Linear and its activation.  The
// chain is therefore cut at the BatchNorms, and each kernel
//     (a) applies the PREVIOUS layer's BN affine + LeakyReLU while staging its A operand (never materialised), and
//     (b) emits Σ / Σ² of its OWN output in the epilogue (double-precision atomics, one per column per CTA),
// so a Linear→BN→act→Linear→BN chain costs one pass per Linear.  Backward mirrors it: the BN-backward transform
//     dH = γ·istd · (dV − mean(dV) − Ĥ·mean(dV·Ĥ)),   dV = dA · lrelu'(V)
// is applied on the fly while staging dH for the dgrad (dX = dH·W) and wgrad (dW = dHᵀ·A) contractions.
// Contractions run on mma.sync m16n8k8 tf32 with 3xTF32 error compensation (mma.cuh) – fp32-grade results.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "../../include/crfconv_b200.h"
#include "common.cuh"
#include "linear_args.cuh"
#include "mma.cuh"

namespace crf {
namespace lin {

constexpr int kThreads = 256;
constexpr int BM = 128;      // rows per CTA tile (fwd / dgrad)
constexpr int BK = 32;       // reduction chunk
constexpr int AS = BK + 4;   // smem row stride for [row][k] operands read as (g, t): bank = 4g + t

// ------------------------------------------------------------------------------------------ forward


template <int BN, bool X3>
__global__ void __launch_bounds__(kThreads) fwd_kernel(const FwdArgs a) {
    __shared__ __align__(16) float As[BM][AS];
    __shared__ __align__(16) float Ws[BN][AS];
    // per-warp partial Σ / Σ² (no shared-memory atomics: the statistics, and with them every LeakyReLU branch decision
    // downstream, are bit-reproducible from run to run as long as at most kStatSlots row tiles exist)
    __shared__ float s_part[kThreads / 32][2][BN];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int Ktot = a.C1 + a.C2;

    float acc[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

    const int c4 = tid & 7;          // float4 column slot inside the 32-wide chunk
    const int r0 = tid >> 3;         // 0..31

    for (int seg = 0; seg < 2; ++seg) {
        const float* X = seg == 0 ? a.X1 : a.X2;
        const int C = seg == 0 ? a.C1 : a.C2;
        if (C == 0 || X == nullptr) continue;
        const int coloff = seg == 0 ? 0 : a.C1;
        const bool pro = (seg == 0) && a.scale1 != nullptr;
        const bool vecA = ((C & 3) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
        const bool vecW = ((Ktot & 3) == 0) && ((coloff & 3) == 0) && ((C & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.W) & 15) == 0);
        for (int kc = 0; kc < C; kc += BK) {
            const int k = kc + 4 * c4;
            float sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
            if (pro) {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (k + e < C) { sc[e] = __ldg(a.scale1 + k + e); sh[e] = __ldg(a.shift1 + k + e); }
            }
            // ---- stage A (4 rows per thread)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int r = r0 + 32 * j;
                const int64_t m = m0 + r;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (m < a.M && k < C) {
                    int64_t srow = m;
                    if (seg == 0 && a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
                    const float* p = X + srow * C + k;
                    if (vecA) {
                        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
                        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (k + e < C) v[e] = __ldg(p + e);
                    }
                    if (pro) {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (k + e < C) v[e] = lrelu(fmaf(v[e], sc[e], sh[e]), a.slope1);
                    }
                }
                *reinterpret_cast<float4*>(&As[r][4 * c4]) = make_float4(v[0], v[1], v[2], v[3]);
            }
            // ---- stage W: Ws[n][kk] = W[n0+n][coloff + kc + kk]
            for (int q = tid; q < BN * 8; q += kThreads) {
                const int n = q >> 3, kk = 4 * (q & 7);
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (n0 + n < a.Cout && kc + kk < C) {
                    const float* p = a.W + (int64_t)(n0 + n) * Ktot + coloff + kc + kk;
                    if (vecW) {
                        const float4 x = __ldg(reinterpret_cast<const float4*>(p));
                        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (kc + kk + e < C) v[e] = __ldg(p + e);
                    }
                }
                *reinterpret_cast<float4*>(&Ws[n][kk]) = make_float4(v[0], v[1], v[2], v[3]);
            }
            __syncthreads();
            // ---- tensor-core contraction of this chunk
            const int kmax = min(BK, C - kc);
#pragma unroll
            for (int ks = 0; ks < BK / 8; ++ks) {
                if (ks * 8 < kmax) {
                    const float af[4] = {As[16 * w + g][ks * 8 + t], As[16 * w + g + 8][ks * 8 + t],
                                         As[16 * w + g][ks * 8 + t + 4], As[16 * w + g + 8][ks * 8 + t + 4]};
                    FragA fa;
                    make_frag_a<X3>(fa, af);
#pragma unroll
                    for (int nt = 0; nt < BN / 8; ++nt) {
                        FragB fb;
                        make_frag_b<X3>(fb, Ws[nt * 8 + g][ks * 8 + t], Ws[nt * 8 + g][ks * 8 + t + 4]);
                        mma_frag<X3>(acc[nt], fa, fb);
                    }
                }
            }
            __syncthreads();
        }
    }

    // ---- epilogue: bias, store, column statistics
    const int64_t row_a = m0 + 16 * w + g, row_b = row_a + 8;
    const bool va = row_a < a.M, vb = row_b < a.M;
    const bool vec_st = (a.Cout & 1) == 0;
#pragma unroll
    for (int nt = 0; nt < BN / 8; ++nt) {
        const int col = n0 + nt * 8 + 2 * t;
        float c0 = acc[nt][0], c1 = acc[nt][1], c2 = acc[nt][2], c3 = acc[nt][3];
        if (a.bias) {
            const float b0 = col < a.Cout ? __ldg(a.bias + col) : 0.f, b1 = col + 1 < a.Cout ? __ldg(a.bias + col + 1) : 0.f;
            c0 += b0; c1 += b1; c2 += b0; c3 += b1;
        }
        if (vec_st && col + 1 < a.Cout) {
            if (va) *reinterpret_cast<float2*>(a.Y + row_a * a.Cout + col) = make_float2(c0, c1);
            if (vb) *reinterpret_cast<float2*>(a.Y + row_b * a.Cout + col) = make_float2(c2, c3);
        } else {
            if (va && col < a.Cout) a.Y[row_a * a.Cout + col] = c0;
            if (va && col + 1 < a.Cout) a.Y[row_a * a.Cout + col + 1] = c1;
            if (vb && col < a.Cout) a.Y[row_b * a.Cout + col] = c2;
            if (vb && col + 1 < a.Cout) a.Y[row_b * a.Cout + col + 1] = c3;
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
                s_part[w][0][nt * 8 + 2 * t] = s0; s_part[w][0][nt * 8 + 2 * t + 1] = s1;
                s_part[w][1][nt * 8 + 2 * t] = q0; s_part[w][1][nt * 8 + 2 * t + 1] = q1;
            }
        }
    }
    if (a.stats) {
        __syncthreads();
        if (tid < BN && n0 + tid < a.Cout) {
            float ssum = 0.f, ssq = 0.f;
#pragma unroll
            for (int ww = 0; ww < kThreads / 32; ++ww) { ssum += s_part[ww][0][tid]; ssq += s_part[ww][1][tid]; }
            float* st = a.stats + (size_t)(blockIdx.x % kStatSlots) * 2 * a.Cout;
            atomicAdd(st + n0 + tid, ssum);
            atomicAdd(st + a.Cout + n0 + tid, ssq);
        }
    }
}

// ------------------------------------------------------------------------------- BatchNorm bookkeeping
// Training: batch statistics from Σ / Σ² → scale/shift (+ saved mean / invstd, running-stat update with momentum and
// unbiased variance, exactly nn.BatchNorm1d).  Eval: scale/shift from the running statistics.
__global__ void __launch_bounds__(128) bn_finalize_fwd_kernel(const float* __restrict__ stats, double count, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float eps, float momentum, int training,
                                       float* running_mean, float* running_var, float* __restrict__ scale,
                                       float* __restrict__ shift, float* __restrict__ mean_out, float* __restrict__ invstd_out, int C) {
    // one CTA per channel: sums the kStatSlots partial (Σ, Σ²) pairs in a fixed order, then the BatchNorm bookkeeping
    __shared__ double r1[4], r2[4];
    const int c = blockIdx.x;
    double s1 = 0.0, s2 = 0.0;
    if (training) {
        for (int p = threadIdx.x; p < kStatSlots; p += blockDim.x) {
            s1 += (double)stats[(size_t)p * 2 * C + c];
            s2 += (double)stats[(size_t)p * 2 * C + C + c];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
        if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
        __syncthreads();
        s1 = r1[0] + r1[1] + r1[2] + r1[3];
        s2 = r2[0] + r2[1] + r2[2] + r2[3];
    }
    if (threadIdx.x != 0) return;
    float mean, invstd;
    if (training) {
        const double mu = s1 / count;
        double var = s2 / count - mu * mu;
        if (var < 0.0) var = 0.0;
        mean = (float)mu;
        invstd = (float)(1.0 / sqrt(var + (double)eps));
        if (running_mean) {
            const double unb = count > 1.0 ? var * count / (count - 1.0) : var;
            running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mu;
            running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)unb;
        }
    } else {
        mean = running_mean[c];
        invstd = 1.0f / sqrtf(running_var[c] + eps);
    }
    const float gm = gamma ? gamma[c] : 1.0f, bt = beta ? beta[c] : 0.0f;
    const float sc = gm * invstd;
    scale[c] = sc;
    shift[c] = bt - mean * sc;
    if (mean_out) mean_out[c] = mean;
    if (invstd_out) invstd_out[c] = invstd;
}

// Y = lrelu(H*scale + shift (+ R), slope).  C % 4 == 0.
__global__ void __launch_bounds__(256) bn_act_fwd_kernel(const float* __restrict__ H, const float* __restrict__ scale,
                                                         const float* __restrict__ shift, const float* __restrict__ R,
                                                         float slope, float* __restrict__ Y, int64_t total4, int C4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C4) * 4;
        const float4 h = __ldg(reinterpret_cast<const float4*>(H) + i);
        const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + c));
        const float4 sh = __ldg(reinterpret_cast<const float4*>(shift + c));
        float4 v = make_float4(fmaf(h.x, sc.x, sh.x), fmaf(h.y, sc.y, sh.y), fmaf(h.z, sc.z, sh.z), fmaf(h.w, sc.w, sh.w));
        if (R) {
            const float4 r = __ldg(reinterpret_cast<const float4*>(R) + i);
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        v.x = lrelu(v.x, slope); v.y = lrelu(v.y, slope); v.z = lrelu(v.z, slope); v.w = lrelu(v.w, slope);
        reinterpret_cast<float4*>(Y)[i] = v;
    }
}

// ------------------------------------------------------------------------------------------ backward

__device__ __forceinline__ float bn_dv(float dy, float h, float ref, bool has_ref, float sc, float sh, float slope) {
    const float pre = has_ref ? ref : fmaf(h, sc, sh);
    return pre > 0.0f ? dy : dy * slope;
}

// s1[c] = Σ_rows dV, s2[c] = Σ_rows dV·Ĥ (double atomics).  C % 4 == 0, C <= 1024.
// REF = false (activation selected by the recomputed pre-activation): 64 registers ⇒ 4 CTAs per SM; with 3 (84 registers) ncu showed
// 15 resident warps on average and the two input streams at 3.3 TB/s — not enough loads in flight.
template <bool REF>
__global__ void __launch_bounds__(256, REF ? 3 : 4) bn_bwd_reduce_kernel(const float* __restrict__ dY, const float* __restrict__ H, BnBwd bn,
                                                            float* __restrict__ sums, int64_t M, int C, const cl::BwdFin fin) {
    __shared__ float red[256 * 8];
    const int C4 = C >> 2;
    const int tpr = C4;                           // threads per row
    const int rows_per_it = 256 / tpr;            // C4 divides 256 for C in {8,...,1024}
    const int tid = threadIdx.x;
    const int cslot = tid % tpr, rslot = tid / tpr;
    float s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    if (rslot < rows_per_it) {
        const int c = cslot * 4;
        const float4 sc = __ldg(reinterpret_cast<const float4*>(bn.scale + c)), sh = __ldg(reinterpret_cast<const float4*>(bn.shift + c));
        const float4 mu = __ldg(reinterpret_cast<const float4*>(bn.mean + c)), is = __ldg(reinterpret_cast<const float4*>(bn.invstd + c));
        constexpr bool has_ref = REF;
        // 4 rows per thread per trip: 8-12 independent 128-bit loads in flight per thread (the kernel is pure streaming)
        constexpr int U = 4;
        const int64_t stride = (int64_t)gridDim.x * rows_per_it;
        for (int64_t m0 = (int64_t)blockIdx.x * rows_per_it + rslot; m0 < M; m0 += U * stride) {
            float4 dy[U], h[U], rf[REF ? U : 1];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t m = m0 + u * stride;
                if (m < M) {
                    dy[u] = __ldg(reinterpret_cast<const float4*>(dY + m * C + c));
                    h[u] = __ldg(reinterpret_cast<const float4*>(H + m * C + c));
                    if (REF) rf[u] = __ldg(reinterpret_cast<const float4*>(bn.act_ref + m * C + c));
                } else {
                    dy[u] = make_float4(0, 0, 0, 0); h[u] = mu;
                    if (REF) rf[u] = make_float4(0, 0, 0, 0);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float4 r = rf[REF ? u : 0];
                const float d0 = bn_dv(dy[u].x, h[u].x, r.x, has_ref, sc.x, sh.x, bn.slope), d1 = bn_dv(dy[u].y, h[u].y, r.y, has_ref, sc.y, sh.y, bn.slope);
                const float d2 = bn_dv(dy[u].z, h[u].z, r.z, has_ref, sc.z, sh.z, bn.slope), d3 = bn_dv(dy[u].w, h[u].w, r.w, has_ref, sc.w, sh.w, bn.slope);
                s1[0] += d0; s1[1] += d1; s1[2] += d2; s1[3] += d3;
                s2[0] += d0 * (h[u].x - mu.x) * is.x; s2[1] += d1 * (h[u].y - mu.y) * is.y;
                s2[2] += d2 * (h[u].z - mu.z) * is.z; s2[3] += d3 * (h[u].w - mu.w) * is.w;
            }
        }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) { red[tid * 8 + e] = s1[e]; red[tid * 8 + 4 + e] = s2[e]; }
    __syncthreads();
    // thread j < tpr*8 owns (column slot, which of 8 values); sums over the row slots
    for (int j = tid; j < tpr * 8; j += 256) {
        const int cs = j / 8, e = j % 8;
        float tot = 0.0f;
        for (int r = 0; r < rows_per_it; ++r) tot += red[(r * tpr + cs) * 8 + e];
        const int c = cs * 4 + (e & 3);
        atomicAdd(sums + (size_t)(blockIdx.x % (fin.part ? 32 : kStatSlots)) * 2 * C + (e < 4 ? 0 : C) + c, tot);
    }
    if (fin.part) {                                               // k1 / k2 / dγ / dβ by the last CTA (C <= 128, checked by the launcher)
        __shared__ double s_red[256];
        if (!cl::arrive_is_last(fin.counter)) return;
        if (tid < 2 * C) {
            double acc = 0.0;
            for (int p = 0; p < 32; ++p) acc += (double)__ldcg(fin.part + (size_t)p * 2 * C + tid);
            s_red[tid] = acc;
        }
        __syncthreads();
        if (tid < C) cl::bn_bwd_finalize(fin, s_red[tid], s_red[C + tid], tid);
    }
}

// k1 = s1/M, k2 = s2/M; dγ += s2, dβ += s1.
__global__ void __launch_bounds__(128) bn_finalize_bwd_kernel(const float* __restrict__ sums, double count, float* __restrict__ k1, float* __restrict__ k2,
                                       float* dgamma, float* dbeta, int C) {
    __shared__ double r1[4], r2[4];
    const int c = blockIdx.x;
    double s1 = 0.0, s2 = 0.0;
    for (int p = threadIdx.x; p < kStatSlots; p += blockDim.x) {
        s1 += (double)sums[(size_t)p * 2 * C + c];
        s2 += (double)sums[(size_t)p * 2 * C + C + c];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
    __syncthreads();
    if (threadIdx.x != 0) return;
    s1 = r1[0] + r1[1] + r1[2] + r1[3];
    s2 = r2[0] + r2[1] + r2[2] + r2[3];
    k1[c] = (float)(s1 / count);
    k2[c] = (float)(s2 / count);
    if (dgamma) dgamma[c] += (float)s2;
    if (dbeta) dbeta[c] += (float)s1;
}

// dW[i] += Σ_slots scratch[slot][i]   (fixed order ⇒ deterministic for a given launch configuration)
__global__ void __launch_bounds__(256) grad_slots_reduce_kernel(const float* __restrict__ scratch, float* dW, int n, int64_t stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
#pragma unroll 8
    for (int p = 0; p < kGradSlots; ++p) s += scratch[(size_t)p * stride + i];
    dW[i] += s;
}

// dH for 4 consecutive channels starting at c (c % 4 == 0, c + 3 < C).
__device__ __forceinline__ void load_dh4(const float* __restrict__ dY, const float* __restrict__ H, const BnBwd& bn, int64_t m, int C,
                                         int c, float (&out)[4]) {
    const float4 dy = __ldg(reinterpret_cast<const float4*>(dY + m * C + c));
    if (bn.scale == nullptr) { out[0] = dy.x; out[1] = dy.y; out[2] = dy.z; out[3] = dy.w; return; }
    const float4 h = __ldg(reinterpret_cast<const float4*>(H + m * C + c));
    const bool has_ref = bn.act_ref != nullptr;
    float4 rf = make_float4(0, 0, 0, 0);
    if (has_ref) rf = __ldg(reinterpret_cast<const float4*>(bn.act_ref + m * C + c));
    const float4 sc = __ldg(reinterpret_cast<const float4*>(bn.scale + c)), sh = __ldg(reinterpret_cast<const float4*>(bn.shift + c));
    const float4 mu = __ldg(reinterpret_cast<const float4*>(bn.mean + c)), is = __ldg(reinterpret_cast<const float4*>(bn.invstd + c));
    const float4 k1 = __ldg(reinterpret_cast<const float4*>(bn.k1 + c)), k2 = __ldg(reinterpret_cast<const float4*>(bn.k2 + c));
    out[0] = sc.x * (bn_dv(dy.x, h.x, rf.x, has_ref, sc.x, sh.x, bn.slope) - k1.x - (h.x - mu.x) * is.x * k2.x);
    out[1] = sc.y * (bn_dv(dy.y, h.y, rf.y, has_ref, sc.y, sh.y, bn.slope) - k1.y - (h.y - mu.y) * is.y * k2.y);
    out[2] = sc.z * (bn_dv(dy.z, h.z, rf.z, has_ref, sc.z, sh.z, bn.slope) - k1.z - (h.z - mu.z) * is.z * k2.z);
    out[3] = sc.w * (bn_dv(dy.w, h.w, rf.w, has_ref, sc.w, sh.w, bn.slope) - k1.w - (h.w - mu.w) * is.w * k2.w);
}

// scalar variant for Cout % 4 != 0 (plain Linear only, e.g. the 13-class head)
__device__ __forceinline__ float load_dh1(const float* __restrict__ dY, int64_t m, int C, int c) { return __ldg(dY + m * C + c); }



constexpr int BS8 = 8;   // extra stride so that [k][n] operands read as (t, g) hit bank 8t + g

template <int BN, bool X3>
__global__ void __launch_bounds__(kThreads) dgrad_kernel(const DgradArgs a) {
    __shared__ __align__(16) float As[BM][AS];           // dH tile [row][cout chunk]
    __shared__ __align__(16) float Ws[BK][BN + BS8];     // W chunk [cout][cin tile]
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;                      // input-channel tile
    const int Ktot = a.C1 + a.C2;
    const int C = a.Cout;
    const bool vecA = (C & 3) == 0;
    const bool vecW = ((Ktot & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.W) & 15) == 0);

    float acc[BN / 8][4];
#pragma unroll
    for (int i = 0; i < BN / 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    const int c4 = tid & 7, r0 = tid >> 3;

    for (int kc = 0; kc < C; kc += BK) {
        const int k = kc + 4 * c4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = r0 + 32 * j;
            const int64_t m = m0 + r;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (m < a.M && k < C) {
                if (vecA) load_dh4(a.dY, a.H, a.bn, m, C, k, v);
                else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (k + e < C) v[e] = load_dh1(a.dY, m, C, k + e);
                }
            }
            *reinterpret_cast<float4*>(&As[r][4 * c4]) = make_float4(v[0], v[1], v[2], v[3]);
        }
        // Ws[kk][n] = W[kc+kk][n0+n]
        for (int q = tid; q < BK * (BN / 4); q += kThreads) {
            const int kk = q / (BN / 4), n = 4 * (q % (BN / 4));
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (kc + kk < C && n0 + n < Ktot) {
                const float* p = a.W + (int64_t)(kc + kk) * Ktot + n0 + n;
                if (vecW) {
                    const float4 x = __ldg(reinterpret_cast<const float4*>(p));
                    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (n0 + n + e < Ktot) v[e] = __ldg(p + e);
                }
            }
            *reinterpret_cast<float4*>(&Ws[kk][n]) = make_float4(v[0], v[1], v[2], v[3]);
        }
        __syncthreads();
        const int kmax = min(BK, C - kc);
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            if (ks * 8 < kmax) {
                const float af[4] = {As[16 * w + g][ks * 8 + t], As[16 * w + g + 8][ks * 8 + t],
                                     As[16 * w + g][ks * 8 + t + 4], As[16 * w + g + 8][ks * 8 + t + 4]};
                FragA fa;
                make_frag_a<X3>(fa, af);
#pragma unroll
                for (int nt = 0; nt < BN / 8; ++nt) {
                    FragB fb;
                    make_frag_b<X3>(fb, Ws[ks * 8 + t][nt * 8 + g], Ws[ks * 8 + t + 4][nt * 8 + g]);
                    mma_frag<X3>(acc[nt], fa, fb);
                }
            }
        }
        __syncthreads();
    }
    const int64_t row_a = m0 + 16 * w + g, row_b = row_a + 8;
    const bool va = row_a < a.M, vb = row_b < a.M;
#pragma unroll
    for (int nt = 0; nt < BN / 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int col = n0 + nt * 8 + 2 * t + e;
            if (col >= Ktot) continue;
            float* dst; int cc, ld, accm;
            if (col < a.C1) { dst = a.dX1; cc = col; ld = a.C1; accm = a.acc1; }
            else            { dst = a.dX2; cc = col - a.C1; ld = a.C2; accm = a.acc2; }
            if (!dst) continue;
            if (va) { float* p = dst + row_a * ld + cc; *p = accm ? *p + acc[nt][e] : acc[nt][e]; }
            if (vb) { float* p = dst + row_b * ld + cc; *p = accm ? *p + acc[nt][2 + e] : acc[nt][2 + e]; }
        }
    }
}

// ---- weight gradient for very narrow inputs (Ktot <= 4: the 3-d relative positions feeding PointConv's edge MLP,
// point_conv_big.py:37-44).  dW is Cout × 3 while the contraction runs over millions of edges: the tiled kernel below spends its
// time in atomics onto a few dozen addresses (measured 2.1 ms per call at 3.9 M edges, 44 % of the full network's step).  Here one
// thread owns a 4-channel slice of a row, keeps its 4 × Ktot partial sums in registers over all its rows, and the CTA folds them
// through shared memory into one partial slot.  Pure streaming: rows × (2·Cout + Ktot) × 4 bytes.
template <int KT>
__global__ void __launch_bounds__(256) wgrad_tiny_kernel(const WgradArgs a) {
    __shared__ float red[256 * 4 * KT];
    const int C = a.Cout, C4 = C >> 2;
    const int rows_per_it = 256 / C4;                // C4 divides 256 for Cout in {4, 8, ..., 1024}
    const int tid = threadIdx.x;
    const int cslot = tid % C4, rslot = tid / C4;
    const bool plain = a.bn.scale == nullptr;
    const bool has_ref = !plain && a.bn.act_ref != nullptr;
    float acc[4][KT];
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int k = 0; k < KT; ++k) acc[e][k] = 0.f;
    if (rslot < rows_per_it) {
        const int c = cslot * 4;
        float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f), pz = sh, pw = sh;
        if (!plain) {
            sc = __ldg(reinterpret_cast<const float4*>(a.bn.scale + c)); sh = __ldg(reinterpret_cast<const float4*>(a.bn.shift + c));
            const float4 mu = __ldg(reinterpret_cast<const float4*>(a.bn.mean + c)), is = __ldg(reinterpret_cast<const float4*>(a.bn.invstd + c));
            const float4 k1 = __ldg(reinterpret_cast<const float4*>(a.bn.k1 + c)), k2 = __ldg(reinterpret_cast<const float4*>(a.bn.k2 + c));
            pz = make_float4(-sc.x * is.x * k2.x, -sc.y * is.y * k2.y, -sc.z * is.z * k2.z, -sc.w * is.w * k2.w);
            pw = make_float4(-sc.x * k1.x - pz.x * mu.x, -sc.y * k1.y - pz.y * mu.y, -sc.z * k1.z - pz.z * mu.z, -sc.w * k1.w - pz.w * mu.w);
        }
        float xs[KT], xh[KT];
#pragma unroll
        for (int k = 0; k < KT; ++k) {
            xs[k] = (a.scale1 && k < a.C1) ? __ldg(a.scale1 + k) : 1.f;
            xh[k] = (a.scale1 && k < a.C1) ? __ldg(a.shift1 + k) : 0.f;
        }
        const float slope = a.bn.slope, slope1 = a.scale1 ? a.slope1 : 1.f;
        constexpr int U = 4;
        const int64_t stride = (int64_t)gridDim.x * rows_per_it;
        for (int64_t m0 = (int64_t)blockIdx.x * rows_per_it + rslot; m0 < a.M; m0 += U * stride) {
            float4 dy[U], h[U], rf[U];
            float x[U][KT];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t m = m0 + u * stride;
                const bool ok = m < a.M;
                const int64_t off = ok ? m * C + c : 0;
                dy[u] = ok ? __ldg(reinterpret_cast<const float4*>(a.dY + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                h[u] = (ok && !plain) ? __ldg(reinterpret_cast<const float4*>(a.H + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                rf[u] = (ok && has_ref) ? __ldg(reinterpret_cast<const float4*>(a.bn.act_ref + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
                int64_t srow = ok ? m : 0;
                if (ok && a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
#pragma unroll
                for (int k = 0; k < KT; ++k) x[u][k] = (ok && k < a.C1) ? __ldg(a.X1 + srow * a.C1 + k) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool ok = m0 + u * stride < a.M;
                float d[4] = {dy[u].x, dy[u].y, dy[u].z, dy[u].w};
                if (!plain) {
                    d[0] = fmaf(sc.x, bn_dv(dy[u].x, h[u].x, rf[u].x, has_ref, sc.x, sh.x, slope), fmaf(pz.x, h[u].x, pw.x));
                    d[1] = fmaf(sc.y, bn_dv(dy[u].y, h[u].y, rf[u].y, has_ref, sc.y, sh.y, slope), fmaf(pz.y, h[u].y, pw.y));
                    d[2] = fmaf(sc.z, bn_dv(dy[u].z, h[u].z, rf[u].z, has_ref, sc.z, sh.z, slope), fmaf(pz.z, h[u].z, pw.z));
                    d[3] = fmaf(sc.w, bn_dv(dy[u].w, h[u].w, rf[u].w, has_ref, sc.w, sh.w, slope), fmaf(pz.w, h[u].w, pw.w));
                }
#pragma unroll
                for (int k = 0; k < KT; ++k) {
                    float xv = fmaf(x[u][k], xs[k], xh[k]);
                    xv = xv > 0.f ? xv : xv * slope1;
                    xv = (ok && k < a.C1) ? xv : 0.f;          // padding rows contribute nothing (their dH is not zero under BN)
#pragma unroll
                    for (int e = 0; e < 4; ++e) acc[e][k] = fmaf(d[e], xv, acc[e][k]);
                }
            }
        }
    }
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int k = 0; k < KT; ++k) red[(tid * 4 + e) * KT + k] = acc[e][k];
    __syncthreads();
    for (int j = tid; j < C4 * 4 * KT; j += 256) {               // (channel slot, e, k) summed over the row slots
        const int cs = j / (4 * KT), ek = j % (4 * KT);
        float tot = 0.f;
        for (int r = 0; r < rows_per_it; ++r) tot += red[((r * C4 + cs) * 4) * KT + ek];
        const int co = cs * 4 + ek / KT, k = ek % KT;
        if (k < a.C1) atomicAdd(a.dW + a.slot_stride * (int64_t)(blockIdx.x % kGradSlots) + (int64_t)co * a.C1 + k, tot);
    }
}

inline int try_wgrad_tiny(const WgradArgs& a, cudaStream_t st) {
    if (a.C2 != 0 || a.C1 < 1 || a.C1 > 4 || a.dbias || (a.Cout & 3) || a.Cout > 1024 || (256 % (a.Cout >> 2)) != 0) return kDeclined;
    if (!aligned16(a.dY) || (a.bn.scale && !aligned16(a.H))) return kDeclined;
    if (a.bn.scale && a.bn.act_ref && !aligned16(a.bn.act_ref)) return kDeclined;
    const int rows_per_it = 256 / (a.Cout >> 2);
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(a.M, (int64_t)rows_per_it * 4), (int64_t)kNumSMs * 8);
    return launch(wgrad_tiny_kernel<4>, dim3(grid), dim3(256), 0, st, a);
}

// dW[co, k] += Σ_m dH[m, co] · A[m, k],  A = [prologue(X1) | X2].  Output tile 64 (co) × 64 (k) per CTA; CTAs along
// x split the rows; partial tiles are combined with fp32 atomics.


constexpr int WR = 64;          // rows per staging tile
constexpr int WS = 64 + BS8;    // smem stride

template <bool X3>
__global__ void __launch_bounds__(kThreads) wgrad_kernel(const WgradArgs a) {
    __shared__ __align__(16) float Ds[WR][WS];   // dH tile  [m][co]
    __shared__ __align__(16) float Xs[WR][WS];   // A tile   [m][k]
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
    const int Ktot = a.C1 + a.C2;
    const int co0 = blockIdx.y * 64, k0 = blockIdx.z * 64;
    const int64_t mbeg = (int64_t)blockIdx.x * a.rows_per_cta, mend = min(a.M, mbeg + a.rows_per_cta);
    const int wr = (w & 3) * 16;       // co rows of this warp inside the tile
    const int wc = (w >> 2) * 32;      // k cols of this warp inside the tile
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    float bsum = 0.0f;                 // bias gradient: thread tid<64 owns column co0+tid
    const bool vecD = (a.Cout & 3) == 0;
    const int c16 = tid & 15, rr = tid >> 4;   // 16 float4 per 64-wide row, 16 rows per pass

    for (int64_t mt = mbeg; mt < mend; mt += WR) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = rr + 16 * j;
            const int64_t m = mt + r;
            // dH tile
            {
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                const int c = co0 + 4 * c16;
                if (m < mend && c < a.Cout) {
                    if (vecD) load_dh4(a.dY, a.H, a.bn, m, a.Cout, c, v);
                    else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (c + e < a.Cout) v[e] = load_dh1(a.dY, m, a.Cout, c + e);
                    }
                }
                *reinterpret_cast<float4*>(&Ds[r][4 * c16]) = make_float4(v[0], v[1], v[2], v[3]);
            }
            // A tile (global column k0 + 4*c16 .. +3; may straddle nothing: C1 % 4 == 0 or scalar path)
            {
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                const int kg = k0 + 4 * c16;
                if (m < mend && kg < Ktot) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int kk = kg + e;
                        if (kk >= Ktot) break;
                        if (kk < a.C1) {
                            int64_t srow = m;
                            if (a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
                            float x = __ldg(a.X1 + srow * a.C1 + kk);
                            if (a.scale1) x = lrelu(fmaf(x, __ldg(a.scale1 + kk), __ldg(a.shift1 + kk)), a.slope1);
                            v[e] = x;
                        } else {
                            v[e] = __ldg(a.X2 + m * a.C2 + (kk - a.C1));
                        }
                    }
                }
                *reinterpret_cast<float4*>(&Xs[r][4 * c16]) = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
        __syncthreads();
        if (a.dbias && blockIdx.z == 0 && tid < 64) {
            float s = 0.0f;
            for (int r = 0; r < WR; ++r) s += Ds[r][tid];
            bsum += s;
        }
#pragma unroll
        for (int ks = 0; ks < WR / 8; ++ks) {
            // A operand = dHᵀ: (row = co, col = m)
            const float af[4] = {Ds[ks * 8 + t][wr + g], Ds[ks * 8 + t][wr + g + 8], Ds[ks * 8 + t + 4][wr + g], Ds[ks * 8 + t + 4][wr + g + 8]};
            FragA fa;
            make_frag_a<X3>(fa, af);
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                FragB fb;
                make_frag_b<X3>(fb, Xs[ks * 8 + t][wc + nt * 8 + g], Xs[ks * 8 + t + 4][wc + nt * 8 + g]);
                mma_frag<X3>(acc[nt], fa, fb);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int co = co0 + wr + g + (e >= 2 ? 8 : 0);
            const int k = k0 + wc + nt * 8 + 2 * t + (e & 1);
            if (co < a.Cout && k < Ktot) atomicAdd(a.dW + a.slot_stride * (blockIdx.x % kGradSlots) + (int64_t)co * Ktot + k, acc[nt][e]);
        }
    }
    if (a.dbias && blockIdx.z == 0 && tid < 64 && co0 + tid < a.Cout) atomicAdd(a.dbias + co0 + tid, bsum);
}

// The bf16x3 fast path (≈2^-17 per product) is used from this many rows on; smaller problems are launch-bound anyway and
// take the generic 3xTF32 kernels (≈2^-21), which keeps ill-conditioned tiny batches inside the 1e-3 parity budget.
// Dispatch between the kernel families is by SHAPE only (no environment switches); the one override is the tests' hook below.
constexpr int64_t kFastMinRows = 8192;
static thread_local int t_bwd_launches = 0;   // kernels launched by this thread's last crfconv_linear_bwd call
static int g_fast_override = -1;   // -1: rule above; 0: never; 1: always (crfconv_set_fast_path: lets the tests reach every family at small sizes)
inline bool use_fast(int64_t M) {
    if (g_fast_override >= 0) return g_fast_override == 1;
    return M >= kFastMinRows;
}

template <typename F>
inline int dispatch_bn(int n, F&& f) {
    if (n > 32) return f(std::integral_constant<int, 64>{});
    if (n > 16) return f(std::integral_constant<int, 32>{});
    if (n > 8) return f(std::integral_constant<int, 16>{});
    return f(std::integral_constant<int, 8>{});
}

// The generic kernels take every shape: x3 = 3xTF32, else single-pass TF32.
inline int fwd_generic(const FwdArgs& a, bool x3, cudaStream_t st) {
    return dispatch_bn(a.Cout, [&](auto bn) {
        constexpr int BN = decltype(bn)::value;
        const dim3 grid((unsigned)ceil_div(a.M, BM), (unsigned)ceil_div(a.Cout, BN));
        return launch(x3 ? fwd_kernel<BN, true> : fwd_kernel<BN, false>, grid, dim3(kThreads), 0, st, a);
    });
}

inline int dgrad_generic(const DgradArgs& a, bool x3, cudaStream_t st) {
    const int Ktot = a.C1 + a.C2;
    return dispatch_bn(Ktot, [&](auto bn) {
        constexpr int BN = decltype(bn)::value;
        const dim3 grid((unsigned)ceil_div(a.M, BM), (unsigned)ceil_div(Ktot, BN));
        return launch(x3 ? dgrad_kernel<BN, true> : dgrad_kernel<BN, false>, grid, dim3(kThreads), 0, st, a);
    });
}

inline int wgrad_generic(WgradArgs a, bool x3, cudaStream_t st) {
    const int ty = (int)ceil_div(a.Cout, 64), tz = (int)ceil_div(a.C1 + a.C2, 64);
    int64_t splits = std::max<int64_t>(1, std::min<int64_t>(ceil_div(a.M, 256), (int64_t)(2 * kNumSMs) / (ty * tz) + 1));
    a.rows_per_cta = ceil_div(ceil_div(a.M, splits), WR) * WR;
    splits = ceil_div(a.M, a.rows_per_cta);
    const dim3 grid((unsigned)splits, (unsigned)ty, (unsigned)tz);
    return launch(x3 ? wgrad_kernel<true> : wgrad_kernel<false>, grid, dim3(kThreads), 0, st, a);
}

}  // namespace lin
}  // namespace crf

using namespace crf;

extern "C" {

// Test hook: -1 = default rule (fast bf16x3 kernels from 8,192 rows on), 0 = generic kernels
// only, 1 = fast kernels whenever the shape allows.  Returns the previous setting.
int crfconv_set_fast_path(int mode) {
    const int prev = lin::g_fast_override;
    lin::g_fast_override = mode < 0 ? -1 : (mode ? 1 : 0);
    return prev;
}

// Y[M,Cout] = [lrelu(X1*scale1+shift1) | X2] · Wᵀ (+ bias);  stats[0:Cout] += Σ_rows Y, stats[Cout:2Cout] += Σ_rows Y².
// X1 rows may be gathered: source row of output row m = (m / rows_dst) * rows_src + idx1[m]   (idx1 null ⇒ identity).
// precision: 0 = 3xTF32 (fp32-grade), 1 = single-pass TF32, 2 = single-pass bf16 where the persistent kernels take the shape
// (single-pass TF32 elsewhere).  Families in the order of DESIGN.md §4.3; the first that takes the call launches one kernel.
int crfconv_linear_fwd(const float* X1, int C1, const float* scale1, const float* shift1, float slope1, const int64_t* idx1,
                       int64_t rows_dst, int64_t rows_src, const float* X2, int C2, const float* W, const float* bias, float* Y,
                       float* stats, int64_t M, int Cout, int precision, void* stream) {
    if (M < 0 || Cout <= 0 || C1 < 0 || C2 < 0 || C1 + C2 <= 0 || precision < 0 || precision > 2) return CRF_ERR_INVALID_ARG;
    if (M == 0) return CRF_OK;
    if ((C1 > 0 && !X1) || (C2 > 0 && !X2) || !W || !Y) return CRF_ERR_INVALID_ARG;
    if (idx1 && (rows_dst <= 0 || rows_src <= 0)) return CRF_ERR_INVALID_ARG;
    const lin::FwdArgs a{X1, C1, scale1, shift1, slope1, idx1, rows_dst, rows_src, X2, C2, W, bias, Y, stats, M, Cout};
    cudaStream_t st = (cudaStream_t)stream;
    const bool fast = lin::use_fast(M), x3 = precision == 0;
    int rc = lin::kDeclined;
    if (rc == lin::kDeclined && fast) rc = lin::try_fwd3(a, precision, st);      // tcgen05: also faster than the CUDA-core kernel for 16→16 (17 vs 24 us)
    if (rc == lin::kDeclined && fast) rc = lin::try_narrow_fwd(a, st);
    if (rc == lin::kDeclined && fast) rc = lin::try_fwd2(a, precision, st);
    if (rc == lin::kDeclined && x3) rc = lin::try_fwd_small(a, st);
    if (rc == lin::kDeclined && x3) rc = lin::try_upproj_fwd(a, st);
    if (rc == lin::kDeclined) rc = lin::fwd_generic(a, x3, st);
    return rc;
}

int crfconv_bn_finalize_fwd(const float* stats, int64_t count, const float* gamma, const float* beta, float eps, float momentum,
                            int training, float* running_mean, float* running_var, float* scale, float* shift, float* mean,
                            float* invstd, int C, void* stream) {
    if (C <= 0 || !scale || !shift || (training && !stats) || (!training && (!running_mean || !running_var))) return CRF_ERR_INVALID_ARG;
    lin::bn_finalize_fwd_kernel<<<(unsigned)C, 128, 0, (cudaStream_t)stream>>>(
        stats, (double)count, gamma, beta, eps, momentum, training, running_mean, running_var, scale, shift, mean, invstd, C);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// Y = lrelu(H*scale + shift (+ R), slope)
int crfconv_bn_act_fwd(const float* H, const float* scale, const float* shift, const float* R, float slope, float* Y, int64_t M,
                       int C, void* stream) {
    if (M < 0 || C <= 0 || (C & 3)) return CRF_ERR_INVALID_ARG;
    if (M == 0) return CRF_OK;
    const int64_t total4 = M * (C / 4);
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(total4, 256), (int64_t)kNumSMs * 16);
    lin::bn_act_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(H, scale, shift, R, slope, Y, total4, C / 4);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// sums[0:C] += Σ dV, sums[C:2C] += Σ dV·Ĥ with dV = dY·lrelu'(pre), pre = act_ref ? act_ref : H*scale+shift.
int crfconv_bn_bwd_reduce(const float* dY, const float* H, const float* act_ref, const float* scale, const float* shift,
                          const float* mean, const float* invstd, float slope, float* sums, int64_t M, int C, void* stream) {
    if (M < 0 || C <= 0 || (C & 3) || C > 1024 || (256 % (C / 4)) != 0) return CRF_ERR_UNSUPPORTED;
    if (M == 0) return CRF_OK;
    lin::BnBwd bn{scale, shift, mean, invstd, nullptr, nullptr, act_ref, slope};
    const int rows_per_it = 256 / (C / 4);
    constexpr int mult = 8;                                    // CTAs per SM: measured best of 2 / 4 / 8 / 16 (profiles/README_r02.md)
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(M, rows_per_it * 8), (int64_t)kNumSMs * mult);
    if (act_ref) lin::bn_bwd_reduce_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(dY, H, bn, sums, M, C, cl::BwdFin{});
    else lin::bn_bwd_reduce_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(dY, H, bn, sums, M, C, cl::BwdFin{});
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

int crfconv_bn_finalize_bwd(const float* sums, int64_t count, float* k1, float* k2, float* dgamma, float* dbeta, int C, void* stream) {
    if (C <= 0 || !sums || !k1 || !k2) return CRF_ERR_INVALID_ARG;
    lin::bn_finalize_bwd_kernel<<<(unsigned)C, 128, 0, (cudaStream_t)stream>>>(sums, (double)count, k1, k2, dgamma, dbeta, C);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// dW[i] += Σ_slots scratch[slot·stride + i], i < n  — one call can fold the partial slots of many layers that share a flat layout.
int crfconv_grad_slots_reduce(const float* scratch, float* dW, int64_t n, int64_t stride, void* stream) {
    if (n < 0 || !scratch || !dW || stride < n) return CRF_ERR_INVALID_ARG;
    if (n == 0) return CRF_OK;
    lin::grad_slots_reduce_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(scratch, dW, (int)n, stride);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

int crfconv_linear_bwd_launches(void) { return lin::t_bwd_launches; }

// Gradient of crfconv_linear_fwd wrt its (post-prologue) inputs and its weight.  The upstream gradient is given wrt the
// layer's ACTIVATION output (dY); the BN(+LeakyReLU) backward transform is applied on the fly (scale == NULL ⇒ the layer
// had no BN: dH = dY).   dX1 / dX2 may be NULL (not needed); acc ⇒ accumulate into the destination.  With idx1, dX1 is the
// gradient wrt the GATHERED rows [M, C1]; scatter it with crfconv_scatter_add_rows.
// Families in the order of DESIGN.md §4.3: a one-pass kernel for both gradients, else one kernel per requested gradient.
int crfconv_linear_bwd(const float* dY, const float* H, const float* act_ref, const float* scale, const float* shift,
                       const float* mean, const float* invstd, const float* k1, const float* k2, float slope,
                       const float* X1, int C1, const float* scale1, const float* shift1, float slope1, const int64_t* idx1,
                       int64_t rows_dst, int64_t rows_src, const float* X2, int C2, const float* W, float* dX1, int acc1,
                       float* dX2, int acc2, float* dW, float* dbias, float* dW_scratch, int64_t dW_scratch_stride, int64_t M, int Cout, int precision,
                       void* stream) {
    int& launches = lin::t_bwd_launches;
    launches = 0;
    if (M < 0 || Cout <= 0 || C1 < 0 || C2 < 0 || C1 + C2 <= 0 || !dY || !W || precision < 0 || precision > 2) return CRF_ERR_INVALID_ARG;
    if (M == 0) return CRF_OK;
    if (scale && (Cout & 3)) return CRF_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const bool fast = lin::use_fast(M), x3 = precision == 0;
    const int Ktot = C1 + C2;
    // weight-gradient partial slots: CTAs add into dW_scratch[slot] (zero-initialised by the caller), reduced into dW afterwards
    // here, or by the caller when it gives the slot stride (it reduces all its layers at once)
    const bool slots = dW && dW_scratch;
    const int64_t wstride = slots ? (dW_scratch_stride > 0 ? dW_scratch_stride : (int64_t)Cout * Ktot) : 0;
    const lin::BnBwd bn{scale, shift, mean, invstd, k1, k2, act_ref, slope};
    const lin::DgradArgs d{dY, H, bn, W, dX1, C1, acc1, dX2, C2, acc2, M, Cout};
    const lin::WgradArgs w{dY, H, bn, X1, C1, scale1, shift1, slope1, idx1, rows_dst, rows_src, X2, C2, slots ? dW_scratch : dW, dbias, M, Cout, 0, wstride};
    auto finish = [&](int rc) -> int {
        if (rc != CRF_OK || !slots || dW_scratch_stride > 0) return rc;
        ++launches;
        return lin::launch(lin::grad_slots_reduce_kernel, dim3((unsigned)ceil_div((int64_t)Cout * Ktot, 256)), dim3(256), 0, st,
                                  dW_scratch, dW, Cout * Ktot, (int64_t)Cout * Ktot);
    };

    int rc = lin::kDeclined;                                                      // input and weight gradient in one kernel
    if (rc == lin::kDeclined && fast) rc = lin::try_bwd3(d, w, precision, st);
    if (rc == lin::kDeclined && fast) rc = lin::try_narrow_bwd(d, dW ? &w : nullptr, st);
    if (rc != lin::kDeclined) {
        ++launches;
        return finish(rc);
    }
    if (dX1 || dX2) {                                                             // input gradient
        if (rc == lin::kDeclined && fast) rc = lin::try_dgrad3(d, precision, st);
        if (rc == lin::kDeclined && fast) rc = lin::try_dgrad2(d, precision, st);
        if (rc == lin::kDeclined && x3) rc = lin::try_dgrad_small(d, st);
        if (rc == lin::kDeclined && x3) rc = lin::try_upproj_dgrad(d, st);
        if (rc == lin::kDeclined) rc = lin::dgrad_generic(d, x3, st);
        ++launches;
        if (rc != CRF_OK) return rc;
    }
    if (!dW) return CRF_OK;
    rc = lin::kDeclined;                                                          // weight gradient
    if (rc == lin::kDeclined) rc = lin::try_wgrad_tiny(w, st);
    if (rc == lin::kDeclined && fast) rc = lin::try_wgrad3(w, precision, st);
    if (rc == lin::kDeclined && fast) rc = lin::try_wgrad2(w, precision, st);
    if (rc == lin::kDeclined && x3) rc = lin::try_wgrad_direct(w, st);
    if (rc == lin::kDeclined && x3) rc = lin::try_wgrad_rows(w, st);
    if (rc == lin::kDeclined) rc = lin::wgrad_generic(w, x3, st);
    ++launches;
    return finish(rc);
}

// crfconv_linear_fwd + training-mode BatchNorm finalize of its output (what crfconv_bn_finalize_fwd computes from `stats`), in ONE
// launch when the tcgen05 kernel takes the shape (the last CTA to finish folds the statistics slots), else in two.  stats is
// required ([CRFCONV_STAT_SLOTS][2·Cout], zeroed); counter = one zeroed uint32 (left zero).
int crfconv_linear_fwd_bn(const float* X1, int C1, const float* scale1, const float* shift1, float slope1, const float* X2, int C2,
                          const float* W, float* Y, float* stats, int64_t M, int Cout, int precision, unsigned int* counter,
                          const float* gamma, const float* beta, float* running_mean, float* running_var, float eps, float momentum,
                          float* scale, float* shift, float* mean, float* invstd, void* stream) {
    if (M <= 0 || Cout <= 0 || C1 <= 0 || C2 < 0 || !X1 || (C2 > 0 && !X2) || !W || !Y || !stats || !counter || !scale || !shift) return CRF_ERR_INVALID_ARG;
    if (precision < 0 || precision > 2) return CRF_ERR_INVALID_ARG;
    lin::FwdArgs a{X1, C1, scale1, shift1, slope1, nullptr, 0, 0, X2, C2, W, nullptr, Y, stats, M, Cout};
    a.fin = cl::FwdFin{stats, counter, gamma, beta, running_mean, running_var, eps, momentum, (double)M, scale, shift, mean, invstd};
    if (lin::use_fast(M)) {
        const int rc = lin::try_fwd3(a, precision, (cudaStream_t)stream);
        if (rc != lin::kDeclined) return rc;
    }
    const int rc = crfconv_linear_fwd(X1, C1, scale1, shift1, slope1, nullptr, 0, 0, X2, C2, W, nullptr, Y, stats, M, Cout, precision, stream);
    if (rc != CRF_OK) return rc;
    return crfconv_bn_finalize_fwd(stats, M, gamma, beta, eps, momentum, 1, running_mean, running_var, scale, shift, mean, invstd, Cout, stream);
}

// crfconv_bn_bwd_reduce + crfconv_bn_finalize_bwd in one launch (C == 64) or two.  sums: [CRFCONV_STAT_SLOTS][2·C] zeroed.
int crfconv_bn_bwd_reduce_fin(const float* dY, const float* H, const float* act_ref, const float* scale, const float* shift,
                              const float* mean, const float* invstd, float slope, float* sums, int64_t M, int C, unsigned int* counter,
                              float* k1, float* k2, float* dgamma, float* dbeta, void* stream) {
    if (!sums || !counter || !k1 || !k2) return CRF_ERR_INVALID_ARG;
    if (C > 128 || C < 4 || (C & 3) || (256 % (C / 4)) != 0 || M <= 0) {
        const int rc = crfconv_bn_bwd_reduce(dY, H, act_ref, scale, shift, mean, invstd, slope, sums, M, C, stream);
        if (rc != CRF_OK) return rc;
        return crfconv_bn_finalize_bwd(sums, M, k1, k2, dgamma, dbeta, C, stream);
    }
    lin::BnBwd bn{scale, shift, mean, invstd, nullptr, nullptr, act_ref, slope};
    const int rows_per_it = 256 / (C / 4);
    // exactly one resident wave: 3 (REF, 84 registers) or 4 (64 registers) CTAs per SM
    const cl::BwdFin fin{sums, counter, (double)M, k1, k2, dgamma, dbeta};
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(M, rows_per_it * 8), (int64_t)kNumSMs * (act_ref ? 3 : 4));   // <= cl::kMaxTicketGrid
    if (act_ref) lin::bn_bwd_reduce_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(dY, H, bn, sums, M, C, fin);
    else lin::bn_bwd_reduce_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(dY, H, bn, sums, M, C, fin);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

}  // extern "C"
