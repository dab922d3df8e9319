// CUDA-core kernels for the NARROW Linear layers of the hot path: everything whose input or output is a hidden-width
// tensor (min(Cin, Cout) <= 16: unary_nn / pairwise_nn / out_nn of the CRF layers, lin_in / lin_out / weight_nn of the
// ResNet blocks at the finest levels).  These layers move 10-100 MB but do < 1 GFLOP: on the tensor-core kernels they are
// bound by fragment conversion and per-tile synchronisation (ncu: issue-active ≈ 60 %, tensor pipe < 10 %), not by HBM.
// Here one thread owns one row: the row tile is staged with cp.async into shared memory (coalesced 128-bit copies), each
// thread streams its row from shared memory (conflict-free float4 reads, stride ≡ 4 mod 32) against a weight matrix that
// every lane reads at the same address (broadcast), and accumulates in exact fp32 FFMA — no tf32/bf16 rounding at all.
// 2-3 CTAs per SM overlap one CTA's copy with another's math (no ring needed: compute per tile is short).
//   narrow_fwd : Y = [lrelu(X1*sc+sh) | X2]·Wᵀ (+bias), Σ/Σ² epilogue
//   narrow_bwd : dH on the fly; dX = dH·W (split into the two segments, optional +=); dW += dHᵀ·A
// The dispatch (narrow_shape below) sends them Cout <= 16 AND C1 + C2 <= 16, every count a multiple of 4, no dbias; at >= 8,192
// rows, and the forward only when the tcgen05 kernel turns the call down (gathered rows, slope1 outside [0, 1]).  So the kernels
// are instantiated for a padded Cout of 8 / 16 and, in backward, a padded Ktot of 16.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "linear2.cuh"
#include "linear_args.cuh"

namespace crf {
namespace narrow {

using lin::BnBwd;
using lin::DgradArgs;
using lin::FwdArgs;
using lin::WgradArgs;
using lin2::cp_async16;
using lin2::cp_async_commit;
using lin2::cp_async_wait;
using lin::lrelu;

constexpr int TR = 128;          // rows per tile = threads per CTA

// ------------------------------------------------------------------------------------------ forward
template <int CO>
__global__ void __launch_bounds__(TR) fwd_kernel(const FwdArgs a, const int ntiles) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int Ktot = a.C1 + a.C2, XS = Ktot + 4;
    float* Xs = reinterpret_cast<float*>(smem_raw);          // [TR][XS]
    float* Wt = Xs + TR * XS;                                // [Ktot][CO]   Wt[k][c] = W[c][k]
    float* s_sc = Wt + Ktot * CO;                            // [Ktot]
    float* s_sh = s_sc + Ktot;
    float* s_sum = s_sh + Ktot;                              // [CO]
    float* s_sq = s_sum + CO;
    const int tid = threadIdx.x, lane = tid & 31;
    for (int e = tid; e < Ktot * CO; e += TR) {
        const int k = e / CO, c = e % CO;
        Wt[e] = c < a.Cout ? __ldg(a.W + (int64_t)c * Ktot + k) : 0.f;
    }
    for (int k = tid; k < Ktot; k += TR) {
        const bool pro = a.scale1 && k < a.C1;
        s_sc[k] = pro ? __ldg(a.scale1 + k) : 1.f;
        s_sh[k] = pro ? __ldg(a.shift1 + k) : 0.f;
    }
    if (tid < CO) { s_sum[tid] = 0.f; s_sq[tid] = 0.f; }
    const float slope1 = a.scale1 ? a.slope1 : 1.0f;
    const int f4 = Ktot / 4;                                 // float4 per row

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t m0 = (int64_t)tile * TR;
        __syncthreads();                                     // previous tile fully consumed (and setup visible)
        for (int e = tid; e < TR * f4; e += TR) {
            const int r = e / f4, c = 4 * (e % f4);
            const int64_t m = m0 + r;
            const bool ok = m < a.M;
            const float* src = a.X1;
            if (ok) {
                if (c < a.C1) {
                    int64_t srow = m;
                    if (a.idx1) srow = (m / a.rows_dst) * a.rows_src + __ldg(a.idx1 + m);
                    src = a.X1 + srow * a.C1 + c;
                } else {
                    src = a.X2 + m * a.C2 + (c - a.C1);
                }
            }
            cp_async16(Xs + r * XS + c, src, ok);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        float acc[CO];
#pragma unroll
        for (int c = 0; c < CO; ++c) acc[c] = 0.f;
        const float* xr = Xs + tid * XS;
        for (int k4 = 0; k4 < Ktot; k4 += 4) {
            const float4 xv = *reinterpret_cast<const float4*>(xr + k4);
            const float sl = k4 < a.C1 ? slope1 : 1.0f;
            const float x[4] = {lrelu(fmaf(xv.x, s_sc[k4], s_sh[k4]), sl), lrelu(fmaf(xv.y, s_sc[k4 + 1], s_sh[k4 + 1]), sl),
                                lrelu(fmaf(xv.z, s_sc[k4 + 2], s_sh[k4 + 2]), sl), lrelu(fmaf(xv.w, s_sc[k4 + 3], s_sh[k4 + 3]), sl)};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float* wr = Wt + (k4 + u) * CO;
#pragma unroll
                for (int c = 0; c < CO; c += 4) {
                    const float4 w = *reinterpret_cast<const float4*>(wr + c);
                    acc[c] = fmaf(x[u], w.x, acc[c]); acc[c + 1] = fmaf(x[u], w.y, acc[c + 1]);
                    acc[c + 2] = fmaf(x[u], w.z, acc[c + 2]); acc[c + 3] = fmaf(x[u], w.w, acc[c + 3]);
                }
            }
        }
        const int64_t m = m0 + tid;
        const bool valid = m < a.M;
        if (a.bias) {
#pragma unroll
            for (int c = 0; c < CO; ++c)
                if (c < a.Cout) acc[c] += __ldg(a.bias + c);
        }
        if (valid) {
#pragma unroll
            for (int c = 0; c < CO; c += 4)
                if (c < a.Cout) *reinterpret_cast<float4*>(a.Y + m * a.Cout + c) = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
        }
        if (a.stats) {
#pragma unroll
            for (int c = 0; c < CO; ++c) {
                float s = valid ? acc[c] : 0.f, q = s * s;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
                if (lane == 0) { atomicAdd(&s_sum[c], s); atomicAdd(&s_sq[c], q); }
            }
        }
    }
    if (a.stats) {
        __syncthreads();
        if (tid < CO && tid < a.Cout) {
            float* st = a.stats + (size_t)(blockIdx.x % kStatSlots) * 2 * a.Cout;
            atomicAdd(st + tid, s_sum[tid]);
            atomicAdd(st + a.Cout + tid, s_sq[tid]);
        }
    }
}

template <int CO>
size_t fwd_smem(int Ktot) { return (size_t)(TR * (Ktot + 4) + Ktot * CO + 2 * Ktot + 2 * CO) * 4; }

// ------------------------------------------------------------------------------------------ backward
// One kernel does dgrad and wgrad.  CO = padded Cout held in registers per row; KT = padded Ktot (multiple of 16).
// Phase 1 (thread per row): dH row from (dY, H[, ref]) → registers + shared; dX = dH·W in 32-column chunks.
// Phase 2 (4x4 register blocks): dW[co, k] += Σ_rows dH[row, co]·A[row, k] from the shared tiles.
struct BwdArgs {
    DgradArgs d;          // dY, H, bn, W, dX1/dX2 (+acc), M, Cout, C1, C2
    const float* X1; const float* scale1; const float* shift1; float slope1;
    const int64_t* idx1; int64_t rows_dst; int64_t rows_src;
    const float* X2;
    float* dW;            // may be null (dgrad only)
    int64_t slot_stride;
    int need_dx;
};

template <int CO, int KT, bool REF>
__global__ void __launch_bounds__(TR) bwd_kernel(const BwdArgs b, const int ntiles) {
    constexpr int DS = CO + 4, XS = KT + 4;
    constexpr int NBLK = (CO / 4) * (KT / 4);                 // 4x4 output blocks of dW
    constexpr int RG = (TR >= NBLK) ? TR / NBLK : 1;          // row groups when there are fewer blocks than threads
    constexpr int BPT = (NBLK + TR - 1) / TR;                 // blocks per thread when there are more
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* Dr = reinterpret_cast<float*>(smem_raw);           // [TR][DS] dY  → overwritten by dH
    float* Hr = Dr + TR * DS;                                 // [TR][DS] H
    float* Rr = Hr + TR * DS;                                 // [TR][DS] act_ref (REF only)
    float* Xs = Rr + (REF ? TR * DS : 0);                     // [TR][XS] A = [X1 | X2] raw → activated in place
    float* Ws = Xs + TR * XS;                                 // [CO][KT]  W (row-major, zero padded)
    float4* s_par = reinterpret_cast<float4*>(Ws + CO * KT);  // [CO] (sc, sh, p, q)
    float2* s_pro = reinterpret_cast<float2*>(s_par + CO);    // [KT] X prologue
    const DgradArgs& a = b.d;
    const bool plain = a.bn.scale == nullptr;
    const int tid = threadIdx.x;
    const int Ktot = a.C1 + a.C2, C = a.Cout;

    for (int e = tid; e < CO * KT; e += TR) {
        const int co = e / KT, k = e % KT;
        Ws[e] = (co < C && k < Ktot) ? __ldg(a.W + (int64_t)co * Ktot + k) : 0.f;
    }
    for (int k = tid; k < CO; k += TR) s_par[k] = (!plain && k < C) ? a.bn.coef(k) : make_float4(1.f, 0.f, 0.f, 0.f);
    for (int k = tid; k < KT; k += TR) {
        float2 pr = make_float2(1.f, 0.f);
        if (b.scale1 && k < a.C1) pr = make_float2(__ldg(b.scale1 + k), __ldg(b.shift1 + k));
        s_pro[k] = pr;
    }
    const float slope = a.bn.slope, slope1 = b.scale1 ? b.slope1 : 1.0f;

    float wacc[BPT][4][4];
#pragma unroll
    for (int i = 0; i < BPT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int k = 0; k < 4; ++k) wacc[i][j][k] = 0.f;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t m0 = (int64_t)tile * TR;
        __syncthreads();
        for (int e = tid; e < TR * (CO / 4); e += TR) {
            const int r = e / (CO / 4), c = 4 * (e % (CO / 4));
            const int64_t m = m0 + r;
            const bool ok = (m < a.M) && (c < C);
            const int64_t off = ok ? m * C + c : 0;
            cp_async16(Dr + r * DS + c, a.dY + off, ok);
            if (!plain) cp_async16(Hr + r * DS + c, a.H + off, ok);
            if (REF) cp_async16(Rr + r * DS + c, a.bn.act_ref + off, ok);
        }
        if (b.dW) {
            for (int e = tid; e < TR * (KT / 4); e += TR) {
                const int r = e / (KT / 4), c = 4 * (e % (KT / 4));
                const int64_t m = m0 + r;
                const bool ok = (m < a.M) && (c < Ktot);
                const float* src = b.X1;
                if (ok) {
                    if (c < a.C1) {
                        int64_t srow = m;
                        if (b.idx1) srow = (m / b.rows_dst) * b.rows_src + __ldg(b.idx1 + m);
                        src = b.X1 + srow * a.C1 + c;
                    } else {
                        src = b.X2 + m * a.C2 + (c - a.C1);
                    }
                }
                cp_async16(Xs + r * XS + c, src, ok);
            }
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        // ---- phase 1: this thread's row
        const int64_t m = m0 + tid;
        const bool valid = m < a.M;
        float dh[CO];
        {
            float* dr = Dr + tid * DS;
            const float* hr = Hr + tid * DS;
            const float* rr = Rr + tid * DS;
#pragma unroll
            for (int c = 0; c < CO; ++c) {
                float d = dr[c];
                if (!plain) {
                    const float h = hr[c];
                    const float4 p = s_par[c];
                    const float pre = REF ? rr[c] : fmaf(h, p.x, p.y);
                    const float dv = pre > 0.f ? d : d * slope;
                    d = fmaf(p.x, dv, fmaf(p.z, h, p.w));
                }
                dh[c] = (valid && c < C) ? d : 0.f;
                dr[c] = dh[c];                                   // dH tile for phase 2 (own row only: no hazard)
            }
        }
        if (b.dW) {                                              // activate own row of A in place
            float* xr = Xs + tid * XS;
            for (int k = 0; k < KT; ++k) {
                const float2 pr = s_pro[k];
                const float v = lrelu(fmaf(xr[k], pr.x, pr.y), k < a.C1 ? slope1 : 1.0f);
                xr[k] = (valid && k < Ktot) ? v : 0.f;
            }
        }
        if (b.need_dx) {
#pragma unroll 1
            for (int kc = 0; kc < KT; kc += 16) {
                float acc[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[j] = 0.f;
#pragma unroll
                for (int co = 0; co < CO; ++co) {
                    const float* wr = Ws + co * KT + kc;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const float4 w = *reinterpret_cast<const float4*>(wr + j);
                        acc[j] = fmaf(dh[co], w.x, acc[j]); acc[j + 1] = fmaf(dh[co], w.y, acc[j + 1]);
                        acc[j + 2] = fmaf(dh[co], w.z, acc[j + 2]); acc[j + 3] = fmaf(dh[co], w.w, acc[j + 3]);
                    }
                }
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const int col = kc + j;
                        if (col >= Ktot) continue;
                        float* dst; int cc, ld, accm;
                        if (col < a.C1) { dst = a.dX1; cc = col; ld = a.C1; accm = a.acc1; }
                        else            { dst = a.dX2; cc = col - a.C1; ld = a.C2; accm = a.acc2; }
                        if (!dst) continue;
                        float4* p = reinterpret_cast<float4*>(dst + m * ld + cc);
                        float4 o = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
                        if (accm) { const float4 old = *p; o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
                        *p = o;
                    }
                }
            }
        }
        // ---- phase 2: dW += dHᵀ·A over this tile
        if (b.dW) {
            __syncthreads();
#pragma unroll
            for (int i = 0; i < BPT; ++i) {
                const int blk = (NBLK >= TR) ? tid + i * TR : tid % NBLK;
                const int rg = (NBLK >= TR) ? 0 : tid / NBLK;
                if (blk < NBLK && rg < RG) {
                    const int a0 = 4 * (blk / (KT / 4)), b0 = 4 * (blk % (KT / 4));
                    for (int r = rg; r < TR; r += RG) {
                        const float4 dv = *reinterpret_cast<const float4*>(Dr + r * DS + a0);
                        const float4 xv = *reinterpret_cast<const float4*>(Xs + r * XS + b0);
                        const float d4[4] = {dv.x, dv.y, dv.z, dv.w}, x4[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                        for (int p = 0; p < 4; ++p)
#pragma unroll
                            for (int q = 0; q < 4; ++q) wacc[i][p][q] = fmaf(d4[p], x4[q], wacc[i][p][q]);
                    }
                }
            }
        }
    }
    if (b.dW) {
        // combine the RG row groups in shared memory (re-using the A tile), then ONE add per output element per CTA
        __syncthreads();
        float* red = Xs;                                      // CO*KT floats <= TR*XS
        for (int e = tid; e < CO * KT; e += TR) red[e] = 0.f;
        __syncthreads();
        float* dst = b.dW + b.slot_stride * (blockIdx.x % kGradSlots);
#pragma unroll
        for (int i = 0; i < BPT; ++i) {
            const int blk = (NBLK >= TR) ? tid + i * TR : tid % NBLK;
            const int rg = (NBLK >= TR) ? 0 : tid / NBLK;
            if (blk < NBLK && rg < RG) {
                const int a0 = 4 * (blk / (KT / 4)), b0 = 4 * (blk % (KT / 4));
#pragma unroll
                for (int p = 0; p < 4; ++p)
#pragma unroll
                    for (int q = 0; q < 4; ++q) atomicAdd(&red[(a0 + p) * KT + b0 + q], wacc[i][p][q]);
            }
        }
        __syncthreads();
        for (int e = tid; e < CO * KT; e += TR) {
            const int co = e / KT, k = e % KT;
            if (co < C && k < Ktot) atomicAdd(dst + (int64_t)co * Ktot + k, red[e]);
        }
    }
}

template <int CO, int KT, bool REF>
size_t bwd_smem() { return (size_t)(TR * (CO + 4) * (REF ? 3 : 2) + TR * (KT + 4) + CO * KT) * 4 + (size_t)CO * 16 + (size_t)KT * 8; }

}  // namespace narrow

namespace lin {

// Shapes routed to the CUDA-core kernels.  Measured against the tensor-core kernels on B200 (profiles/README_r01.md), one thread
// per row only wins for hidden×hidden layers
// (16→16 forward 25 vs 28 µs, backward 29 vs 45 µs, GC/GM 27 vs 33 µs per call at 245,760 rows): with one thread per row the
// per-element BN+LeakyReLU prologue and the per-channel butterfly statistics cost more issue slots than the FFMAs they feed.
static inline bool narrow_shape(int Cout, int Ktot) { return Cout <= 16 && Ktot <= 16; }

// CTAs per SM that fit in 200 KB of shared memory (1 KB reserved per CTA), at most 8
static inline int ctas_per_sm(size_t smem) { return (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 1024))); }

int try_narrow_fwd(const FwdArgs& a, cudaStream_t st) {
    using namespace narrow;
    const int Ktot = a.C1 + a.C2;
    if (!narrow_shape(a.Cout, Ktot) || (a.Cout & 3) || (a.C1 & 3) || (a.C2 & 3) || a.C1 == 0) return kDeclined;
    if (!aligned16(a.X1) || (a.C2 && !aligned16(a.X2)) || !aligned16(a.Y)) return kDeclined;
    const int ntiles = (int)ceil_div(a.M, TR);
    auto go = [&](auto kern, size_t smem) {
        return launch(kern, dim3(std::min(ntiles, ctas_per_sm(smem) * kNumSMs)), dim3(TR), smem, st, a, ntiles);
    };
    if (a.Cout > 8) return go(fwd_kernel<16>, fwd_smem<16>(Ktot));
    return go(fwd_kernel<8>, fwd_smem<8>(Ktot));
}

int try_narrow_bwd(const DgradArgs& d, const WgradArgs* w, cudaStream_t st) {
    using namespace narrow;
    const int Ktot = d.C1 + d.C2, C = d.Cout;
    if (!narrow_shape(C, Ktot) || (C & 3) || (d.C1 & 3) || (d.C2 & 3) || d.C1 == 0) return kDeclined;
    if (w && w->dbias) return kDeclined;
    if (!aligned16(d.dY) || (d.bn.scale && !aligned16(d.H)) || (d.bn.act_ref && !aligned16(d.bn.act_ref))) return kDeclined;
    if ((d.dX1 && !aligned16(d.dX1)) || (d.dX2 && !aligned16(d.dX2))) return kDeclined;
    if (w && (!aligned16(w->X1) || (d.C2 && !aligned16(w->X2)))) return kDeclined;
    BwdArgs b{};
    b.d = d;
    b.need_dx = (d.dX1 || d.dX2) ? 1 : 0;
    if (w) {
        b.X1 = w->X1; b.scale1 = w->scale1; b.shift1 = w->shift1; b.slope1 = w->slope1;
        b.idx1 = w->idx1; b.rows_dst = w->rows_dst; b.rows_src = w->rows_src; b.X2 = w->X2; b.dW = w->dW; b.slot_stride = w->slot_stride;
    }
    const bool ref = d.bn.scale && d.bn.act_ref;
    const int ntiles = (int)ceil_div(d.M, TR);
    auto go = [&](auto kern, size_t smem) {
        return launch(kern, dim3(std::min(ntiles, ctas_per_sm(smem) * kNumSMs)), dim3(TR), smem, st, b, ntiles);
    };
    if (C > 8) return ref ? go(bwd_kernel<16, 16, true>, bwd_smem<16, 16, true>()) : go(bwd_kernel<16, 16, false>, bwd_smem<16, 16, false>());
    return ref ? go(bwd_kernel<8, 16, true>, bwd_smem<8, 16, true>()) : go(bwd_kernel<8, 16, false>, bwd_smem<8, 16, false>());
}

}  // namespace lin
}  // namespace crf
