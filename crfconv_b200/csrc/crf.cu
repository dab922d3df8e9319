// Continuous-CRF mean-field message passing on sm_100a — forward and backward of the loop in
// /root/reference/models/continuous_crf_conv_big.py:49-54,60-72 (math in SURVEY.md Appendix B):
//     s_ij = softmax_j( -||y_i - y_j||² )  over the K-1 neighbours j of i (column 0 of neighbor_idx dropped, :45-47)
//     x^t_i = ( z_i + ( Σ_j s_ij x^{t-1}_j ) · C ) · Minv ,   C = cᵀc ,  Minv = (I + C)^{-1} ,  x^0 = z = u[up_idx]
// One fused kernel per mean-field step: distances, the softmax over k (online, flash-style rescaling), the weighted
// aggregation and the two F×F compatibility products happen in registers; neither the [N,K,F] neighbour tensor nor
// the [N,K,F] int64 repeated index of the reference (continuous_crf_conv_big.py:38-43) is ever materialised.
// Layout: F/4 lanes cooperate on one point, each holding a float4 channel slice, so every neighbour row is fetched
// with 128-bit loads (a 16-float row = 64 B = 4 lanes); feature tables are L2 resident at these sizes.
// y is consumed as its pre-BatchNorm tensor Hy with the BN scale applied on the fly (the BN shift cancels in y_i-y_j).
// Backward scatters along the transposed graph with vector reductions (red.global.add.v4.f32) into L2-resident rows.
#include <type_traits>

#include "../../include/crfconv_b200.h"
#include "common.cuh"
#include "fused_common.cuh"

namespace crf {
namespace mf {

__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <int LP>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = LP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// out[c0..c0+3] = Σ_k full[k] * Mat[k][c0+e]  (row vector times matrix; Mat in shared memory, row-major [F][F])
template <int F>
__device__ __forceinline__ float4 rowvec_mat(const float (&full)[F], const float* Mat, int c0) {
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < F; ++k) {
        const float4 m = *reinterpret_cast<const float4*>(Mat + k * F + c0);
        o.x = fmaf(full[k], m.x, o.x); o.y = fmaf(full[k], m.y, o.y); o.z = fmaf(full[k], m.z, o.z); o.w = fmaf(full[k], m.w, o.w);
    }
    return o;
}
// out[c0+e] = Σ_k full[k] * Mat[c0+e][k]   (row vector times matrix transposed)
template <int F>
__device__ __forceinline__ float4 rowvec_matT(const float (&full)[F], const float* Mat, int c0) {
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int k = 0; k < F; ++k) o[e] = fmaf(full[k], Mat[(c0 + e) * F + k], o[e]);
    return make_float4(o[0], o[1], o[2], o[3]);
}

// all-gather of a float4 slice across the LP lanes of a point group → full[F]
template <int F>
__device__ __forceinline__ void gather_full(float4 v, float (&full)[F], int lane) {
    constexpr int LP = F / 4;
    const int gbase = lane & ~(LP - 1);
#pragma unroll
    for (int s = 0; s < LP; ++s) {
        full[4 * s + 0] = __shfl_sync(0xffffffffu, v.x, gbase + s);
        full[4 * s + 1] = __shfl_sync(0xffffffffu, v.y, gbase + s);
        full[4 * s + 2] = __shfl_sync(0xffffffffu, v.z, gbase + s);
        full[4 * s + 3] = __shfl_sync(0xffffffffu, v.w, gbase + s);
    }
}

// The 16 int64 neighbour indices of a point are one 128-byte row.  Per-lane scalar loads of them cost one L1 wavefront per index
// and point (15 of the ≈50 wavefronts a point costs in the forward kernel, which ncu shows bound by l1tex data-pipe
// wavefronts); instead the 4 lanes of a point fetch the row with two 128-bit loads each and hand indices around by shuffle.
// Lane s of the group ends up with indices {2s, 2s+1, 8+2s, 8+2s+1} in r[0..3].
__device__ __forceinline__ void load_idx16(const int64_t* nb, int sub, int (&r)[4]) {
    const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(nb) + sub);
    const longlong2 b = __ldg(reinterpret_cast<const longlong2*>(nb) + 4 + sub);
    r[0] = (int)a.x; r[1] = (int)a.y; r[2] = (int)b.x; r[3] = (int)b.y;
}
template <int k>
__device__ __forceinline__ int idx16_get(const int (&r)[4], int gbase) {
    return __shfl_sync(0xffffffffu, r[(k >> 3) * 2 + (k & 1)], gbase + ((k & 7) >> 1));
}

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 sub4(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

// z[m] = Hu[b*Nc + up[m]] * scale + shift        (continuous_crf_conv_big.py:60 after unary_nn's last BatchNorm)
__global__ void __launch_bounds__(256) upsample_affine_kernel(const float* __restrict__ Hu, const float* __restrict__ scale,
                                                              const float* __restrict__ shift, const int64_t* __restrict__ up,
                                                              float* __restrict__ z, int64_t total, int64_t N, int64_t Nc, int F4) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total * F4) return;
    const int64_t m = i / F4;
    const int c = (int)(i % F4) * 4;
    const int64_t src = (m / N) * Nc + __ldg(up + m);
    const float4 h = ld4(Hu + src * (F4 * 4) + c), sc = ld4(scale + c), sh = ld4(shift + c);
    reinterpret_cast<float4*>(z)[i] = make_float4(fmaf(h.x, sc.x, sh.x), fmaf(h.y, sc.y, sh.y), fmaf(h.z, sc.z, sh.z), fmaf(h.w, sc.w, sh.w));
}

// Gu[b*Nc + up[m]] += Gz[m] + G0[m]
__global__ void __launch_bounds__(256) upsample_bwd_kernel(const float* __restrict__ Gz, const float* __restrict__ G0,
                                                           const int64_t* __restrict__ up, float* Gu, int64_t total, int64_t N,
                                                           int64_t Nc, int F4) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total * F4) return;
    const int64_t m = i / F4;
    const int c = (int)(i % F4) * 4;
    const int64_t dst = (m / N) * Nc + __ldg(up + m);
    float4 a = ld4(Gz + i * 4);
    if (G0) { const float4 b = ld4(G0 + i * 4); a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
    red_add_v4(Gu + dst * (F4 * 4) + c, a);
}

struct StepArgs {
    const float* Hy;       // [B*N, F] pre-BN pairwise embedding
    const float* scale_y;  // [F]  y = Hy*scale_y + shift_y (shift cancels)
    const float* z;        // [B*N, F]
    const float* xprev;    // [B*N, F]  x^{t-1}
    const int64_t* nbr;    // [B*N, K] indices local to the cloud; column 0 skipped
    const float* Cm;       // [F, F]
    const float* Minv;     // [F, F]
    int64_t total, N;
    int K;
    // forward
    float* xout;           // [B*N, F]  x^t
    // backward
    const float* g;        // [B*N, F]  dL/dx^t
    float* Gz;             // [B*N, F]  (+)= h_i          (owner writes; += when gz_acc)
    int gz_acc;
    float* gprev;          // [B*N, F]  += s_ij q_i       (scatter, zero-initialised by the caller)
    float* Gy;             // [B*N, F]  += distance-path gradient wrt y (scatter)
    float* m_out;          // [B*N, F]  m_i               (for GC = mᵀh)
    float* v_out;          // [B*N, F]  z_i + m_i C       (for GM = vᵀg)
    float* h_out;          // [B*N, F]  h_i = g_i Minvᵀ
};

template <int F>
__global__ void __launch_bounds__(256, F == 16 ? 5 : 1) step_fwd_kernel(const StepArgs a) {
    constexpr int LP = F / 4, PPW = 32 / LP;
    constexpr bool TC = F == 16;                           // hidden width of the hot path: the two F×F products on the tensor cores
    __shared__ __align__(16) float Cs[TC ? 4 : F * F];
    __shared__ __align__(16) float Ms[TC ? 4 : F * F];
    __shared__ __align__(16) float4 fC[TC ? 128 : 1], fM[TC ? 128 : 1];
    if constexpr (TC) {
        cl::stage_mat16(fC, [&](int k, int n) { return a.Cm[k * 16 + n]; }, threadIdx.x, blockDim.x);
        cl::stage_mat16(fM, [&](int k, int n) { return a.Minv[k * 16 + n]; }, threadIdx.x, blockDim.x);
    } else {
        for (int i = threadIdx.x; i < F * F; i += blockDim.x) { Cs[i] = a.Cm[i]; Ms[i] = a.Minv[i]; }
    }
    __syncthreads();
    const int lane = lane_id();
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int64_t p = warp * PPW + lane / LP;
    const bool valid = p < a.total;
    if (!valid) p = a.total - 1;
    const int c0 = (lane % LP) * 4;
    const int64_t base = (p / a.N) * a.N;
    const float4 sc = ld4(a.scale_y + c0);
    const float4 yi = mul4(ld4(a.Hy + p * F + c0), sc);

    float mx = -INFINITY, l = 0.f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t* nb = a.nbr + p * a.K;
    auto edge = [&](int64_t row) {
        const float4 df = sub4(yi, mul4(ld4(a.Hy + row * F + c0), sc));
        const float d = group_sum<LP>(dot4(df, df));
        const float4 xj = ld4(a.xprev + row * F + c0);
        const float al = -d;
        const float nm = fmaxf(mx, al);
        const float corr = __expf(mx - nm), pj = __expf(al - nm);
        l = l * corr + pj;
        acc.x = acc.x * corr + pj * xj.x; acc.y = acc.y * corr + pj * xj.y;
        acc.z = acc.z * corr + pj * xj.z; acc.w = acc.w * corr + pj * xj.w;
        mx = nm;
    };
    bool done = false;
    if constexpr (F == 16) {
        if (a.K == 16) {                                   // the reference's kernel_size: indices by vector load + shuffle
            int r[4];
            load_idx16(nb, lane % LP, r);
            const int gb = lane & ~(LP - 1);
            edge(base + idx16_get<1>(r, gb));  edge(base + idx16_get<2>(r, gb));  edge(base + idx16_get<3>(r, gb));
            edge(base + idx16_get<4>(r, gb));  edge(base + idx16_get<5>(r, gb));  edge(base + idx16_get<6>(r, gb));
            edge(base + idx16_get<7>(r, gb));  edge(base + idx16_get<8>(r, gb));  edge(base + idx16_get<9>(r, gb));
            edge(base + idx16_get<10>(r, gb)); edge(base + idx16_get<11>(r, gb)); edge(base + idx16_get<12>(r, gb));
            edge(base + idx16_get<13>(r, gb)); edge(base + idx16_get<14>(r, gb)); edge(base + idx16_get<15>(r, gb));
            done = true;
        }
    }
    if (!done)
        for (int k = 1; k < a.K; ++k) edge(base + __ldg(nb + k));
    const float inv_l = a.K > 1 ? 1.0f / l : 0.0f;
    const float4 msg = make_float4(acc.x * inv_l, acc.y * inv_l, acc.z * inv_l, acc.w * inv_l);
    const float4 zi = ld4(a.z + p * F + c0);
    float4 x;
    if constexpr (TC) {                                    // x = (z + m·C)·Minv, chained through MMA fragments (fused_common.cuh)
        float4 v = cl::rows8_mat16(msg, fC, lane);
        v.x += zi.x; v.y += zi.y; v.z += zi.z; v.w += zi.w;
        x = cl::rows8_mat16(v, fM, lane);
    } else {
        float full[F];
        gather_full<F>(msg, full, lane);
        float4 v = rowvec_mat<F>(full, Cs, c0);
        v.x += zi.x; v.y += zi.y; v.z += zi.z; v.w += zi.w;
        gather_full<F>(v, full, lane);
        x = rowvec_mat<F>(full, Ms, c0);
    }
    if (valid) *reinterpret_cast<float4*>(a.xout + p * F + c0) = x;
}

template <int F>
__global__ void __launch_bounds__(256) step_bwd_kernel(const StepArgs a) {
    constexpr int LP = F / 4, PPW = 32 / LP;
    __shared__ __align__(16) float Cs[F * F];
    __shared__ __align__(16) float Ms[F * F];
    for (int i = threadIdx.x; i < F * F; i += blockDim.x) { Cs[i] = a.Cm[i]; Ms[i] = a.Minv[i]; }
    __syncthreads();
    const int lane = lane_id();
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int64_t p = warp * PPW + lane / LP;
    const bool valid = p < a.total;
    if (!valid) p = a.total - 1;
    const int c0 = (lane % LP) * 4;
    const int64_t base = (p / a.N) * a.N;
    const float4 sc = ld4(a.scale_y + c0);
    const float4 yi = mul4(ld4(a.Hy + p * F + c0), sc);

    // h = g·Minvᵀ ; q = h·Cᵀ
    float full[F];
    const float4 gi = ld4(a.g + p * F + c0);
    gather_full<F>(gi, full, lane);
    const float4 h = rowvec_matT<F>(full, Ms, c0);
    gather_full<F>(h, full, lane);
    const float4 q = rowvec_matT<F>(full, Cs, c0);

    // pass 1 (online): softmax normaliser, message m_i, and dot = Σ_k s_ik <q_i, x_k>
    float mx = -INFINITY, l = 0.f, tacc = 0.f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t* nb = a.nbr + p * a.K;
    for (int k = 1; k < a.K; ++k) {
        const int64_t row = base + __ldg(nb + k);
        const float4 df = sub4(yi, mul4(ld4(a.Hy + row * F + c0), sc));
        const float4 xj = ld4(a.xprev + row * F + c0);
        const float d = group_sum<LP>(dot4(df, df));
        const float gs = group_sum<LP>(dot4(q, xj));
        const float al = -d;
        const float nm = fmaxf(mx, al);
        const float corr = __expf(mx - nm), pj = __expf(al - nm);
        l = l * corr + pj;
        tacc = tacc * corr + pj * gs;
        acc.x = acc.x * corr + pj * xj.x; acc.y = acc.y * corr + pj * xj.y;
        acc.z = acc.z * corr + pj * xj.z; acc.w = acc.w * corr + pj * xj.w;
        mx = nm;
    }
    const float inv_l = a.K > 1 ? 1.0f / l : 0.0f;
    const float sdot = tacc * inv_l;
    const float4 msg = make_float4(acc.x * inv_l, acc.y * inv_l, acc.z * inv_l, acc.w * inv_l);

    // pass 2: per-edge gradients, scattered along the transposed graph
    float4 gyi = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 1; k < a.K; ++k) {
        const int64_t row = base + __ldg(nb + k);
        const float4 df = sub4(yi, mul4(ld4(a.Hy + row * F + c0), sc));
        const float4 xj = ld4(a.xprev + row * F + c0);
        const float d = group_sum<LP>(dot4(df, df));
        const float gs = group_sum<LP>(dot4(q, xj));
        const float s = __expf(-d - mx) * inv_l;
        const float ga2 = 2.0f * s * (gs - sdot);                 // 2·Ga_ij
        // Gy_i += -2 Ga (y_i - y_j) ; Gy_j += +2 Ga (y_i - y_j)
        gyi.x -= ga2 * df.x; gyi.y -= ga2 * df.y; gyi.z -= ga2 * df.z; gyi.w -= ga2 * df.w;
        if (valid) {
            red_add_v4(a.Gy + row * F + c0, make_float4(ga2 * df.x, ga2 * df.y, ga2 * df.z, ga2 * df.w));
            red_add_v4(a.gprev + row * F + c0, make_float4(s * q.x, s * q.y, s * q.z, s * q.w));
        }
    }
    if (valid) {
        red_add_v4(a.Gy + p * F + c0, gyi);
        float* gz = a.Gz + p * F + c0;
        float4 o = h;
        if (a.gz_acc) { const float4 old = *reinterpret_cast<float4*>(gz); o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
        *reinterpret_cast<float4*>(gz) = o;
        *reinterpret_cast<float4*>(a.h_out + p * F + c0) = h;
        *reinterpret_cast<float4*>(a.m_out + p * F + c0) = msg;
    }
    // v = z + m·C
    gather_full<F>(msg, full, lane);
    float4 v = rowvec_mat<F>(full, Cs, c0);
    const float4 zi = ld4(a.z + p * F + c0);
    v.x += zi.x; v.y += zi.y; v.z += zi.z; v.w += zi.w;
    if (valid) *reinterpret_cast<float4*>(a.v_out + p * F + c0) = v;
}

// Single-gather variant for the common neighbourhood size (K-1 = KN known at compile time): every neighbour row is fetched
// ONCE; y_j slices, distances and <q, x_j> stay in registers between the softmax pass and the scatter pass.  The generic
// kernel above re-gathers in its second pass; ncu shows it L1TEX-throughput bound (82 %), so transactions are what to cut.
template <int F, int KN>
__global__ void __launch_bounds__(128) step_bwd_reg_kernel(const StepArgs a) {
    constexpr int LP = F / 4, PPW = 32 / LP;
    __shared__ __align__(16) float CsT[F * F];   // transposed copies: out[c] = Σ_k v[k]·Mat[c][k] becomes a row-vector product
    __shared__ __align__(16) float MsT[F * F];
    __shared__ __align__(16) float Cs[F * F];
    for (int i = threadIdx.x; i < F * F; i += blockDim.x) {
        const int r = i / F, c = i % F;
        Cs[i] = a.Cm[i];
        CsT[c * F + r] = a.Cm[i];
        MsT[c * F + r] = a.Minv[i];
    }
    __syncthreads();
    const int lane = lane_id();
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int64_t p = warp * PPW + lane / LP;
    const bool valid = p < a.total;
    if (!valid) p = a.total - 1;
    const int c0 = (lane % LP) * 4;
    const int64_t base = (p / a.N) * a.N;
    const float4 sc = ld4(a.scale_y + c0);
    const float4 yi = mul4(ld4(a.Hy + p * F + c0), sc);

    float full[F];
    const float4 gi = ld4(a.g + p * F + c0);
    gather_full<F>(gi, full, lane);
    const float4 h = rowvec_mat<F>(full, MsT, c0);       // h = g·Minvᵀ
    gather_full<F>(h, full, lane);
    const float4 q = rowvec_mat<F>(full, CsT, c0);       // q = h·Cᵀ

    int rj[KN];
    float4 dfj[KN];
    float dj[KN], gsj[KN];
    const int64_t* nb = a.nbr + p * a.K + 1;
    if constexpr (F == 16 && KN == 15) {                   // K = 16: the index row by vector load + shuffle (see load_idx16)
        int r[4];
        load_idx16(nb - 1, lane % LP, r);
        const int gb = lane & ~(LP - 1);
        rj[0] = idx16_get<1>(r, gb);   rj[1] = idx16_get<2>(r, gb);   rj[2] = idx16_get<3>(r, gb);   rj[3] = idx16_get<4>(r, gb);
        rj[4] = idx16_get<5>(r, gb);   rj[5] = idx16_get<6>(r, gb);   rj[6] = idx16_get<7>(r, gb);   rj[7] = idx16_get<8>(r, gb);
        rj[8] = idx16_get<9>(r, gb);   rj[9] = idx16_get<10>(r, gb);  rj[10] = idx16_get<11>(r, gb); rj[11] = idx16_get<12>(r, gb);
        rj[12] = idx16_get<13>(r, gb); rj[13] = idx16_get<14>(r, gb); rj[14] = idx16_get<15>(r, gb);
    } else {
#pragma unroll
        for (int k = 0; k < KN; ++k) rj[k] = (int)__ldg(nb + k);
    }
    float mx = -INFINITY;
    float4 xj[KN];
#pragma unroll
    for (int k = 0; k < KN; ++k) {                       // all gathers issued back to back
        const int64_t row = base + rj[k];
        dfj[k] = ld4(a.Hy + row * F + c0);
        xj[k] = ld4(a.xprev + row * F + c0);
    }
#pragma unroll
    for (int k = 0; k < KN; ++k) {
        dfj[k] = sub4(yi, mul4(dfj[k], sc));
        dj[k] = group_sum<LP>(dot4(dfj[k], dfj[k]));
        gsj[k] = group_sum<LP>(dot4(q, xj[k]));
        mx = fmaxf(mx, -dj[k]);
    }
    float l = 0.f, tacc = 0.f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < KN; ++k) {
        const float pj = __expf(-dj[k] - mx);
        dj[k] = pj;                                      // reuse the slot for the unnormalised weight
        l += pj;
        tacc = fmaf(pj, gsj[k], tacc);
        acc.x = fmaf(pj, xj[k].x, acc.x); acc.y = fmaf(pj, xj[k].y, acc.y);
        acc.z = fmaf(pj, xj[k].z, acc.z); acc.w = fmaf(pj, xj[k].w, acc.w);
    }
    const float inv_l = 1.0f / l;
    const float sdot = tacc * inv_l;
    const float4 msg = make_float4(acc.x * inv_l, acc.y * inv_l, acc.z * inv_l, acc.w * inv_l);
    float4 gyi = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < KN; ++k) {
        const float s_ = dj[k] * inv_l;
        const float ga2 = 2.0f * s_ * (gsj[k] - sdot);
        const float4 df = dfj[k];
        gyi.x -= ga2 * df.x; gyi.y -= ga2 * df.y; gyi.z -= ga2 * df.z; gyi.w -= ga2 * df.w;
        if (valid) {
            const int64_t row = base + rj[k];
            red_add_v4(a.Gy + row * F + c0, make_float4(ga2 * df.x, ga2 * df.y, ga2 * df.z, ga2 * df.w));
            red_add_v4(a.gprev + row * F + c0, make_float4(s_ * q.x, s_ * q.y, s_ * q.z, s_ * q.w));
        }
    }
    if (valid) {
        red_add_v4(a.Gy + p * F + c0, gyi);
        float* gz = a.Gz + p * F + c0;
        float4 o = h;
        if (a.gz_acc) { const float4 old = *reinterpret_cast<float4*>(gz); o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
        *reinterpret_cast<float4*>(gz) = o;
        *reinterpret_cast<float4*>(a.h_out + p * F + c0) = h;
        *reinterpret_cast<float4*>(a.m_out + p * F + c0) = msg;
    }
    gather_full<F>(msg, full, lane);
    float4 v = rowvec_mat<F>(full, Cs, c0);
    const float4 zi = ld4(a.z + p * F + c0);
    v.x += zi.x; v.y += zi.y; v.z += zi.z; v.w += zi.w;
    if (valid) *reinterpret_cast<float4*>(a.v_out + p * F + c0) = v;
}

// ---- F×F compatibility algebra (single CTA, double precision in a global scratch of 3·F·F doubles)
// Cm = cᵀc ; Minv = (I + Cm)^{-1} by Gauss-Jordan (I + cᵀc is SPD with eigenvalues >= 1: no pivoting needed).
__global__ void __launch_bounds__(256) compat_fwd_kernel(const float* __restrict__ c, float* __restrict__ Cm, float* __restrict__ Minv,
                                                         double* scratch, int F) {
    __shared__ double colp[128];
    __shared__ double piv;
    double* aug = scratch;   // [F][2F]
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < F * F; i += nt) {
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += (double)c[k * F + r] * (double)c[k * F + cc];
        Cm[i] = (float)s;
        aug[r * 2 * F + cc] = s + (r == cc ? 1.0 : 0.0);
        aug[r * 2 * F + F + cc] = (r == cc ? 1.0 : 0.0);
    }
    __syncthreads();
    for (int pcol = 0; pcol < F; ++pcol) {
        if (tid == 0) piv = aug[pcol * 2 * F + pcol];
        for (int r = tid; r < F; r += nt) colp[r] = aug[r * 2 * F + pcol];
        __syncthreads();
        const double ip = 1.0 / piv;
        for (int j = tid; j < 2 * F; j += nt) aug[pcol * 2 * F + j] *= ip;
        __syncthreads();
        for (int i = tid; i < F * 2 * F; i += nt) {
            const int r = i / (2 * F), j = i % (2 * F);
            if (r != pcol) aug[i] -= colp[r] * aug[pcol * 2 * F + j];
        }
        __syncthreads();
    }
    for (int i = tid; i < F * F; i += nt) Minv[i] = (float)aug[(i / F) * 2 * F + F + (i % F)];
}

// Gc += c·(G + Gᵀ),  G = GC − Minvᵀ·GM·Minvᵀ      (C = cᵀc, Minv = (I+C)^{-1})
__global__ void __launch_bounds__(256) compat_bwd_kernel(const float* __restrict__ c, const float* __restrict__ Minv,
                                                         const float* __restrict__ GC, const float* __restrict__ GM, float* Gc,
                                                         double* scratch, int F) {
    double* T = scratch;            // T = Minvᵀ·GM
    double* G = scratch + F * F;    // G = GC − T·Minvᵀ
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < F * F; i += nt) {
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += (double)Minv[k * F + r] * (double)GM[k * F + cc];
        T[i] = s;
    }
    __syncthreads();
    for (int i = tid; i < F * F; i += nt) {
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += T[r * F + k] * (double)Minv[cc * F + k];
        G[i] = (double)GC[i] - s;
    }
    __syncthreads();
    for (int i = tid; i < F * F; i += nt) {
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += (double)c[r * F + k] * (G[k * F + cc] + G[cc * F + k]);
        Gc[i] += (float)s;
    }
}

// Shared-memory versions for F <= 64 (the network's decoder has F = 8, 16, 32, 64): the augmented matrix of the Gauss-Jordan sweep
// and all operands of the three products live in shared memory, 1024 threads.  The global-scratch kernels above paid three dependent
// global round trips per pivot (286 us forward / 375 us backward at F = 64, ≈0.5 ms of a PointConvResNet step on its critical path).
__global__ void __launch_bounds__(1024) compat_fwd_smem_kernel(const float* __restrict__ c, float* __restrict__ Cm, float* __restrict__ Minv,
                                                               int F) {
    extern __shared__ __align__(16) double sm_d[];              // aug [F][2F] | colp [F] | c as doubles [F][F]
    double* aug = sm_d;
    double* colp = aug + F * 2 * F;
    double* cs = colp + F;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < F * F; i += nt) cs[i] = (double)c[i];
    __syncthreads();
    for (int i = tid; i < F * F; i += nt) {
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += cs[k * F + r] * cs[k * F + cc];
        Cm[i] = (float)s;
        aug[r * 2 * F + cc] = s + (r == cc ? 1.0 : 0.0);
        aug[r * 2 * F + F + cc] = (r == cc ? 1.0 : 0.0);
    }
    __syncthreads();
    // thread (r0, j) owns column j of rows r0, r0 + rstep, ...: no index arithmetic inside the sweep (the 1024-thread CTA is issue-bound;
    // a div / mod per element made a pivot cost 2 us)
    const int W = 2 * F, j = tid % W, r0 = tid / W, rstep = nt / W;          // W divides nt (W <= 128, nt = 256 or 1024)
    for (int pcol = 0; pcol < F; ++pcol) {
        const double ip = 1.0 / aug[pcol * W + pcol];
        const double pj = aug[pcol * W + j] * ip;                // scaled pivot-row entry of this thread's column
        if (tid < F) colp[tid] = aug[tid * W + pcol];
        __syncthreads();
        for (int r = r0; r < F; r += rstep) {
            if (r != pcol) aug[r * W + j] -= colp[r] * pj;
            else aug[r * W + j] = pj;
        }
        __syncthreads();
    }
    for (int i = tid; i < F * F; i += nt) Minv[i] = (float)aug[(i / F) * 2 * F + F + (i % F)];
}

__global__ void __launch_bounds__(1024) compat_bwd_smem_kernel(const float* __restrict__ c, const float* __restrict__ Minv,
                                                               const float* __restrict__ GC, const float* __restrict__ GM, float* Gc, int F) {
    extern __shared__ __align__(16) double sm_d[];              // T [F][F+1] | G [F][F+1] | then floats: Minv [F][F+1], GM / c [F][F+1]
    const int L = F + 1;                                        // odd pitch: column walks (stride L) are bank-conflict free
    double* T = sm_d;
    double* G = T + F * L;
    float* Ms = reinterpret_cast<float*>(G + F * L);
    float* Xs = Ms + F * L;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < F * F; i += nt) { Ms[(i / F) * L + i % F] = Minv[i]; Xs[(i / F) * L + i % F] = GM[i]; }
    __syncthreads();
    for (int i = tid; i < F * F; i += nt) {                     // T = Minvᵀ·GM
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += (double)Ms[k * L + r] * (double)Xs[k * L + cc];
        T[r * L + cc] = s;
    }
    __syncthreads();
    for (int i = tid; i < F * F; i += nt) {                     // G = GC − T·Minvᵀ
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += T[r * L + k] * (double)Ms[cc * L + k];
        G[r * L + cc] = (double)GC[i] - s;
    }
    for (int i = tid; i < F * F; i += nt) Xs[(i / F) * L + i % F] = c[i];   // GM's last reads are behind the barrier above
    __syncthreads();
    for (int i = tid; i < F * F; i += nt) {                     // Gc += c·(G + Gᵀ)
        const int r = i / F, cc = i % F;
        double s = 0.0;
        for (int k = 0; k < F; ++k) s += (double)Xs[r * L + k] * (G[k * L + cc] + G[cc * L + k]);
        Gc[i] += (float)s;
    }
}

template <typename Fn>
inline int dispatch_f(int F, Fn&& fn) {
    switch (F) {
        case 4: return fn(std::integral_constant<int, 4>{});
        case 8: return fn(std::integral_constant<int, 8>{});
        case 16: return fn(std::integral_constant<int, 16>{});
        case 32: return fn(std::integral_constant<int, 32>{});
        case 64: return fn(std::integral_constant<int, 64>{});
        default: return CRF_ERR_UNSUPPORTED;
    }
}

}  // namespace mf
}  // namespace crf

using namespace crf;

extern "C" {

int crfconv_crf_compat_fwd(const float* c, float* Cm, float* Minv, double* scratch, int F, void* stream) {
    if (!c || !Cm || !Minv || !scratch || F <= 0 || F > 128) return CRF_ERR_INVALID_ARG;
    if (F <= 64) {
        const size_t smem = ((size_t)F * 2 * F + F + (size_t)F * F) * sizeof(double);
        static bool attr = false;
        if (!attr) { CRF_CUDA(cudaFuncSetAttribute(mf::compat_fwd_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024)); attr = true; }
        mf::compat_fwd_smem_kernel<<<1, F >= 32 ? 1024 : 256, smem, (cudaStream_t)stream>>>(c, Cm, Minv, F);
        CRF_LAUNCH_CHECK();
        return CRF_OK;
    }
    mf::compat_fwd_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(c, Cm, Minv, scratch, F);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

int crfconv_crf_compat_bwd(const float* c, const float* Minv, const float* GC, const float* GM, float* Gc, double* scratch, int F,
                           void* stream) {
    if (!c || !Minv || !GC || !GM || !Gc || !scratch || F <= 0 || F > 128) return CRF_ERR_INVALID_ARG;
    if (F <= 64) {
        const size_t smem = (size_t)2 * F * (F + 1) * sizeof(double) + (size_t)2 * F * (F + 1) * sizeof(float);
        static bool attr = false;
        if (!attr) { CRF_CUDA(cudaFuncSetAttribute(mf::compat_bwd_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024)); attr = true; }
        mf::compat_bwd_smem_kernel<<<1, F >= 32 ? 1024 : 256, smem, (cudaStream_t)stream>>>(c, Minv, GC, GM, Gc, F);
        CRF_LAUNCH_CHECK();
        return CRF_OK;
    }
    mf::compat_bwd_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(c, Minv, GC, GM, Gc, scratch, F);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// z[B*N, F] = affine(Hu[B*Nc, F])[up_idx]
int crfconv_crf_upsample_fwd(const float* Hu, const float* scale, const float* shift, const int64_t* up_idx, float* z, int64_t B,
                             int64_t N, int64_t Nc, int F, void* stream) {
    if (B < 0 || N < 0 || Nc <= 0 || F <= 0 || (F & 3)) return CRF_ERR_INVALID_ARG;
    const int64_t total = B * N;
    if (total == 0) return CRF_OK;
    mf::upsample_affine_kernel<<<(unsigned)ceil_div(total * (F / 4), 256), 256, 0, (cudaStream_t)stream>>>(Hu, scale, shift, up_idx, z, total,
                                                                                                    N, Nc, F / 4);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// Gu[B*Nc, F] += (Gz + G0)[·] scattered through up_idx (G0 may be NULL)
int crfconv_crf_upsample_bwd(const float* Gz, const float* G0, const int64_t* up_idx, float* Gu, int64_t B, int64_t N, int64_t Nc,
                             int F, void* stream) {
    if (B < 0 || N < 0 || Nc <= 0 || F <= 0 || (F & 3)) return CRF_ERR_INVALID_ARG;
    const int64_t total = B * N;
    if (total == 0) return CRF_OK;
    mf::upsample_bwd_kernel<<<(unsigned)ceil_div(total * (F / 4), 256), 256, 0, (cudaStream_t)stream>>>(Gz, G0, up_idx, Gu, total, N, Nc,
                                                                                                 F / 4);
    CRF_LAUNCH_CHECK();
    return CRF_OK;
}

// One mean-field step:  xout = (z + (S·xprev)·Cm)·Minv  with S from Hy*scale_y (continuous_crf_conv_big.py:68-72).
int crfconv_crf_step_fwd(const float* Hy, const float* scale_y, const float* z, const float* xprev, const int64_t* neighbor_idx,
                         const float* Cm, const float* Minv, float* xout, int64_t B, int64_t N, int K, int F, void* stream) {
    if (B < 0 || N < 0 || K < 1 || !Hy || !scale_y || !z || !xprev || !neighbor_idx || !Cm || !Minv || !xout) return CRF_ERR_INVALID_ARG;
    if (B * N == 0) return CRF_OK;
    mf::StepArgs a{};
    a.Hy = Hy; a.scale_y = scale_y; a.z = z; a.xprev = xprev; a.nbr = neighbor_idx; a.Cm = Cm; a.Minv = Minv;
    a.total = B * N; a.N = N; a.K = K; a.xout = xout;
    return mf::dispatch_f(F, [&](auto f) {
        constexpr int FF = decltype(f)::value;
        constexpr int PPW = 32 / (FF / 4);
        const int64_t warps = ceil_div(a.total, PPW);
        mf::step_fwd_kernel<FF><<<(unsigned)ceil_div(warps, 8), 256, 0, (cudaStream_t)stream>>>(a);
        CRF_LAUNCH_CHECK();
        return CRF_OK;
    });
}

// Backward of one step.  g = dL/dx^t.  Gz = h, or += h when gz_acc (owner rows), gprev += Σ s_ij q_i (must be zero-initialised),
// Gy += distance-path gradient (zero-initialised by the caller before the first step), m/v/h rows for GC = mᵀh, GM = vᵀg.
int crfconv_crf_step_bwd(const float* Hy, const float* scale_y, const float* z, const float* xprev, const int64_t* neighbor_idx,
                         const float* Cm, const float* Minv, const float* g, float* Gz, float* gprev, float* Gy, float* m_out,
                         float* v_out, float* h_out, int gz_acc, int64_t B, int64_t N, int K, int F, void* stream) {
    if (B < 0 || N < 0 || K < 1 || !Hy || !scale_y || !z || !xprev || !neighbor_idx || !Cm || !Minv || !g || !Gz || !gprev || !Gy ||
        !m_out || !v_out || !h_out)
        return CRF_ERR_INVALID_ARG;
    if (B * N == 0) return CRF_OK;
    mf::StepArgs a{};
    a.Hy = Hy; a.scale_y = scale_y; a.z = z; a.xprev = xprev; a.nbr = neighbor_idx; a.Cm = Cm; a.Minv = Minv;
    a.total = B * N; a.N = N; a.K = K;
    a.g = g; a.Gz = Gz; a.gz_acc = gz_acc; a.gprev = gprev; a.Gy = Gy; a.m_out = m_out; a.v_out = v_out; a.h_out = h_out;
    return mf::dispatch_f(F, [&](auto f) {
        constexpr int FF = decltype(f)::value;
        constexpr int PPW = 32 / (FF / 4);
        const int64_t warps = ceil_div(a.total, PPW);
        if constexpr (FF <= 16) {
            if (K == 16) {      // the reference's neighbourhood size everywhere (kernel_size = 16): single-gather register kernel
                mf::step_bwd_reg_kernel<FF, 15><<<(unsigned)ceil_div(warps, 4), 128, 0, (cudaStream_t)stream>>>(a);
                CRF_LAUNCH_CHECK();
                return CRF_OK;
            }
        }
        mf::step_bwd_kernel<FF><<<(unsigned)ceil_div(warps, 8), 256, 0, (cudaStream_t)stream>>>(a);
        CRF_LAUNCH_CHECK();
        return CRF_OK;
    });
}

}  // extern "C"
