// Argument blocks, device helpers and the launcher protocol shared by the Linear kernel families (linear*.cu).
#pragma once
#include <cstdint>

#include "fused_common.cuh"

namespace crf {
namespace lin {

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.0f ? v : v * slope; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct FwdArgs {
    const float* X1; int C1;                      // segment 1: [M, C1] (row-gathered through idx1 when given)
    const float* scale1; const float* shift1; float slope1;   // prologue of segment 1: lrelu(x*scale+shift); null = identity
    const int64_t* idx1; int64_t rows_dst; int64_t rows_src;  // gather: src row = (m / rows_dst) * rows_src + idx1[m]
    const float* X2; int C2;                      // segment 2: [M, C2] raw (may be null / 0)
    const float* W;                               // [Cout, C1 + C2] row-major (nn.Linear.weight)
    const float* bias;                            // [Cout] or null
    float* Y;                                     // [M, Cout]
    float* stats;                                 // [kStatSlots][2*Cout] partial Σ, Σ² over rows (or null)
    int64_t M; int Cout;
    cl::FwdFin fin;                               // optional: BatchNorm finalize by the last CTA (kernels that support it; part = stats)
};

// Per-channel description of a BatchNorm(+LeakyReLU) node for the on-the-fly backward transform.
struct BnBwd {
    const float* scale;    // γ·istd        (null ⇒ plain Linear output: dH = dY)
    const float* shift;    // β − μ·scale
    const float* mean;
    const float* invstd;
    const float* k1;       // mean over rows of dV
    const float* k2;       // mean over rows of dV·Ĥ
    const float* act_ref;  // [M, C] saved activation output whose sign selects the LeakyReLU branch (null ⇒ use V)
    float slope;           // 1 ⇒ no activation

    // Channel c's constants of dH = sc·dV + pz·H + pw, returned as (sc, sh, pz, pw):
    // pz = −sc·istd·k2, pw = −sc·k1 + sc·istd·k2·mean; the LeakyReLU branch of dV is selected by sc·H + sh.
    __device__ __forceinline__ float4 coef(int c) const {
        const float sc = __ldg(scale + c), sh = __ldg(shift + c), mu = __ldg(mean + c), is = __ldg(invstd + c);
        const float q1 = __ldg(k1 + c), q2 = __ldg(k2 + c);
        return make_float4(sc, sh, -sc * is * q2, -sc * q1 + sc * is * q2 * mu);
    }
};

struct DgradArgs {
    const float* dY; const float* H; BnBwd bn;    // upstream gradient wrt this layer's activation output, pre-BN output
    const float* W;                               // [Cout, C1 + C2]
    float* dX1; int C1; int acc1;                 // gradient wrt segment 1 input (post-prologue), [M, C1]; acc ⇒ +=
    float* dX2; int C2; int acc2;
    int64_t M; int Cout;
};

struct WgradArgs {
    const float* dY; const float* H; BnBwd bn;
    const float* X1; int C1; const float* scale1; const float* shift1; float slope1;
    const int64_t* idx1; int64_t rows_dst; int64_t rows_src;
    const float* X2; int C2;
    float* dW;            // [Cout, C1 + C2]
    float* dbias;         // [Cout] or null: += Σ_m dH
    int64_t M; int Cout;
    int64_t rows_per_cta;
    int64_t slot_stride;  // 0, or Cout·Ktot when dW points at [kGradSlots][Cout·Ktot] partial slots
};

// Launchers.  Each try_* returns kDeclined when the call is outside its family's shape range (the dispatch in linear.cu then
// tries the next family), else the status of its launch: CRF_OK or a cudaError_t.
constexpr int kDeclined = -1000;   // below every CRF_ERR_* code; cudaError_t values are >= 0

// Raises kernel's dynamic shared-memory limit to smem (when smem > 0), launches it and returns CRF_OK or the CUDA error.
template <typename... KArgs, typename... Args>
inline int launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaError_t e = cudaSuccess;
    if (smem > 0) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        kernel<<<grid, block, smem, st>>>(static_cast<KArgs>(args)...);
        e = cudaPeekAtLastError();
    }
    return e == cudaSuccess ? CRF_OK : (int)e;
}

// tcgen05 / TMEM (linear3*.cu): forward, weight gradient, input gradient
int try_fwd3(const FwdArgs& a, int precision, cudaStream_t st);
int try_wgrad3(const WgradArgs& a, int precision, cudaStream_t st);
int try_dgrad3(const DgradArgs& a, int precision, cudaStream_t st);
// input and weight gradient in one pass (linear3b.cu); needs dW and at least one of dX1 / dX2
int try_bwd3(const DgradArgs& d, const WgradArgs& w, int precision, cudaStream_t st);
// persistent cp.async kernels (linear2.cu)
int try_fwd2(const FwdArgs& a, int precision, cudaStream_t st);
int try_dgrad2(const DgradArgs& a, int precision, cudaStream_t st);
int try_wgrad2(const WgradArgs& a, int precision, cudaStream_t st);
// narrow layers over many rows: operands straight from global memory in fragment order (linear_direct.cu)
int try_wgrad_direct(const WgradArgs& a, cudaStream_t st);
int try_upproj_fwd(const FwdArgs& a, cudaStream_t st);      // narrow input → wide output (output-bound streams)
int try_upproj_dgrad(const DgradArgs& a, cudaStream_t st);
// few rows, wide channels (deep levels): 32-row tiles with register prefetch (linear_small.cu)
int try_fwd_small(const FwdArgs& a, cudaStream_t st);
int try_dgrad_small(const DgradArgs& a, cudaStream_t st);
int try_wgrad_rows(WgradArgs a, cudaStream_t st);
// CUDA-core kernels for hidden-width layers (linear_narrow.cu); w == nullptr ⇒ dgrad only
int try_narrow_fwd(const FwdArgs& a, cudaStream_t st);
int try_narrow_bwd(const DgradArgs& d, const WgradArgs* w, cudaStream_t st);

}  // namespace lin
}  // namespace crf
