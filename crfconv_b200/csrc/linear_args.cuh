// Argument blocks shared by the generic (linear.cu) and fast-path (linear2.cu) Linear kernels.
#pragma once
#include <cstdint>

#include "fused_common.cuh"

namespace crf {
namespace lin {

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

// fast-path launchers (linear2.cu); return true when the shape was handled
bool try_fwd2(const FwdArgs& a, int precision, cudaStream_t st, int* rc);
bool try_dgrad2(const DgradArgs& a, int precision, cudaStream_t st, int* rc);
bool try_wgrad2(const WgradArgs& a, int precision, cudaStream_t st, int* rc);
// tcgen05 / TMEM forward (linear3.cu)
bool try_fwd3(const FwdArgs& a, int precision, cudaStream_t st, int* rc);
bool try_wgrad3(const WgradArgs& a, int precision, cudaStream_t st, int* rc);   // linear3w.cu
bool try_dgrad3(const DgradArgs& a, int precision, cudaStream_t st, int* rc);   // linear3d.cu
// input and weight gradient in one pass (linear3b.cu); needs dW and at least one of dX1 / dX2
bool try_bwd3(const DgradArgs& d, const WgradArgs& w, int precision, cudaStream_t st, int* rc);
// narrow layers over many rows: operands straight from global memory in fragment order (linear_direct.cu)
bool try_wgrad_direct(const WgradArgs& a, cudaStream_t st, int* rc);
bool try_upproj_fwd(const FwdArgs& a, cudaStream_t st, int* rc);      // narrow input → wide output (output-bound streams)
bool try_upproj_dgrad(const DgradArgs& a, cudaStream_t st, int* rc);
// few rows, wide channels (deep levels): 32-row tiles with register prefetch (linear_small.cu)
bool try_fwd_small(const FwdArgs& a, cudaStream_t st, int* rc);
bool try_dgrad_small(const DgradArgs& a, cudaStream_t st, int* rc);
bool try_wgrad_rows(WgradArgs a, cudaStream_t st, int* rc);
// CUDA-core kernels for hidden-width layers (linear_narrow.cu); w == nullptr ⇒ dgrad only
bool try_narrow_fwd(const FwdArgs& a, cudaStream_t st, int* rc);
bool try_narrow_bwd(const DgradArgs& d, const WgradArgs* w, cudaStream_t st, int* rc);

}  // namespace lin
}  // namespace crf
