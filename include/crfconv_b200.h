/* crfconv_b200 — C ABI of the B200 (sm_100a) hot path of CRFConv.
 *
 * Plain pointers and sizes only: no torch, numpy or C++ types cross this boundary.  Every entry point returns an
 * `int` status (0 = ok, <0 = CRF_ERR_* argument / support errors, >0 = cudaError_t) and never throws.
 * "device" pointers are CUDA device memory of the current device; `stream` is a cudaStream_t passed as void*
 * (NULL = legacy default stream).  Device entry points are stream-ordered and do not synchronise unless stated.
 * Each declaration cites the reference interface it stands in for (paths relative to the reference repository
 * yangfei1223/CRFConv).  INTEGRATION.md shows the binding a reference maintainer would add.
 */
#ifndef CRFCONV_B200_H_
#define CRFCONV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRFCONV_OK 0
#define CRFCONV_ERR_INVALID_ARG (-1)
#define CRFCONV_ERR_WORKSPACE (-2)   /* workspace_bytes smaller than the matching *_workspace_bytes() */
#define CRFCONV_ERR_UNSUPPORTED (-3) /* e.g. K > 1024, dim != 3 */
#define CRFCONV_ERR_NO_DEVICE (-4)

int crfconv_abi_version(void);
/* Static string for a status code returned by any function below. */
const char* crfconv_status_string(int status);

/* ------------------------------------------------------------------------------------------------- kNN
 * Replaces utils/nearest_neighbors/knn_.h:4-19 (cpp_knn, cpp_knn_omp, cpp_knn_batch, cpp_knn_batch_omp) and their
 * Cython callers knn.pyx:33-109.  Exact K nearest neighbours, squared L2 in f32 with nanoflann's operation order
 * (nanoflann.hpp:343-346), ascending (distance, index).  dim is fixed to 3.  K <= 1024 (passes of 32).  If K > npts the trailing
 * slots hold 0 (the observable behaviour of cpp_knn_omp, knn_.cxx:59-67).                                      */

size_t crfconv_knn_workspace_bytes(int64_t batch_size, int64_t npts, int64_t nqueries, int64_t K);

/* Device pointers.  pts [B,npts,3] f32, queries [B,nqueries,3] f32, out_idx [B,nqueries,K] i64. */
int crfconv_knn_batch(const float* pts, int64_t batch_size, int64_t npts, const float* queries, int64_t nqueries,
                      int64_t K, int64_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);

/* HOST pointers — the drop-in for `void cpp_knn_batch(const float* batch_data, size_t batch_size, size_t npts,
 * size_t dim, const float* queries, size_t nqueries, size_t K, long* batch_indices)` (knn_.h:13-15) and, with
 * batch_size = 1, for cpp_knn (knn_.h:4-6): copies to the device, searches, copies back, synchronises. dim must be 3. */
int crfconv_cpp_knn_batch(const float* batch_data, size_t batch_size, size_t npts, size_t dim, const float* queries,
                          size_t nqueries, size_t K, int64_t* batch_indices);

/* Coverage sampler — replaces cpp_knn_batch_distance_pick / _omp (utils/nearest_neighbors/knn_.h:21-27, knn_.cxx:138-271) and
 * knn.pyx:111-149: nqueries times per cloud, pick uniformly (std::mt19937 draw % count) among the points whose coverage counter
 * is at the current minimum level, take its K nearest neighbours, bump their counters (+1; +100 for the picked point).  The
 * reference seeds the generator with time(0); here the seed is an argument, and the single RNG stream of the reference's serial
 * loop (one draw per query, clouds in order) is reproduced.  K <= 32. */
size_t crfconv_knn_distance_pick_workspace_bytes(int64_t batch_size, int64_t npts);
/* Device pointers.  pts [B,npts,3] f32 -> out_idx [B,nqueries,K] i64, out_queries [B,nqueries,3] f32 (the picked points). */
int crfconv_knn_batch_distance_pick(const float* pts, int64_t batch_size, int64_t npts, int64_t nqueries, int64_t K, uint32_t seed,
                                    int64_t* out_idx, float* out_queries, void* workspace, size_t workspace_bytes, void* stream);
/* HOST pointers: the reference's C signature (knn_.h:21-23) plus the seed. */
int crfconv_cpp_knn_batch_distance_pick(const float* batch_data, size_t batch_size, size_t npts, size_t dim, float* batch_queries,
                                        size_t nqueries, size_t K, int64_t* batch_indices, uint32_t seed);

/* Radius search on the kNN grid (device pointers): per query the up-to-K smallest indices of the support points within distance r,
 * ascending, padded with -1 — torch_cluster.radius(x, y, r, max_num_neighbors = K), the graph builder of
 * models/continuous_crf_conv.py:52, models/discrete_crf_conv.py:44 and models/point_conv.py:150,180 (third party; semantics
 * restated).  Workspace: crfconv_knn_workspace_bytes. */
int crfconv_radius_batch(const float* pts, int64_t batch_size, int64_t npts, const float* queries, int64_t nqueries, float r, int64_t K,
                         int64_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------- grid subsampling
 * Replaces grid_subsampling() (utils/cpp_wrappers/cpp_subsampling/grid_subsampling/grid_subsampling.h:84-91,
 * grid_subsampling.cpp:5-106) and the array handling of wrapper.cpp:58-286.  Barycentre per voxel, mean feature,
 * plurality label; f32 sums in original point order (bit-exact).  order: 0 = ascending voxel key,
 * 1 = the reference's row order (libstdc++ unordered_map iteration order, replayed on the host).
 * Outputs must hold N rows; *M_out receives the number of occupied voxels.  Synchronises (M is data dependent). */

size_t crfconv_grid_subsample_workspace_bytes(int64_t N, int64_t fdim, int64_t ldim);

/* Device pointers.  features / classes / out_keys may be NULL (with fdim / ldim = 0). */
int crfconv_grid_subsample(const float* points, int64_t N, const float* features, int64_t fdim, const int32_t* classes,
                           int64_t ldim, float sampleDl, int order, float* out_points, float* out_features,
                           int32_t* out_classes, unsigned long long* out_keys, int64_t* M_out, void* workspace,
                           size_t workspace_bytes, void* stream);

/* HOST pointers (what wrapper.cpp:205-229 does with its numpy buffers). */
int crfconv_grid_subsample_host(const float* points, int64_t N, const float* features, int64_t fdim,
                                const int32_t* classes, int64_t ldim, float sampleDl, int order, float* out_points,
                                float* out_features, int32_t* out_classes, int64_t* M_out);

/* ------------------------------------------------------------- Linear + BatchNorm + LeakyReLU chains (MLP)
 * Replaces models/common.py:26-40 (MLP = nn.Linear(bias = not bn) → FastBatchNorm1d → activation) as it is used by
 * models/continuous_crf_conv_big.py:20-29 and models/point_conv_big.py:20-23,65-70.  All pointers are device
 * pointers, tensors are row-major [rows, channels] f32.  precision: 0 = 3xTF32 (fp32-grade), 1 = one TF32 pass, 2 = one bf16
 * pass in the persistent kernels (one TF32 pass elsewhere); any other value is refused with CRF_ERR_INVALID_ARG.  */

/* Kernel selection knob for tests / experiments: -1 = default rule (persistent bf16x3 kernels for large row counts,
 * generic 3xTF32 kernels otherwise), 0 = generic only, 1 = fast whenever the shape allows.  Returns the previous mode. */
int crfconv_set_fast_path(int mode);

#define CRFCONV_STAT_SLOTS 64 /* Σ/Σ² buffers (`stats`, `sums`) are [CRFCONV_STAT_SLOTS][2·C] floats (per-slot partials of <= 4 CTAs; summed in f64 by the finalize calls), zero-initialised by the caller */
#define CRFCONV_GRAD_SLOTS 32

/* Y[M,Cout] = [ lrelu(X1*scale1 + shift1, slope1) | X2 ] · Wᵀ (+ bias).  scale1 == NULL ⇒ X1 is used as is.
 * idx1 != NULL ⇒ X1 rows are gathered: source row of output row m is (m / rows_dst) * rows_src + idx1[m]
 * (point_conv_big.py:97-101).  stats != NULL ⇒ Σ_rows Y and Σ_rows Y² are accumulated into the slotted
 * partial buffer stats[CRFCONV_STAT_SLOTS][2·Cout] (CTA b adds into slot b % SLOTS); crfconv_bn_finalize_fwd sums the slots. */
int crfconv_linear_fwd(const float* X1, int C1, const float* scale1, const float* shift1, float slope1, const int64_t* idx1,
                       int64_t rows_dst, int64_t rows_src, const float* X2, int C2, const float* W, const float* bias, float* Y,
                       float* stats, int64_t M, int Cout, int precision, void* stream);

/* nn.BatchNorm1d bookkeeping (momentum, eps, biased variance for normalisation, unbiased for running_var).
 * training: scale = γ·istd, shift = β − μ·scale from Σ/Σ², running stats updated in place (may be NULL);
 * eval: from running statistics.  mean / invstd (saved for backward) may be NULL. */
int crfconv_bn_finalize_fwd(const float* stats, int64_t count, const float* gamma, const float* beta, float eps, float momentum,
                            int training, float* running_mean, float* running_var, float* scale, float* shift, float* mean,
                            float* invstd, int C, void* stream);

/* Y = lrelu(H*scale + shift (+ R), slope);  C % 4 == 0.  R (residual, point_conv_big.py:88) may be NULL. */
int crfconv_bn_act_fwd(const float* H, const float* scale, const float* shift, const float* R, float slope, float* Y, int64_t M,
                       int C, void* stream);

/* BatchNorm backward reductions into sums[CRFCONV_STAT_SLOTS][2·C]: [0:C] += Σ dV, [C:2C] += Σ dV·Ĥ, dV = dY·lrelu'(pre), Ĥ = (H−mean)·invstd,
 * pre = act_ref ? act_ref : H*scale+shift. */
int crfconv_bn_bwd_reduce(const float* dY, const float* H, const float* act_ref, const float* scale, const float* shift,
                          const float* mean, const float* invstd, float slope, float* sums, int64_t M, int C, void* stream);

/* Sums the slots: k1 = Σ dV / count, k2 = Σ dV·Ĥ / count; dgamma += Σ dV·Ĥ, dbeta += Σ dV (either may be NULL). */
int crfconv_bn_finalize_bwd(const float* sums, int64_t count, float* k1, float* k2, float* dgamma, float* dbeta, int C, void* stream);

/* Backward of crfconv_linear_fwd.  dY is the gradient wrt the layer's activation output; the BN(+LeakyReLU) backward
 * dH = scale·(dV − k1 − Ĥ·k2) is applied on the fly (scale == NULL ⇒ no BN, dH = dY).  Produces dX1 [M,C1] / dX2 [M,C2]
 * (gradients wrt the post-prologue inputs; NULL ⇒ skipped; acc ⇒ +=), dW [Cout,C1+C2] += dHᵀ·[prologue(X1)|X2],
 * dbias += Σ dH (NULL ⇒ skipped).  dW_scratch (optional): CRFCONV_GRAD_SLOTS slots of zero-initialised floats (pitch Cout·(C1+C2), or dW_scratch_stride); when given,
 * CTAs accumulate into per-slot partial copies that a follow-up kernel sums into dW (same-address atomics serialise in L2). */
int crfconv_linear_bwd(const float* dY, const float* H, const float* act_ref, const float* scale, const float* shift,
                       const float* mean, const float* invstd, const float* k1, const float* k2, float slope,
                       const float* X1, int C1, const float* scale1, const float* shift1, float slope1, const int64_t* idx1,
                       int64_t rows_dst, int64_t rows_src, const float* X2, int C2, const float* W, float* dX1, int acc1,
                       float* dX2, int acc2, float* dW, float* dbias, float* dW_scratch, int64_t dW_scratch_stride, int64_t M, int Cout,
                       int precision, void* stream);
/* Number of kernels the calling thread's last crfconv_linear_bwd call launched (input and weight gradient may share one). */
int crfconv_linear_bwd_launches(void);
/* dW[i] += Σ_slots scratch[slot·stride + i] for i < n.  With dW_scratch_stride > 0 crfconv_linear_bwd only accumulates into the
 * slots (slot pitch = stride floats) and the caller folds all layers that share one flat gradient layout with ONE call here. */
int crfconv_grad_slots_reduce(const float* scratch, float* dW, int64_t n, int64_t stride, void* stream);

/* ------------------------------------------------------------------------ continuous-CRF mean-field
 * Replaces the body of ContinuousGaussianCRFConv.forward, models/continuous_crf_conv_big.py:56-72 (and its autograd
 * backward).  F = hidden channels ∈ {4,8,16,32,64}; neighbor_idx [B,N,K] i64 local to each cloud, column 0 skipped
 * (:45-47); up_idx [B,N,1] i64 into the Nc coarse points of the same cloud (:60). */

/* Cm = cᵀc, Minv = (I + Cm)^{-1} (:66,72).  scratch: 3·F·F doubles. */
int crfconv_crf_compat_fwd(const float* c, float* Cm, float* Minv, double* scratch, int F, void* stream);
/* Gc += c·(G + Gᵀ), G = GC − Minvᵀ·GM·Minvᵀ. */
int crfconv_crf_compat_bwd(const float* c, const float* Minv, const float* GC, const float* GM, float* Gc, double* scratch, int F,
                           void* stream);
/* z[B·N,F] = (Hu*scale + shift)[up_idx]  — unary_nn's last BatchNorm fused into the nearest-coarse upsample. */
int crfconv_crf_upsample_fwd(const float* Hu, const float* scale, const float* shift, const int64_t* up_idx, float* z, int64_t B,
                             int64_t N, int64_t Nc, int F, void* stream);
/* Gu[B·Nc,F] += (Gz + G0) scattered through up_idx (G0 may be NULL). */
int crfconv_crf_upsample_bwd(const float* Gz, const float* G0, const int64_t* up_idx, float* Gu, int64_t B, int64_t N, int64_t Nc,
                             int F, void* stream);
/* xout = (z + (S·xprev)·Cm)·Minv, S = softmax_k(−‖y_i − y_j‖²), y = Hy*scale_y (+shift, which cancels). */
int crfconv_crf_step_fwd(const float* Hy, const float* scale_y, const float* z, const float* xprev, const int64_t* neighbor_idx,
                         const float* Cm, const float* Minv, float* xout, int64_t B, int64_t N, int K, int F, void* stream);
/* Backward of one step given g = dL/dxout: Gz = (gz_acc ? Gz : 0) + g·Minvᵀ (=h); gprev += Σ_i s_ij·(h_i·Cmᵀ) (zero-initialised by caller);
 * Gy += gradient through the distances wrt y; m_out / v_out / h_out rows feed GC = mᵀh and GM = vᵀg. */
int crfconv_crf_step_bwd(const float* Hy, const float* scale_y, const float* z, const float* xprev, const int64_t* neighbor_idx,
                         const float* Cm, const float* Minv, const float* g, float* Gz, float* gprev, float* Gy, float* m_out,
                         float* v_out, float* h_out, int gz_acc, int64_t B, int64_t N, int K, int F, void* stream);

/* --------------------------------------------- layer-specialised ("fused") kernels of the dense CRF layer, F = 16
 * The same arithmetic as the entry points above for models/continuous_crf_conv_big.py:20-29,56-78, cut at the BatchNorm
 * boundaries so that each boundary costs ONE streaming pass: the BatchNorm bookkeeping (crfconv_bn_finalize_fwd / _bwd) runs in
 * the tail of the producing kernel (last CTA to finish), the backward sums of the NEXT BatchNorm are emitted by the kernel that
 * produces its upstream gradient, and out_nn's backward (:74) collapses to a per-point affine map (see csrc/crf_fused.cu).
 * `part` scratches hold per-CTA partial sums (no initialisation needed unless stated); every `counter` points at
 * crfconv_fused_counter_ints() zeroed uint32 (two-level arrival tickets) that the kernel leaves zero.  Weight gradients go to CRFCONV_GRAD_SLOTS zero-initialised partial slots (slot_stride floats
 * apart) that crfconv_grad_slots_reduce folds. */

int crfconv_fused_max_parts(void);        /* largest grid of a kernel with an arrival tail */
int crfconv_fused_part_floats(void);      /* floats of every `part` scratch argument (per-CTA rows + per-group rows) */
int crfconv_fused_counter_ints(void);     /* uint32 per `counter` argument */
int crfconv_out_bwd_part_floats(void);    /* floats of crfconv_out16_bwd's `part` (zero-initialised) */

/* H[M,16] = act(X[M,Cin])·Wᵀ + BatchNorm finalize of H (MLP(Cin,16), common.py:26-40).  Cin ∈ {64,128}: X raw; Cin = 16: X is the
 * previous layer's pre-BN output and pscale/pshift/pslope its BN affine + LeakyReLU. */
int crfconv_lin16_fwd(const float* X, int Cin, const float* W, const float* pscale, const float* pshift, float pslope, float* Y, int64_t M,
                      float* part, unsigned int* counter, const float* gamma, const float* beta, float* running_mean, float* running_var,
                      float eps, float momentum, float* scale, float* shift, float* mean, float* invstd, void* stream);
/* H[M,Cout] = X[M,16]·Wᵀ + BatchNorm finalize of H (MLP(16,Cout), Cout = 64: out_nn).  stats [CRFCONV_STAT_SLOTS][2·Cout] zeroed. */
int crfconv_up16_fwd(const float* X, const float* W, int Cout, float* Y, int64_t M, float* stats, unsigned int* counter, const float* gamma,
                     const float* beta, float* running_mean, float* running_var, float eps, float momentum, float* scale, float* shift,
                     float* mean, float* invstd, void* stream);
/* crfconv_linear_fwd (no gather, no bias) + BatchNorm finalize of its output; stats [CRFCONV_STAT_SLOTS][2·Cout] zeroed. */
int crfconv_linear_fwd_bn(const float* X1, int C1, const float* scale1, const float* shift1, float slope1, const float* X2, int C2,
                          const float* W, float* Y, float* stats, int64_t M, int Cout, int precision, unsigned int* counter,
                          const float* gamma, const float* beta, float* running_mean, float* running_var, float eps, float momentum,
                          float* scale, float* shift, float* mean, float* invstd, void* stream);
/* crfconv_bn_bwd_reduce + crfconv_bn_finalize_bwd (one launch for C = 64). */
int crfconv_bn_bwd_reduce_fin(const float* dY, const float* H, const float* act_ref, const float* scale, const float* shift,
                              const float* mean, const float* invstd, float slope, float* sums, int64_t M, int C, unsigned int* counter,
                              float* k1, float* k2, float* dgamma, float* dbeta, void* stream);
/* Backward of y = BN2(lrelu(BN1(H1))·W2ᵀ) given dY: dV1 = (dH2·W2)⊙lrelu'(BN1(H1)), dW2 slots, BN1's backward constants. */
int crfconv_mid16_bwd(const float* dY, const float* H2, const float* sc2, const float* mu2, const float* is2, const float* k1_2,
                      const float* k2_2, const float* H1, const float* sc1, const float* sh1, const float* mu1, const float* is1,
                      float slope1, const float* W2, float* dV1, float* dW2, int64_t slot_stride, int64_t M, float* part,
                      unsigned int* counter, float* k1_1, float* k2_1, float* dgamma1, float* dbeta1, void* stream);
/* dX[M,Cin] (= or +=) BNbwd(dV1,H1)·W1 ;  dW1 slots += BNbwd(dV1,H1)ᵀ·X.  Cin ∈ {64,128}. */
int crfconv_in16_dgrad(const float* dV1, const float* H1, const float* sc1, const float* mu1, const float* is1, const float* k1,
                       const float* k2, const float* W1, int Cin, float* dX, int accumulate, int64_t M, void* stream);
int crfconv_in16_wgrad(const float* dV1, const float* H1, const float* sc1, const float* mu1, const float* is1, const float* k1,
                       const float* k2, const float* X, int Cin, float* dW, int64_t slot_stride, int64_t M, void* stream);
/* out_nn = MLP(16,64) backward in one pass over dO: T = W3ᵀ·(sc3⊙dv3), k1/k2, dγ/dβ, dW3 +=, and Q[16,16], a0[16] with
 * dL/dx_i = T_i − a0 − Q·x_i. */
int crfconv_out16_bwd(const float* dO, const float* H3, const float* sc3, const float* sh3, const float* mu3, const float* is3,
                      float slope3, const float* X, const float* W3, float* T, int64_t M, float* part, unsigned int* counter,
                      float* k1, float* k2, float* dgamma, float* dbeta, float* dW3, float* Q, float* a0, void* stream);
/* crfconv_crf_step_bwd for F = K = 16 with GC/GM accumulated in-kernel (slots), the out_nn correction g ← g − a0 − Q·xT applied on
 * the fly (Q may be NULL) and the BatchNorm-backward constants of the y layer (gamma_y = its weight) finalized on the last
 * launch (finalize != 0).  ysum: 8·16 zeroed floats shared by all steps of one backward. */
int crfconv_crf_step_bwd_fused(const float* Hy, const float* sc_y, const float* z, const float* xprev, const int64_t* neighbor_idx,
                               const float* Cm, const float* Minv, const float* g, const float* xT, const float* Q, const float* a0,
                               float* Gz, int gz_acc, float* gprev, float* Gy, float* GC, float* GM, int64_t slot_stride,
                               float* ysum, int64_t B, int64_t N, int K, int F, int finalize, unsigned int* counter,
                               const float* gamma_y, float* k1, float* k2, float* dgamma, float* dbeta, void* stream);
/* crfconv_crf_upsample_bwd for F = 16 + the BatchNorm-backward constants of unary_nn[1] (Hu = its pre-BN output). */
int crfconv_crf_upsample_bwd_fused(const float* Gz, const float* G0, const int64_t* up_idx, const float* Hu, const float* mu,
                                   const float* is, float* Gu, int64_t B, int64_t N, int64_t Nc, float* part, unsigned int* counter,
                                   float* k1, float* k2, float* dgamma, float* dbeta, void* stream);

/* ------------------------------------------------------- neighbour gather / point-conv aggregation
 * Replaces PointConv.gather_neighbors / _compute_weights / forward (models/point_conv_big.py:25-58),
 * ResNetBBlock.max_pooling (:74-77) and the backward of Upsampling.upsampling (:97-101).  idx [B,Nq,K] i64 indexes the
 * Ns support points of the same cloud.  C % 4 == 0. */

/* rel[(b·Nq+i)·K+k, 0:3] = centres[b,i] − support[b, idx[b,i,k]]   (point_conv_big.py:40) */
int crfconv_relpos(const float* support, const float* centres, const int64_t* idx, float* rel, int64_t B, int64_t Ns, int64_t Nq, int K,
                   void* stream);
/* out[b,i,:] = Σ_k (H2[e,:]*scale + shift) ⊙ x[b, idx[b,i,k], :]   — (w * x).sum(2) with weight_nn's last BatchNorm fused (:56-57) */
int crfconv_pointconv_aggregate_fwd(const float* x, const float* H2, const float* scale, const float* shift, const int64_t* idx, float* out,
                                    int64_t B, int64_t Ns, int64_t Nq, int K, int C, void* stream);
/* dWgt[e,:] = g[b,i,:] ⊙ x[src,:];  dx[src,:] += w[e,:] ⊙ g[b,i,:]  (dx may be NULL; zero-initialised by the caller) */
int crfconv_pointconv_aggregate_bwd(const float* x, const float* H2, const float* scale, const float* shift, const int64_t* idx,
                                    const float* g, float* dWgt, float* dx, int64_t B, int64_t Ns, int64_t Nq, int K, int C, void* stream);
/* out[b,i,:] = max_k x[b, idx[b,i,k], :];  arg = flat source row of the first maximum (for the backward scatter) */
int crfconv_gather_max_fwd(const float* x, const int64_t* idx, float* out, int32_t* arg, int64_t B, int64_t Ns, int64_t Nq, int K, int C,
                           void* stream);
int crfconv_gather_max_bwd(const float* g, const int32_t* arg, float* dx, int64_t rows, int C, void* stream);
/* dS = g · (out > 0 ? 1 : slope)  — backward of F.leaky_relu(x + residual) (point_conv_big.py:88) */
int crfconv_lrelu_bwd(const float* g, const float* out, float slope, float* dS, int64_t numel, void* stream);
/* y += x */
int crfconv_add_inplace(float* y, const float* x, int64_t numel, void* stream);
/* dst[b·Ns + idx[b,m], :] += src[b·Nq + m, :]  — backward of a K=1 row gather (point_conv_big.py:97-101) */
int crfconv_scatter_add_rows(const float* src, const int64_t* idx, float* dst, int64_t B, int64_t Nq, int64_t Ns, int C, void* stream);

/* ------------------------------------------------------- graph builders and edge-list message passing (PyG-API family)
 * models/continuous_crf_conv.py:9-133, models/discrete_crf_conv.py:11-63, models/point_conv.py:140-195.  All device pointers.
 * Edge lists are grouped by TARGET node: node i owns edges [eptr[i], eptr[i+1]), col[e] = source node. */

/* Farthest point sampling per cloud (ptr = CSR offsets of the clouds in pos [ptr[B],3]); out gets GLOBAL indices; dist_ws: ptr[B] floats. */
int crfconv_fps(const float* pos, const int64_t* ptr, int64_t B, const int64_t* nsample, const int64_t* start, int64_t* out,
                const int64_t* out_ptr, float* dist_ws, void* stream);
/* s[e] = softmax over the edges of each target of -||y_i - y_col||^2 (+1e-16 in the denominator, torch_geometric.utils.softmax). */
int crfconv_edge_softmax_fwd(const float* y, const int64_t* eptr, const int64_t* col, float* s, int64_t N, int C, void* stream);
int crfconv_edge_softmax_bwd(const float* y, const int64_t* eptr, const int64_t* col, const float* s, const float* ds, float* dy, int64_t N,
                             int C, void* stream);
/* w[e] = sum_k Wk[k] exp(-||f_k[col] - f_k[row]||^2), f [N, Kk*H]; g [E, Kk] saves the exponentials (discrete_crf_conv.py:49-56). */
int crfconv_edge_gauss_fwd(const float* f, const int64_t* eptr, const int64_t* col, const float* Wk, float* w, float* g, int64_t N, int Kk,
                           int H, void* stream);
int crfconv_edge_gauss_bwd(const float* f, const int64_t* eptr, const int64_t* col, const float* Wk, const float* g, const float* dw,
                           float* df, float* dWk, int64_t N, int Kk, int H, void* stream);
/* out[i,:] = sum over the edges of i of w[e] x[col[e],:]  (scatter_add of weighted messages) and its backward (dw / dx may be NULL). */
int crfconv_spmm_fwd(const float* x, const int64_t* eptr, const int64_t* col, const float* w, float* out, int64_t N, int C, void* stream);
int crfconv_spmm_bwd(const float* x, const int64_t* eptr, const int64_t* col, const float* w, const float* g, float* dw, float* dx, int64_t N,
                     int C, void* stream);

/* ------------------------------------------------------- PointConv without per-edge tensors (hidden width D = 8 / 16: levels 0 and 1)
 * models/point_conv_big.py:8-58.  out_i = Σ_k BN2(W2·lrelu(BN1(W1·r_ik))) ⊙ x_j with the 3→D→D edge MLP recomputed from r in every pass;
 * only sums cross kernels (csrc/pointconv_fused.cu).  All scratch buffers are [CRFCONV_STAT_SLOTS][n] zero-initialised floats. */
int crfconv_pcf_supported(int D);
int crfconv_pcf_fwd_scratch_floats(int D);
int crfconv_pcf_bwd_scratch_floats(int D);
/* rel [B·Nq·K, 3] = centre − support[idx] and mom [SLOTS][9] = Σr | Σrrᵀ (upper triangle) */
int crfconv_pcf_relpos_moments(const float* support, const float* centres, const int64_t* idx, float* rel, float* mom, int64_t B, int64_t Ns,
                               int64_t Nq, int K, void* stream);
/* Σh1, Σh1² of h1 = W1·r from the moments → slot 0 of stats1 [SLOTS][2D] (then crfconv_bn_finalize_fwd with count = B·Nq·K) */
int crfconv_pcf_stats1(const float* mom, const float* W1, float* stats1, int D, void* stream);
/* P_i = Σ_k h2 ⊙ x_j, Q_i = Σ_k x_j; stats2 [SLOTS][2D] += Σh2 | Σh2²; asum [SLOTS][D + D·D] += Σa1 | Σa1a1ᵀ (D = 8: upper triangle) */
int crfconv_pcf_fwd(const float* x, const float* rel, const int64_t* idx, const float* W1, const float* W2, const float* sc1, const float* sh1,
                    float slope1, float* P, float* Q, float* stats2, float* asum, int64_t B, int64_t Ns, int64_t Nq, int K, int D, void* stream);
/* out = sc2 ⊙ P + sh2 ⊙ Q */
int crfconv_pcf_out(const float* P, const float* Q, const float* sc2, const float* sh2, float* out, int64_t rows, int D, void* stream);
/* dw = g_i ⊙ x_j: sums2 [SLOTS][2D] += Σdw | Σdw·ĥ2, mdw [SLOTS][D·D] += Σ dw a1ᵀ; dx[j] += w ⊙ g_i (dx zero-initialised, may be NULL) */
int crfconv_pcf_bwd1(const float* x, const float* rel, const int64_t* idx, const float* g, const float* W1, const float* W2, const float* sc1,
                     const float* sh1, float slope1, const float* sc2, const float* sh2, const float* mu2, const float* is2, float* dx,
                     float* sums2, float* mdw, int64_t B, int64_t Ns, int64_t Nq, int K, int D, void* stream);
/* dv1 = (W2ᵀ·BN2'(dw)) ⊙ lrelu': sums1 [SLOTS][2D] += Σdv1 | Σdv1·ĥ1, s1 [SLOTS][3D] += Σ dv1 rᵀ   (k1b / k2b: BN2 backward constants) */
int crfconv_pcf_bwd2(const float* x, const float* rel, const int64_t* idx, const float* g, const float* W1, const float* W2, const float* sc1,
                     const float* sh1, float slope1, const float* mu1, const float* is1, const float* sc2, const float* mu2, const float* is2,
                     const float* k1b, const float* k2b, float* sums1, float* s1, int64_t B, int64_t Ns, int64_t Nq, int K, int D, void* stream);
/* dW1 [D,3] += , dW2 [D,D] += from the sums and both BatchNorms' finalized backward constants */
int crfconv_pcf_param_grads(const float* mom, const float* asum, const float* mdw, const float* s1, const float* W1, const float* W2,
                            const float* sc1, const float* mu1, const float* is1, const float* k1a, const float* k2a, const float* sc2,
                            const float* mu2, const float* is2, const float* k1b, const float* k2b, float* dW1, float* dW2, int D, void* stream);

/* ------------------------------------------------------- training criterion (trainval.py:66-70,100-104: class-weighted cross entropy)
 * sums[0] += Σ w[t]·(logsumexp(x) − x[t]), sums[1] += Σ w[t] over the rows whose target != ignore_index (two zeroed doubles); C <= 64.
 * The backward recomputes the softmax: dlogits = g·w[t]·(softmax − onehot), g = *gout (mean == 0) or *gout / sums[1] (mean != 0). */
int crfconv_cross_entropy_fwd(const float* logits, const int64_t* target, const float* weight, int64_t M, int C, int64_t ignore_index,
                              double* sums, void* stream);
int crfconv_cross_entropy_bwd(const float* logits, const int64_t* target, const float* weight, int64_t M, int C, int64_t ignore_index,
                              const double* sums, const float* gout, int mean, float* dlogits, void* stream);

/* ------------------------------------------------------- host staging of index tensors (the PCIe leg of an end-to-end step)
 * The reference hands neighbour / up-sampling indices over as int64 (knn.pyx:58,100 `np.zeros(..., dtype=np.int64)`; models/
 * continuous_crf_conv_big.py:40-44 gathers with them), i.e. 8 bytes per index whose value is < npts.  crfconv_pack_index_host narrows
 * `n` HOST int64 indices to `bits` (16 or 32) unsigned bits with `threads` host threads (out: HOST, n·bits/8 bytes, e.g. pinned memory);
 * CRFCONV_ERR_INVALID_ARG if any index is negative or does not fit — nothing is truncated silently.  crfconv_unpack_index widens the
 * packed DEVICE buffer back to the int64 DEVICE tensor the kernels read.  Values are bit-exact by construction. */
int crfconv_pack_index_host(const int64_t* idx, int64_t n, int bits, void* out, int threads);
int crfconv_unpack_index(const void* packed, int64_t n, int bits, int64_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CRFCONV_B200_H_ */
