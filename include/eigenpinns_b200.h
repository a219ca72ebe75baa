/* eigenpinns_b200.h — C ABI of the B200 (sm_100a) kernels behind the eigen-pinns hot path.
 *
 * The reference (bornexmachina/eigen-pinns) is pure Python and has no FFI of its own; the
 * boundary it exposes is the Python method surface of MultigridGNN / SimpleCorrector /
 * SpectralCorrector and the two sampler functions.  Every entry point below names the
 * reference lines whose arithmetic it replaces (paths under /root/reference/src).  The
 * Python host layer (eigen-pinns_b200/) binds these with ctypes; INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary
 *   - all array pointers are DEVICE pointers unless the function name ends in _host; the tiny
 *     parameter arrays `dims`, `lo` (voxel grid) and the layer tables of ep_tc_chain_fwd_bf16 are HOST arrays
 *   - one device and one stream per process are assumed by the cached launch configuration
 *     (SM count, opted-in shared-memory sizes, the gradient-norm scratch)
 *   - dense matrices are row-major with an explicit leading dimension (elements)
 *   - CSR: int32 rowptr[n+1], int32 col[nnz], fp32 val[nnz]; the *_f64 entries take fp64 val[nnz] and fp64
 *     dense operands (the notebook variants, which train in double)
 *   - every call takes the CUDA stream it is enqueued on (cudaStream_t as void*); nothing
 *     synchronises unless stated; no hidden allocation: workspaces are sized by *_workspace_bytes
 *   - return value: 0 = EP_OK, negative = error (see ep_status); ep_last_error_string()
 *     describes the last failure on the calling thread; nothing throws
 */
#ifndef EIGENPINNS_B200_H
#define EIGENPINNS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define EP_API __attribute__((visibility("default")))
#else
#define EP_API
#endif

typedef void* ep_stream_t;

enum ep_status {
  EP_OK = 0,
  EP_ERR_INVALID = -1,      /* bad argument (null pointer, negative size, misalignment) */
  EP_ERR_CUDA = -2,         /* a CUDA runtime call failed */
  EP_ERR_UNSUPPORTED = -3,  /* shape outside what the kernels are instantiated for */
  EP_ERR_WORKSPACE = -4     /* workspace too small */
};

/* ---- library ------------------------------------------------------------------------- */
EP_API int ep_version(void);                               /* 10000*major + 100*minor + patch */
EP_API const char* ep_last_error_string(void);
/* sm_count, compute capability of the current device; fails (EP_ERR_CUDA) without a GPU. */
EP_API int ep_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Knobs for experiments.  Key 1: SpMM persistent grid = value full-machine waves (1..64, default 4).
 * Keys 3 / 4: low / high 32 bits of the address of a device buffer of 64 x 8 uint64 (0 = off) that
 * ep_tc_chain_fwd_bf16 fills with clock64 stamps of its first CTA, 8 per (layer, slot) step.  Any other key returns
 * EP_ERR_INVALID. */
EP_API int ep_tune_set(int key, int value);

/* ---- sparse operators: torch.sparse.mm(K_t, U), torch.sparse.mm(M_t, U) ----------------
 * replaces multigrid_model.py:309-310 (loss), :126,:375 (normalisation), :403-404 (Rayleigh-
 * Ritz), :183-184 (features) and the autograd transposes behind :258.  The per-epoch
 * scipy->torch COO conversion of utils.py:14-20 (called at multigrid_model.py:306-307)
 * disappears: operators are converted to CSR fp32/int32 once and stay resident in HBM. */
/* Y = A X.  X: n_cols_of_A x k (ldx), Y: n_rows x k (ldy). */
EP_API int ep_spmm_csr_f32(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const float* val,
                    const float* X, int ldx, float* Y, int ldy, ep_stream_t stream);
/* YA = A X and YB = B X for two operators that share one sparsity pattern (FEM K and M):
 * each gathered row of X is read once for both products. */
EP_API int ep_spmm2_csr_f32(int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                     const float* valA, const float* valB, const float* X, int ldx,
                     float* YA, float* YB, int ldy, ep_stream_t stream);
/* Y = out_scale * (A XA + B XB + D)   (D may be NULL; out_scale_dev, a device scalar, overrides out_scale
 * when non-NULL so that a captured CUDA graph can follow the epoch-dependent scale ramp).  Backward of the eigen-loss:
 * U_bar = K^T KU_bar + M^T MU_bar + D (SURVEY Appendix A); pass the CSR of the transposes
 * (identical to K, M for the symmetric FEM / tufted operators). */
EP_API int ep_spmm2_sum_csr_f32(int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                         const float* valA, const float* valB, const float* XA, const float* XB,
                         int ldx, const float* D, int ldd, float out_scale, const float* out_scale_dev,
                         float* Y, int ldy, ep_stream_t stream);

/* fp64 forms of the three products above (same argument order, double in place of float; out_scale_dev is a
 * device double).  They serve the notebook variants in double precision: K U, M U of
 * scripts/simplified_loss.ipynb cell 0 and scripts/loss_with_rigid_body.ipynb cell 0 (torch.sparse.mm in fp64),
 * L u, M u of delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1, L corr of
 * delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4, and the transposed products of their backward. */
EP_API int ep_spmm_csr_f64(int n_rows, int k, const int32_t* rowptr, const int32_t* col, const double* val,
                    const double* X, int ldx, double* Y, int ldy, ep_stream_t stream);
EP_API int ep_spmm2_csr_f64(int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                     const double* valA, const double* valB, const double* X, int ldx,
                     double* YA, double* YB, int ldy, ep_stream_t stream);
EP_API int ep_spmm2_sum_csr_f64(int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                         const double* valA, const double* valB, const double* XA, const double* XB,
                         int ldx, const double* D, int ldd, double out_scale, const double* out_scale_dev,
                         double* Y, int ldy, ep_stream_t stream);

/* ---- corrector input: h = cat([x, agg], dim=1) -----------------------------------------
 * SimpleCorrector.forward, corrector_model.py:23-30: agg_i = (sum over edges (i<-j) of x_j) /
 * max(deg_i, 1), edges given as CSR over destination rows (rowptr/col), summed in edge order.
 * H: n x 2d (ldh >= 2d): H[:, :d] = x, H[:, d:] = agg. */
EP_API int ep_neighbor_mean_concat_f32(int n, int d, const int32_t* rowptr, const int32_t* col,
                                const float* x, int ldx, float* H, int ldh, ep_stream_t stream);
/* SpectralCorrector.forward, corrector_model.py:76-79: H = [x | A_norm x], A_norm as CSR. */
EP_API int ep_spmm_concat_f32(int n, int d, const int32_t* rowptr, const int32_t* col, const float* val,
                       const float* x, int ldx, float* H, int ldh, ep_stream_t stream);

/* ---- eigen-loss: multigrid_model.py:291-348 --------------------------------------------
 * Phase 1 (per level, per rank): column/Gram partial sums in fp64,
 *   out[0 .. k*k)        G[a*k+b]  = sum_i U[i,a] * MU[i,b]          (:321; diag = den of :313)
 *   out[k*k + 0k ..)     num[j]    = sum_i U[i,j] * KU[i,j]           (:313)
 *   out[k*k + 1k ..)     sKK[j]    = sum_i KU[i,j]^2
 *   out[k*k + 2k ..)     sKM[j]    = sum_i KU[i,j] * MU[i,j]
 *   out[k*k + 3k ..)     sMM[j]    = sum_i MU[i,j]^2
 *   out[k*k + 4k ..)     sMU[j]    = sum_i MU[i,j]                    (1^T M u_j, zero-mean term of the notebooks)
 * (the last three give sum_i (KU - lam MU)^2 of :317-318 without a second pass; num and these
 * three are accumulated in fp64 from the first product on - products of fp32 values are exact in
 * fp64 - so the expansion keeps ~9 digits when the residual is 1e-4 of |KU|, i.e. near convergence).  Partials of all ranks are summed
 * (allreduce) before phase 2.  Deterministic: fixed grid, fixed reduction order. */
EP_API size_t ep_eigen_partials_len(int k);                        /* k*k + 5*k doubles */
EP_API size_t ep_eigen_partials_workspace_bytes(int k);
EP_API int ep_eigen_partials_f32(int n, int k, const float* U, int ldu, const float* KU, const float* MU,
                          int ld, double* out, void* workspace, size_t workspace_bytes,
                          ep_stream_t stream);
/* fp64 inputs, same output layout, workspace size and k <= 128; every product and sum is fp64 (no fp32 stage).
 * The Gram matrices U^T K U and U^T M U of scripts/simplified_loss.ipynb cell 0 (UKU, UMU) and
 * scripts/loss_with_rigid_body.ipynb cell 0 (B and the Rayleigh matrix) in the notebooks' precision. */
EP_API int ep_eigen_partials_f64(int n, int k, const double* U, int ldu, const double* KU, const double* MU,
                          int ld, double* out, void* workspace, size_t workspace_bytes,
                          ep_stream_t stream);

/* Phase 2 (per level, one tiny launch): from the summed partials compute
 *   lam_j = num_j / (G_jj + 1e-12);  L_res = sum_j(sKK - 2 lam sKM + lam^2 sMM) / (n_global k);
 *   L_orth = sum_ab (G_ab - I_ab)^2 / k;  and for level 0 the eigenvalue terms of :326-348
 *   (trace = mean lam, order = sum relu(lam_j - lam_{j+1}), eigen = mean (lam - lam_target)^2).
 * and the two additive terms of the notebook variants (SURVEY 8a-bis; weight 0 in src/):
 *   mean   = sum_{j>=1} (1^T M u_j)^2 / (k - 1)       multigrid_gnn_farthest_point_sampling.ipynb cell 0 ("L_mean")
 *   smooth = sum_j u_j^T K u_j / (n_global k)         multigrid_gnn_refine_fixed.ipynb cell 4 ("L_smooth_total")
 * loss_acc (9 doubles) += {w_res L_res, w_orth L_orth, w_trace trace, w_order order, w_eigen eigen, TOTAL,
 *                          projection (added by the caller, see ep_loss_add_sum_f64), w_mean mean, w_smooth smooth}
 *   (flags & EP_FINALIZE_OVERWRITE: "=" instead of "+=", for the first level of a step)
 * coef receives what the backward needs (layout below, fp32):
 *   coef[0] = c_res = 2 w_res / (n_global k)
 *   coef[1 .. 1+k)      lam
 *   coef[1+k .. 1+2k)   num_bar   (dL/dnum)
 *   coef[1+2k .. 1+3k)  den_bar   (dL/dden)
 *   coef[1+3k .. 1+3k+k*k)   G_bar[a*k+b] = 2 w_orth / k * (G_ab - I_ab)
 *   coef[1+3k+k*k .. )  g_mean[j] = 2 w_mean (1^T M u_j) / (k - 1)  (dL/dMU_ij of the zero-mean term, same for all i)
 * (the smoothness term needs no extra coefficient: it is linear in num, so w_smooth / (n k) is added to num_bar)
 * lam_target may be NULL (eigen term = 0).  flags & EP_FINALIZE_EIGENVALUE_TERMS enables the :326-348
 * terms (the reference applies them to level 0 only).
 * lam_bar_extra (k floats, may be NULL) is added to dL/dlam: the gradient arriving from any
 * further use of the returned eigenvalues (autograd path of the drop-in modules). */
enum ep_finalize_flags { EP_FINALIZE_EIGENVALUE_TERMS = 1, EP_FINALIZE_OVERWRITE = 2 };
EP_API size_t ep_eigen_coef_len(int k);                            /* 1 + 4k + k*k floats */
EP_API int ep_eigen_finalize_f32(int k, double n_global, const double* partials, float w_res, float w_orth,
                          int flags, const float* lam_target, float w_trace, float w_order,
                          float w_eigen, float w_mean, float w_smooth, const float* lam_bar_extra,
                          float* lam_out, float* coef, double* loss_acc, ep_stream_t stream);
/* loss_acc[slot] += weight * sum(values[0..len)) and the same into loss_acc[5] (total).  Bookkeeping for terms that are
 * assembled from the SpMM / partials kernels on the caller's side - the projection term
 *   w_proj * sum (P^T U - U_coarse)^2 / (n_coarse k)          (multigrid_gnn_refine_fixed.ipynb cell 0, "L_proj")
 * = SpMM with P^T, ep_axpy_out_f32, ep_eigen_partials_f32 (its `num` block is the column-wise sum of squares). */
EP_API int ep_loss_add_sum_f64(int len, const double* values, double weight, int slot, double* loss_acc,
                        ep_stream_t stream);

/* Phase 3 (backward, per level): analytic gradient of the loss w.r.t. the three tensors it
 * was built from (what autograd derives from :309-322):
 *   R_bar  = c_res (KU - MU lam)
 *   KU_bar = R_bar + U num_bar
 *   MU_bar = -R_bar lam + U den_bar + U G_bar + 1 g_mean^T
 *   D      = KU num_bar + MU den_bar + MU G_bar^T        (direct dependence on U)
 * followed by ep_spmm2_sum_csr_f32(K^T, M^T, KU_bar, MU_bar, D) -> dL/dU. */
EP_API int ep_eigen_bwd_prepare_f32(int n, int k, const float* U, int ldu, const float* KU, const float* MU,
                             int ld, const float* coef, float* KU_bar, float* MU_bar, float* D,
                             ep_stream_t stream);

/* Phase 3, fused variant for SYMMETRIC K and M (one gather pass, nothing materialised):
 *   dU = out_scale * [ c_res * sum_j (K_ij - lam M_ij)(KU_j - lam MU_j) + 2 num_bar KU_i + MU_i (Gp + Gp^T)
 *                      + (sum_j M_ij) g_mean ]
 * with Gp = G_bar + diag(den_bar).  Algebraically equal to prepare + ep_spmm2_sum_csr_f32 when K = K^T,
 * M = M^T.  Needs k % 4 == 0, k <= 128, 16-byte aligned rows (EP_ERR_UNSUPPORTED otherwise).
 * Only the output rows [row0, row0 + n_rows) are written (row0 = 0, n_rows = n: all); every pointer keeps its row-0
 * base.  The vertex-sharded step computes the interior rows while the halo rows of KU / MU are in flight, then the
 * boundary rows. */
EP_API int ep_eigen_bwd_fused_sym_rows_f32(int row0, int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                                    const float* valK, const float* valM, const float* KU, const float* MU, int ld,
                                    const float* coef, float out_scale, const float* out_scale_dev, float* dU, int ldo,
                                    ep_stream_t stream);

/* Two-kernel form of the same backward with the dense k x k product on the TENSOR CORES (tcgen05 kind::tf32, 3-pass
 * hi/lo split = fp32 accuracy, accumulators in TMEM):
 *   1. ep_eigen_bwd_gram_term_tf32x3     dU[row0 .. row0+n) = out_scale * MU_i (Gp + Gp^T)          (k = 64 only)
 *   2. ep_eigen_bwd_gather_sym_rows_f32  with gram_in_out = 1: dU += out_scale * (gathered terms), product skipped
 * The one-kernel form spends 53 % (k = 32) to 75 % (k = 64) of its time issuing that product with shuffles, yet at
 * k = 32 it is still the faster one: step 1 is built for k = 64 only and returns EP_ERR_UNSUPPORTED for any other k. */
EP_API int ep_eigen_bwd_gram_term_tf32x3(int row0, int n_rows, int k, const float* MU, int ld, const float* coef,
                                  float out_scale, const float* out_scale_dev, float* dU, int ldo, ep_stream_t stream);
EP_API int ep_eigen_bwd_gather_sym_rows_f32(int row0, int n_rows, int k, const int32_t* rowptr, const int32_t* col,
                                     const float* valK, const float* valM, const float* KU, const float* MU, int ld,
                                     const float* coef, float out_scale, const float* out_scale_dev, float* dU, int ldo,
                                     int gram_in_out, ep_stream_t stream);

/* ---- column M-normalisation: multigrid_model.py:120-130, :366-380 ----------------------
 * out[:, j] = U[:, j] / sqrt(colsum_j + 1e-12) where colsum_j = sum_i U_ij MU_ij is read from
 * the diagonal of a partials block (G_jj).  */
EP_API int ep_scale_columns_rsqrt_f32(int n, int k, const float* U, int ldu, const double* G, int ldg,
                               double eps, float* out, int ldo, ep_stream_t stream);

/* out = a + alpha * b  (U_pred = U_base + adaptive_scale * corr_raw, multigrid_model.py:243-245);
 * alpha_dev, when non-NULL, is a device scalar that overrides alpha (graph-capturable ramp). */
EP_API int ep_axpy_out_f32(size_t n, float alpha, const float* alpha_dev, const float* a, const float* b,
                    float* out, ep_stream_t stream);

/* ---- learnable per-mode scales and the smoothness of the correction -------------------------
 * AdaptiveCorrector of delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4: corr = c o s (c: raw MLP output,
 * n x k; s: k scales, column scaling), U_pred = U_base + sigma corr, and the `train_gnn` term
 *   L_sc = w / (n_global k) sum_ij corr_ij (K corr)_ij = w / (n_global k) sum_j s_j^2 P_j,  P_j = sum_i c_ij (K c)_ij
 * (K symmetric, K (c o s) = (K c) o s: only K c is formed, with ep_spmm_csr_f32).  k <= 256.
 * Forward: U_pred = U_base + sigma * (c o s), rounded product by product (c s, then sigma (c s), then the sum; with
 * s == NULL bit-identical to ep_axpy_out_f32).  s == NULL means unit scales; sigma_dev (device float, may be NULL)
 * overrides sigma (graph-capturable ramp).  16-byte accesses when k % 4 == 0 and rows are 16-byte aligned. */
EP_API int ep_mode_scale_fwd_f32(int n, int k, const float* c, int ldc, const float* U_base, int ldb, const float* s,
                          float sigma, const float* sigma_dev, float* U_pred, int ldu, ep_stream_t stream);
/* Backward, per level.  dcorr holds g = dL/dcorr from the eigen-loss backward (sigma already applied) and is rewritten
 * in place to dL/dc, with w2 = 2 w_smooth_corr / (n_global k):
 *   dcorr_ij <- s_j g_ij + w2 s_j^2 (K c)_ij
 *   grad_s_j  = sum_i c_ij g_ij + w2 s_j P_j          (accumulate = 0: "=", first level of a step; 1: "+=")
 *   loss_acc[8] and loss_acc[5] += L_sc
 * Kc == NULL (w_smooth_corr = 0) skips the smoothness part; s == NULL means unit scales, grad_s must then be NULL.
 * One streaming pass writes per-CTA fp64 column sums to the workspace (ep_mode_scale_bwd_workspace_bytes(k)), one CTA
 * reduces them in a fixed order: deterministic, no host synchronisation (graph-capturable).  2 launches. */
EP_API size_t ep_mode_scale_bwd_workspace_bytes(int k);
EP_API int ep_mode_scale_bwd_f32(int n, int k, double n_global, const float* c, int ldc, const float* Kc, int ldkc,
                          const float* s, float w_smooth_corr, float* dcorr, int ldd, float* grad_s, int accumulate,
                          double* loss_acc, void* workspace, size_t workspace_bytes, ep_stream_t stream);

/* ---- corrector MLP, fp32 SIMT path ("parity mode"): corrector_model.py:12-21,31 ---------
 * Y = act(X W^T + b), W: out x in row-major (nn.Linear layout), act: 0 none, 1 ReLU. */
EP_API int ep_linear_fwd_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* b,
                      float* Y, int ldy, int act, ep_stream_t stream);
/* Backward of one layer.  dY: n x out (gradient w.r.t. the pre-activation of this layer).
 *   dX = (dY W) * [X > 0]  if dX != NULL (X is the previous layer's ReLU output, so its sign
 *        pattern is the ReLU mask; relu_mask == 0 skips the mask for a non-ReLU input)
 *   dW = dY^T X  (out x in),  db = column sums of dY.
 * workspace: ep_linear_bwd_workspace_bytes(n, in, out) bytes (split-K partials, deterministic). */
EP_API size_t ep_linear_bwd_workspace_bytes(int n, int in, int out);
EP_API int ep_linear_bwd_f32(int n, int in, int out, const float* X, int ldx, const float* W,
                      const float* dY, int lddy, float* dX, int lddx, int relu_mask,
                      float* dW, float* db, void* workspace, size_t workspace_bytes,
                      ep_stream_t stream);

/* ---- dropout after a hidden ReLU (the nn.Dropout(p) of corrector_model.py::_build_net in training mode) ----------
 * Keep masks are regenerated, never stored: unit (row, col) of hidden layer `layer` is kept iff the 16-bit lane of
 * Philox4x32-10(key = seed, counter = (row0 + row, col / 8, layer, step)) that belongs to col is >= thr, with
 * thr = round(p * 65536) (0 <= p, thr < 65536, else EP_ERR_INVALID); kept units are scaled by s = 1 / (1 - thr / 65536)
 * (fp32), so E[y] = relu(z).  Lane of feature 8c + 2j: low half of output word j; 8c + 2j + 1: its high half.  `row`
 * is the row of the MLP input, `col` the output feature, `step` the Adam step t the forward feeds; step_dev (device,
 * may be NULL) overrides step so a captured graph draws fresh masks each replay.  Not torch's RNG stream: dropout
 * runs match the reference in distribution, not bit for bit.  Both MLP modes draw identical masks.
 * The backward needs no mask: the stored activation is non-zero exactly where the unit is kept and z > 0.
 * ep_dropout_keep_mask_u8: keep[r * width + c] = 1 / 0 for rows 0..n-1 (tests, hosts that apply the mask themselves). */
EP_API int ep_dropout_keep_mask_u8(long long n, int width, float p, unsigned long long seed, int step,
                                   const int* step_dev, int layer, long long row0, unsigned char* keep,
                                   ep_stream_t stream);
/* Y = keep ? relu(X W^T + b) * s : 0  (ep_linear_fwd_f32 with act = 1, then nn.Dropout) */
EP_API int ep_linear_fwd_dropout_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* b,
                              float* Y, int ldy, float p, unsigned long long seed, int step,
                              const int* step_dev, int layer, long long row0, ep_stream_t stream);
/* ep_linear_bwd_f32 for a layer whose input X is the output of a hidden layer with dropout p:
 * dX = (dY W) * [X > 0] * s;  dW, db, workspace as there. */
EP_API int ep_linear_bwd_dropout_f32(int n, int in, int out, const float* X, int ldx, const float* W,
                              const float* dY, int lddy, float* dX, int lddx, float p,
                              float* dW, float* db, void* workspace, size_t workspace_bytes,
                              ep_stream_t stream);
/* fp64 forms (plain DFMA, same tiling and fixed-order split-K): the dense layers of the notebook networks in double -
 * `MLP` of scripts/simplified_loss.ipynb cell 0 and scripts/loss_with_rigid_body.ipynb cell 0, `EigenfunctionNN` of
 * delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1. */
EP_API int ep_linear_fwd_f64(int n, int in, int out, const double* X, int ldx, const double* W, const double* b,
                      double* Y, int ldy, int act, ep_stream_t stream);
EP_API size_t ep_linear_bwd_workspace_bytes_f64(int n, int in, int out);
EP_API int ep_linear_bwd_f64(int n, int in, int out, const double* X, int ldx, const double* W,
                      const double* dY, int lddy, double* dX, int lddx, int relu_mask,
                      double* dW, double* db, void* workspace, size_t workspace_bytes,
                      ep_stream_t stream);
/* Dense layers with an activation epilogue: the SiLU / sin / tanh networks of the notebooks (CoordinateMLP,
 * EigenfunctionNN in variants.py), same tiling and summation order as ep_linear_{fwd,bwd}_*, accurate libm math
 * (expf / exp, sinf / sin, cosf / cos, tanhf / tanh).  act: 0 none, 1 ReLU, 2 SiLU z / (1 + e^-z), 3 sin, 4 tanh;
 * any other value is EP_ERR_INVALID.
 * Forward: z = X W^T + b (b may be NULL), Y = act(z); Z (may be NULL) receives z.  The backward of the next layer needs
 * Z when act is SiLU or sin; Z may be NULL when no backward follows or act is 0, 1 or 4. */
EP_API int ep_linear_act_fwd_f32(int n, int in, int out, const float* X, int ldx, const float* W, const float* b,
                                 float* Y, int ldy, float* Z, int ldz, int act, ep_stream_t stream);
EP_API int ep_linear_act_fwd_f64(int n, int in, int out, const double* X, int ldx, const double* W, const double* b,
                                 double* Y, int ldy, double* Z, int ldz, int act, ep_stream_t stream);
/* Backward of one layer whose input X = act_x(Zx) is the output of the layer below (act_x = 0 for the network input).
 * dY: n x out, the gradient w.r.t. this layer's pre-activation.
 *   dX = (dY W) * act_x'   if dX != NULL: the gradient w.r.t. the pre-activation of the layer below.
 *        act_x' = [X > 0] (ReLU), sigmoid(z) (1 + z (1 - sigmoid(z))) (SiLU), cos z (sin) with z read from Zx, and
 *        1 - X^2 (tanh); act_x = 0 gives dX = dY W.  Zx (ldzx) must be non-NULL when dX is and act_x is 2 or 3.
 *   dW = dY^T X (out x in), db = column sums of dY, exactly as ep_linear_bwd_*.
 * workspace: ep_linear_bwd_workspace_bytes(n, in, out) bytes (_f64 for the double form). */
EP_API int ep_linear_act_bwd_f32(int n, int in, int out, const float* X, int ldx, const float* Zx, int ldzx, int act_x,
                                 const float* W, const float* dY, int lddy, float* dX, int lddx, float* dW, float* db,
                                 void* workspace, size_t workspace_bytes, ep_stream_t stream);
EP_API int ep_linear_act_bwd_f64(int n, int in, int out, const double* X, int ldx, const double* Zx, int ldzx,
                                 int act_x, const double* W, const double* dY, int lddy, double* dX, int lddx,
                                 double* dW, double* db, void* workspace, size_t workspace_bytes, ep_stream_t stream);

/* ---- corrector MLP, bf16 tcgen05 path ("perf mode") --------------------------------------
 * Same Linear / ReLU network, evaluated layer by layer on the 5th-generation tensor cores:
 * bf16 operands, fp32 accumulation in TMEM, TMA bulk copies, persistent CTAs with the layer's
 * weights resident in shared memory.  Activations and their gradients are kept in HBM as bf16 in a
 * packed tile layout  packed[tile][feature/8][vertex in tile (128)][8]  that is at once the
 * tcgen05 no-swizzle K-major operand (forward, dX) and MN-major operand (dW = dZ^T H); see
 * csrc/mlp_tc.cu.  Feature counts are padded: ep_tc_pad_features(d, wide) -> multiple of 32, or of
 * 128 for hidden widths (wide = 1); padded sizes must be <= 256.  Padding is zero-filled. */
EP_API int ep_tc_pad_features(int d, int wide);
EP_API size_t ep_tc_packed_rows_bytes(int n, int d_padded);
EP_API size_t ep_tc_packed_weight_bytes(int out_padded, int in_padded);
/* fp32 rows [n x d] -> packed bf16 tiles (corrector input h; gradient w.r.t. the network output). */
EP_API int ep_tc_pack_rows_bf16(int n, int d, int d_padded, const float* X, int ldx, void* packed,
                         ep_stream_t stream);
/* W fp32 [out x in] (nn.Linear layout) -> Wp [in_p/8][out_p][8] and, if WTp != NULL, WTp [out_p/8][in_p][8].
 * Each buffer holds TWO copies (ep_tc_packed_weight_bytes accounts for both): the layout above, then the same matrix
 * as [K/32][half of N][4][N/2][8] - the order in which a CTA pair of the chain kernel (tcgen05 cta_group::2) streams
 * its half of every K = 32 slab with one contiguous bulk copy. */
EP_API int ep_tc_pack_weight_bf16(int out, int in, int out_padded, int in_padded, const float* W, void* Wp,
                           void* WTp, ep_stream_t stream);
/* hidden layer: out_packed = relu(A W^T + b) (relu must be 1); relu_mask_out (may be NULL) receives one bit per
 * activation, [row][out_padded/32] words.  Bit order inside a word (block of 32 features = 16 stored bf16 pairs):
 * bit i = "feature 32w + 2i is > 0", bit 16 + i = "feature 32w + 2i + 1 is > 0", > 0 referring to the stored bf16
 * activation (this order makes building and applying the mask 1.5 / 2 integer instructions per element). */
EP_API size_t ep_tc_relu_mask_bytes(int n, int d_padded);
EP_API int ep_tc_linear_fwd_bf16(int n, int in_padded, int out, int out_padded, const void* A_packed, const void* Wp,
                          const float* bias, int relu, void* out_packed, void* relu_mask_out,
                          ep_stream_t stream);
/* last layer: corr = A W^T + b as fp32 rows and, fused, U_pred = U_base + scale * corr
 * (multigrid_model.py:243-245); U_base / U_pred may both be NULL. */
EP_API int ep_tc_linear_final_bf16(int n, int in_padded, int out, int out_padded, const void* A_packed, const void* Wp,
                            const float* bias, float* corr, int ldc, const float* U_base, float scale,
                            const float* scale_dev, float* U_pred, int ldu, ep_stream_t stream);
/* dZ_prev = (dZ W) * [act > 0]; the ReLU mask of the previous layer is the bit mask its forward wrote.
 * max_ctas > 0 limits the persistent grid (dX and dW of one layer run concurrently on two streams, half the
 * SMs each and the same tile order, so the dZ tiles one of them pulls from HBM are L2 hits for the other). */
EP_API int ep_tc_linear_dx_bf16(int n, int out_padded, int in_padded, const void* dZ_packed, const void* WTp,
                         const void* relu_mask, void* dZprev_packed, int max_ctas, ep_stream_t stream);
/* All layers in ONE launch ("fused MLP over vertex tiles", corrector_model.py:12-21,31), run by persistent clusters of
 * two CTAs (tcgen05 cta_group::2): one MMA covers 256 vertices, 128 from each CTA, and each CTA keeps its own two tiles
 * in ping-pong, so the tensor cores work on one tile while the epilogue drains the other.  An activation tile stays in
 * shared memory between layers (the epilogue of layer l writes the A operand of layer l+1 in place); weights stream
 * from L2 in K = 32 slabs, each CTA holding its half of the output columns (the second copy of ep_tc_pack_weight_bf16),
 * so a cluster reads every layer once per four tiles.  Hidden activations and ReLU masks are still written to HBM (the
 * backward needs them) but never read back.
 * Layer tables are HOST arrays of n_layers entries (device pointers inside): dims_padded[n_layers + 1] padded widths
 * (input first), dims_out[n_layers] true output widths (bias lengths; dims_out[n_layers-1] = k), Wp / bias per layer,
 * act_out / relu_mask_out per hidden layer (tables or entries may be NULL: not stored).  The last layer writes fp32
 * rows: corr (may be NULL) and, fused, U_pred = U_base + scale * corr (multigrid_model.py:243-245).
 * Results are bit-identical to the layer-by-layer entry points above. */
EP_API int ep_tc_chain_fwd_bf16(int n, int n_layers, const int* dims_padded, const int* dims_out, const void* A0_packed,
                         const void* const* Wp, const float* const* bias, void* const* act_out,
                         void* const* relu_mask_out, float* corr, int ldc, const float* U_base, float scale,
                         const float* scale_dev, float* U_pred, int ldu, ep_stream_t stream);
/* Dropout forms of the bf16 path (masks and scale as for ep_linear_fwd_dropout_f32; corrector_model.py::_build_net,
 * nn.Dropout after every hidden ReLU).  The forward scales by s and zeroes dropped units before the bf16 pack, so the
 * ReLU bit mask it writes is "kept and > 0"; the dX form multiplies by s in fp32 and rounds once.
 * Chain: hidden layer l uses layer index l and p_layers[l] (HOST array of n_layers - 1 entries) or, when p_layers is
 * NULL, p for every hidden layer.  Bit-identical to the layer-by-layer dropout entry points. */
EP_API int ep_tc_linear_fwd_dropout_bf16(int n, int in_padded, int out, int out_padded, const void* A_packed,
                                  const void* Wp, const float* bias, void* out_packed, void* relu_mask_out, float p,
                                  unsigned long long seed, int step, const int* step_dev, int layer, long long row0,
                                  ep_stream_t stream);
EP_API int ep_tc_linear_dx_dropout_bf16(int n, int out_padded, int in_padded, const void* dZ_packed, const void* WTp,
                                 const void* relu_mask, void* dZprev_packed, float p, int max_ctas,
                                 ep_stream_t stream);
EP_API int ep_tc_chain_fwd_dropout_bf16(int n, int n_layers, const int* dims_padded, const int* dims_out,
                                 const void* A0_packed, const void* const* Wp, const float* const* bias,
                                 void* const* act_out, void* const* relu_mask_out, float* corr, int ldc,
                                 const float* U_base, float scale, const float* scale_dev, float* U_pred, int ldu,
                                 const float* p_layers, float p, unsigned long long seed, int step,
                                 const int* step_dev, long long row0, ep_stream_t stream);
/* dW = dZ^T act (fp32 [out x in]) and db = column sums of dZ; deterministic two-stage reduction. */
EP_API size_t ep_tc_dw_workspace_bytes(void);
EP_API int ep_tc_linear_dw_bf16(int n, int out, int in, int out_padded, int in_padded, const void* dZ_packed,
                         const void* act_packed, float* dW, float* db, void* workspace, size_t workspace_bytes,
                         int max_ctas, ep_stream_t stream);

/* ---- optimiser: clip_grad_norm_ + Adam(weight_decay) step, multigrid_model.py:218-220,259-260
 * Parameters / gradients / moments live in one flat fp32 buffer each.
 *   norm   = sqrt(sum g^2)                      (ep_grad_sqnorm_f32 -> sq_out, fp64, device)
 *   coef   = min(1, max_norm / (norm + 1e-6));  g = coef * g + weight_decay * p
 *   m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2
 *   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
 * The bias corrections 1 - b^t are evaluated on the device in double from the integer step t, whether t
 * arrives by value or from device memory, so a replayed CUDA graph is bit-identical to eager launches.
 * hyper_dev (device, may be NULL) = {float lr, int32 t} (8 bytes) overrides lr and step, so a captured
 * graph can follow the ReduceLROnPlateau schedule of :221-223 and the step count. */
EP_API int ep_grad_sqnorm_f32(size_t n, const float* g, double* sq_out, ep_stream_t stream);
EP_API int ep_adam_clip_step_f32(size_t n, float* p, const float* g, float* m, float* v, float lr,
                          const float* hyper_dev, float beta1, float beta2, float eps,
                          float weight_decay, int step, float max_norm, const double* sq_norm,
                          ep_stream_t stream);
/* fp64 forms for networks trained in double (delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1 trains
 * EigenfunctionNN with Adam(betas=(0.999, 0.9999)) in fp64).  Same update, order and clipping semantics (no clipping
 * when max_norm <= 0 or sq_norm is NULL); hyper_dev (device, may be NULL) = {double lr, double t} with t an integer. */
EP_API int ep_grad_sqnorm_f64(size_t n, const double* g, double* sq_out, ep_stream_t stream);
EP_API int ep_adam_clip_step_f64(size_t n, double* p, const double* g, double* m, double* v, double lr,
                                 const double* hyper_dev, double beta1, double beta2, double eps, double weight_decay,
                                 int step, double max_norm, const double* sq_norm, ep_stream_t stream);

/* ---- one eigenfunction at a time: delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1 ---------------
 * (EigenfunctionNN; compute_eigenvalue_loss, compute_normalization_loss, compute_orthogonality_loss), the pieces of an
 * autograd-free training step (csrc/single_mode.cu).  u, Lu = L u, Mu = M u: n x 1 contiguous (ep_spmm2_csr_* at k = 1);
 * w: the eigenvalue weight (device, one value), lambda = |w|; Q: n x P row-major (ldq >= P), column p = M u_p of the
 * p-th earlier mode (constant; may be NULL when P = 0).  0 <= P <= ep_single_mode_max_prev() (64; larger P is
 * EP_ERR_UNSUPPORTED), n >= 1.  With r = Lu - lambda Mu:
 *   forward   loss[0..4) = [total, eig, norm, ortho] (fp64, device): eig = mean(r^2), norm = (u^T M u - 1)^2,
 *             ortho = sum_p (u^T Q_p)^2, total = eig + norm + ortho_weight * ortho;
 *             coef[0..3+P) (fp64, device) = [2/n, 4 (u^T M u - 1), dL/dlambda = -(2/n) sum r o Mu, c_p = 2 ortho_weight
 *             u^T Q_p].  Sums are fp64, per CTA into the workspace (ep_single_mode_workspace_bytes(P)), then reduced
 *             by one CTA in a fixed order: deterministic and graph-capturable.
 *   backward  gL = (2/n) r, gM = -(2/n) lambda r, D = 4 (u^T M u - 1) Mu + Q c  (r recomputed, not stored); then
 *             ep_spmm2_sum_csr_*(L, M, gL, gM, D) = dL/du for symmetric L, M. */
EP_API int ep_single_mode_max_prev(void);
EP_API size_t ep_single_mode_workspace_bytes(int P);
EP_API int ep_single_mode_fwd_f32(int n, int P, const float* u, const float* Lu, const float* Mu, const float* Q,
                                  int ldq, const float* w, double ortho_weight, double* loss, double* coef,
                                  void* workspace, size_t workspace_bytes, ep_stream_t stream);
EP_API int ep_single_mode_fwd_f64(int n, int P, const double* u, const double* Lu, const double* Mu, const double* Q,
                                  int ldq, const double* w, double ortho_weight, double* loss, double* coef,
                                  void* workspace, size_t workspace_bytes, ep_stream_t stream);
EP_API int ep_single_mode_bwd_f32(int n, int P, const float* Lu, const float* Mu, const float* Q, int ldq,
                                  const float* w, const double* coef, float* gL, float* gM, float* D,
                                  ep_stream_t stream);
EP_API int ep_single_mode_bwd_f64(int n, int P, const double* Lu, const double* Mu, const double* Q, int ldq,
                                  const double* w, const double* coef, double* gL, double* gM, double* D,
                                  ep_stream_t stream);
/* lambda appended to every layer's input, folded into the bias: layer(h (+) lambda) = h W[:, :d]^T + (b + lambda
 * W[:, d]).  dims: HOST array of n_layers + 1 widths (input first), 1 <= n_layers <= 8.  Flat device layouts, per layer
 * l with input width d and output width o, in layer order:
 *   params, grad     [W_l (o x (d + 1), row-major) | b_l (o)] ... then w (one value)
 *   eff, grad_eff    [W_eff,l (o x d) | b_eff,l (o)] ...
 * Forward: W_eff,l = W_l[:, :d], b_eff,l = b_l + lambda W_l[:, d] (product, then sum: as the autograd form rounds).
 * Backward from dW_eff, db_eff (grad_eff) and dL/dlambda of the loss (device fp64, may be NULL = 0):
 *   dW_l[:, :d] = dW_eff,l, dW_l[:, d] = lambda db_eff,l, db_l = db_eff,l,
 *   dw = sign(w) (dL/dlambda + sum_l db_eff,l^T W_l[:, d])   (sign(0) = 0, torch's gradient of |w|). */
EP_API int ep_single_mode_fold_fwd_f32(int n_layers, const int* dims, const float* params, float* eff,
                                       ep_stream_t stream);
EP_API int ep_single_mode_fold_fwd_f64(int n_layers, const int* dims, const double* params, double* eff,
                                       ep_stream_t stream);
EP_API int ep_single_mode_fold_bwd_f32(int n_layers, const int* dims, const float* params, const float* grad_eff,
                                       const double* dloss_dlam, float* grad, ep_stream_t stream);
EP_API int ep_single_mode_fold_bwd_f64(int n_layers, const int* dims, const double* params, const double* grad_eff,
                                       const double* dloss_dlam, double* grad, ep_stream_t stream);

/* ---- samplers: samplers.py:97-143 (farthest point), :9-94 (voxel) ----------------------
 * fp64, bit-exact w.r.t. numpy: d = sqrt((dx*dx + dy*dy) + dz*dz) with IEEE round-to-nearest
 * and no FMA contraction, running minimum, first index wins arg-max / arg-min ties.
 * pts: N x 3 row-major doubles.  out_order: n_samples int64 (selection order; out_order[0]
 * = start).  One persistent cooperative kernel runs all n_samples-1 dependent iterations. */
EP_API size_t ep_fps_workspace_bytes(int64_t n_points);
EP_API int ep_fps_f64(int64_t n_points, const double* pts, int n_samples, int64_t start,
               int64_t* out_order, void* workspace, size_t workspace_bytes, ep_stream_t stream);
/* Host-buffer variant (allocates, copies in, runs, copies out, synchronises). */
EP_API int ep_fps_f64_host(int64_t n_points, const double* pts_host, int n_samples, int64_t start,
                    int64_t* out_order_host);

/* Axis-aligned bounds: lo_hi[0..3) = min, lo_hi[3..6) = max  (samplers.py:21-22). */
EP_API int ep_bounds_f64(int64_t n_points, const double* pts, double* lo_hi, ep_stream_t stream);
/* One voxel pass for one voxel size (body of the scale loop, samplers.py:45-74): cell =
 * clip(trunc((p - lo) / voxel), 0, dims-1); id = cx*dy*dz + cy*dz + cz; for every occupied
 * voxel pick the point nearest the voxel centre lo + (c + 0.5) * voxel (first index on ties).
 * out_idx receives the picks in ascending voxel id, *out_count (device int64) their number.
 * max_out bounds the write (count is still the true total). */
EP_API size_t ep_voxel_workspace_bytes(int64_t n_points, int64_t n_voxels);
EP_API int ep_voxel_select_f64(int64_t n_points, const double* pts, const double* lo, double voxel,
                        const int64_t* dims, int64_t* out_idx, int64_t max_out, int64_t* out_count,
                        void* workspace, size_t workspace_bytes, ep_stream_t stream);
EP_API int ep_voxel_select_f64_host(int64_t n_points, const double* pts_host, const double* lo, double voxel,
                             const int64_t* dims, int64_t* out_idx_host, int64_t max_out,
                             int64_t* out_count_host);

/* ---- "next" row: sparse FEM assembly on the device (Mesh.py:180-198, :228-234, :348-364) -----------
 * Step 1: per-triangle 3x3 stiffness / mass blocks (fp64, row-major, 9 entries per triangle) and the
 *         linear keys row * n_verts + col of those entries.
 * Step 2 (caller): STABLE sort of the keys, run starts / lengths of equal keys (= CSR entries).
 * Step 3: ordered sum of every run (triangle order, like the reference loop) -> col, fp32 values for the
 *         hot path and optionally the fp64 values. */
EP_API int ep_fem_elements_f64(int64_t n_tris, const double* verts, const int32_t* tris, int64_t n_verts,
                        double* k_el, double* m_el, int64_t* keys, ep_stream_t stream);
EP_API int ep_fem_segment_sum_f64(int64_t nnz, const int64_t* seg_start, const int64_t* seg_count,
                           const int64_t* perm, const double* k_el, const double* m_el,
                           const int64_t* uniq_keys, int64_t n_verts, int32_t* col, float* valK, float* valM,
                           double* valK64, double* valM64, ep_stream_t stream);

/* ---- "next" row: k nearest neighbours for the aggregation graph and the prolongation (utils.py:39-75) -----------
 * Replaces sklearn NearestNeighbors(n_neighbors=k).fit(ref).kneighbors(query).  Reference points are binned on a
 * uniform grid by the caller: cell id = (cx * dims[1] + cy) * dims[2] + cz with c = clip(floor((p - lo) / cell)),
 * `order` = reference indices sorted by cell id (stable), cell_start[c] .. cell_start[c+1] = the slice of `order` that
 * lies in cell c (dims[0]*dims[1]*dims[2] + 1 entries).  Distances are fp64 ((dx*dx + dy*dy) + dz*dz, no FMA); ties are
 * broken by the smaller reference index.  out_idx: n_query x k int64 sorted by (distance, index); out_dist (may be
 * NULL): the distances.  lo, dims: HOST arrays. */
EP_API int ep_knn_grid_f64(int64_t n_query, const double* query, int64_t n_ref, const double* ref, const int64_t* order,
                    const int64_t* cell_start, const double* lo, double cell, const int64_t* dims, int k,
                    int64_t* out_idx, double* out_dist, ep_stream_t stream);

/* ---- multi-GPU plumbing: halo rows --------------------------------------------------------
 * dst[r, :] = src[idx[r], :]  (pack the boundary rows of U that a peer needs). */
EP_API int ep_gather_rows_f32(int n_idx, int k, const int32_t* idx, const float* src, int lds,
                       float* dst, int ldd, ep_stream_t stream);
/* dst[idx[r], :] += src[r, :]   (idx values must be unique within one call). */
EP_API int ep_scatter_add_rows_f32(int n_idx, int k, const int32_t* idx, const float* src, int lds,
                            float* dst, int ldd, ep_stream_t stream);

/* ---- multi-GPU: the exchanges of the vertex-sharded step, for hosts that do not go through torch.distributed ----
 * The reference has no distributed code; these are the communication steps the sharded path adds around
 * src/multigrid_model.py:301-324 (SURVEY 8e).  `nccl_comm` is the caller's ncclComm_t (one rank per GPU).  NCCL is not
 * linked: its entry points are resolved at run time from the libnccl.so.2 the process already uses, so the
 * communicator and the calls always belong to the same NCCL instance.  Everything is enqueued on `stream`; run the
 * exchange on a side stream to overlap it with the interior rows (what dist_engine.py does).
 *
 * ep_halo_exchange_f32: row space of a rank = [owned rows | halo rows], `rows` points at the owned block and
 * `halo_rows` at the halo block of the same dense (ld == k) array.  For peer p (rank peer_rank[p]) the owned rows
 * send_idx[send_offset[p] .. send_offset[p+1]) (device int32) are packed into send_buf (device, send_offset[n_peers] x k)
 * and sent, and recv_offset[p+1] - recv_offset[p] rows are received into halo_rows + recv_offset[p] * k, all in one
 * NCCL group.  The three offset / rank arrays are host arrays of n_peers (+1) entries. */
EP_API int ep_dist_nccl_version(void);        /* 0: no NCCL library could be resolved in this process */
EP_API int ep_halo_exchange_f32(void* nccl_comm, int n_peers, const int* peer_rank, const int* send_offset,
                         const int32_t* send_idx, const int* recv_offset, int k, const float* rows, int ld,
                         float* send_buf, float* halo_rows, ep_stream_t stream);
/* in-place sum over all ranks: the packed fp64 partials of a level / the flat fp32 gradient buffer. */
EP_API int ep_allreduce_sum_f64(void* nccl_comm, size_t count, double* buf, ep_stream_t stream);
EP_API int ep_allreduce_sum_f32(void* nccl_comm, size_t count, float* buf, ep_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* EIGENPINNS_B200_H */
