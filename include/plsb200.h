/*
 * plsb200 -- C ABI of the B200-native resampling engine for plspy (McIntosh-Lab/plspy).
 *
 * This is the drop-in boundary for ONE path of the reference: the permutation test, the bootstrap
 * test and the split-half loops of `plspy.core` (reference seam:
 * plspy/core/bootstrap_permutation.py:53-63,139-263 `ResampleTest._create` and
 * plspy/core/split_half_resampling.py:23,404).  The reference is pure Python/numpy, so the binding a
 * maintainer adds is a ctypes stub (see INTEGRATION.md); every entry point takes plain pointers and
 * sizes only.
 *
 * Conventions
 *  - all matrices are float64, row-major, resident in DEVICE memory unless the name ends in `_host`;
 *  - index matrices are int32, row-major, one resample per row (values in [0, N));
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream); all calls are asynchronous
 *    with respect to the host except where stated;
 *  - every function returns 0 on success, a negative PLSB200_E* code otherwise;
 *    plsb200_last_error() returns a thread-local message for the last failure;
 *  - the library allocates nothing that outlives a call: workspaces are caller-provided and sized by
 *    the matching *_workspace() query (bytes).
 *  - the caller owns all buffers (reference ownership: fresh numpy arrays owned by the result object,
 *    bootstrap_permutation.py:496-532).
 *
 * Notation (SURVEY.md section 8): N rows of X (subjects x conditions), p voxels, K columns of the
 * coefficient matrix (latent variables / contrasts), R resamples in the batch.
 *   E  (N x K)  = Lop^T . U   : design-side weights pulled back to row space, constant per analysis
 *   C_r (N x K) = S_r^T . E   : C_r[idx_r[i], :] += E[i, :]          (scatter of E by one index vector)
 *   VS_r (p x K) = X^T . C_r  : the resampled, projected cross-block matrix `permuted.T @ U`
 *                               (bootstrap_permutation.py:404, :620)
 */
#ifndef PLSB200_H
#define PLSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLSB200_ABI_VERSION 3

#define PLSB200_OK 0
#define PLSB200_EINVAL (-1)   /* bad argument (shape, alignment, null pointer) */
#define PLSB200_ECUDA (-2)    /* CUDA runtime / launch error                   */
#define PLSB200_EWORKSPACE (-3) /* workspace too small                          */
#define PLSB200_EUNSUPPORTED (-4) /* shape outside what the kernels are built for */

int plsb200_abi_version(void);
const char* plsb200_last_error(void);
/* number of kernels launched by this library in this process since load (bench.py's gpu_launches) */
int64_t plsb200_launch_count(void);

/* strided host -> device copy (cudaMemcpy2DAsync): uploads a voxel range (column block) of a pinned row-major X */
int plsb200_copy2d_h2d(void* dst, size_t dst_pitch, const void* src_host, size_t src_pitch, size_t width_bytes,
                       size_t height, void* stream);

/* float32 -> float64 widening on the device: X may be stored and uploaded as float32 (plspy_b200/io.py: the data a NIfTI
 * file holds are float32 / int16; plspy/io/io.py:10-700 assembles them into a float64 matrix on the host)         */
int plsb200_widen_f32_f64(const float* src, double* dst, int64_t n, void* stream);

/* ---- float32-resident X.  Every entry point named *_x32* is its FP64 twin with X given as float32 (N x p, leading
 * dimension ldx in elements, any 4-byte aligned address and any ldx): each element is widened to float64 where the
 * kernel loads it, so the results are bit-identical to the twin's on the widened matrix.  Sizes and workspaces are
 * the twin's (plsb200_gram_f64_workspace, plsb200_xv_f64_workspace, plsb200_boot_moments_f64_workspace,
 * plsb200_boot_quad_f64_workspace, plsb200_tf32_ximage_bytes, plsb200_gram_tf32_image_bytes).                */

/* ---- K1: Gram matrix G = X . X^T (N x N), FP64 DMMA, split over voxel chunks, deterministic --------
 * Replaces the N x p work that every resample redoes in the reference (row gather + means + projection,
 * resample.py:79,153 + class_functions.py:7-95 + bootstrap_permutation.py:404): once G is known every
 * per-resample quantity except std_errs lives in N-space (SURVEY.md App. A).
 * X: N x p with leading dimension ldx (elements).  G: N x N dense, both triangles written.        */
size_t plsb200_gram_f64_workspace(int N, int64_t p);
int plsb200_gram_f64(const double* X, int N, int64_t p, int64_t ldx, double* G,
                     void* workspace, size_t workspace_bytes, void* stream);
int plsb200_gram_x32_f64(const float* X, int N, int64_t p, int64_t ldx, double* G,
                         void* workspace, size_t workspace_bytes, void* stream);
/* The same for the row stack [X1; X2] ((N1 + N2) x p) without materialising it: the multiblock methods need the Gram
 * matrix of [X; Zb] (class_functions.py:454-516 through N-space quadratic forms).  Workspace:
 * plsb200_gram_f64_workspace(N1 + N2, p).                                                                      */
int plsb200_gram_stacked_f64(const double* X1, int N1, int64_t ld1, const double* X2, int N2, int64_t ld2, int64_t p,
                             double* G, void* workspace, size_t workspace_bytes, void* stream);
/* 1 when the stack of N rows and K more has the same row tiles as the N rows alone: then the N x N block of its Gram
 * matrix is bit-identical to plsb200_gram_f64 of the N rows (same tiles, same voxel splits).                    */
int plsb200_gram_stack_fuses(int N, int K);

/* ---- latent projection XL = X . V (N x K); replaces class_functions._compute_X_latents
 * (class_functions.py:165-182) as used for U_hat (bootstrap_permutation.py:617).
 * V: p x K row-major.                                                                              */
size_t plsb200_xv_f64_workspace(int N, int64_t p, int K);
int plsb200_xv_f64(const double* X, int N, int64_t p, int64_t ldx, const double* V, int K,
                   double* XL, void* workspace, size_t workspace_bytes, void* stream);
int plsb200_xv_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* V, int K,
                       double* XL, void* workspace, size_t workspace_bytes, void* stream);

/* ---- K2/K6: N-space pass over a batch of resamples ------------------------------------------------
 * For each resample r (index vector idx[r, 0..N)):
 *     H_r  = G . C_r                                   (N x K)
 *     d2[r, k] = C_r[:, k]^T . H_r[:, k] = ||VS_r[:, k]||^2     (squared singular-value estimate,
 *                                                       bootstrap_permutation.py:405 / :432)
 *     if Lmat != NULL:  T[r] = Lmat (Kt x N) . H_r . diag(1/sqrt(d2[r]))   (Kt x K)
 *                       = cellmeans(X @ normalize(VS_r)), the bootstrap `Tdistrib`
 *                       (bootstrap_permutation.py:633-634, :665-666); zero where d2 == 0.
 * Gather formulation, no atomics, deterministic.  d2: R x K.  T: R x Kt x K (may be NULL).          */
int plsb200_nspace_f64(const double* G, int N, const double* E, int K, const int32_t* idx, int R,
                       const double* Lmat, int Kt, double* d2, double* T, void* stream);

/* ---- per-resample SVD mode ("rotate_method = 0" of the older plspy API: re-run the SVD for every permutation).
 * With E = Lop^T (N x K: the rows of the cross-block builder, NOT projected on the original singular vectors)
 *     B[r] = C_r^T G C_r  (K x K)  =  M_r M_r^T,  M_r = Lop . X[idx_r]  the resampled cross-block matrix,
 * whose eigenvalues (plsb200_sym_eig_f64) are the squared singular values of M_r.  d2[r] = diag(B[r]).
 * B: R x K x K.  Needs 2 N K doubles of shared memory in one chunk.                                          */
int plsb200_nspace_gram_f64(const double* G, int N, const double* E, int K, const int32_t* idx, int R,
                            double* d2, double* B, void* stream);

/* ---- permutation counters -------------------------------------------------------------------------
 * s_hat = sqrt(d2) (set to 0 where |s_hat| < thresh when thresh > 0: bootstrap_permutation.py:436),
 * counts[k]     += (s_hat[r,k] >= s_ref[k])                              (:427/:433/:437)
 * counts[K + k] += (sum_{j>=k} s_hat[r,j]^2 >= totcov_ref[k])            (stepdown, :446-451)
 * `mb_total` (R) non-NULL applies the multiblock rescale s_hat <- sqrt(s_hat^4 / sum s_hat^4 * mb_total[r])
 * first (:419-424).  counts: int64[2K], ACCUMULATED into (caller zeroes).  s_hat: R x K out.         */
int plsb200_perm_count_f64(const double* d2, int R, int K, const double* s_ref, const double* totcov_ref,
                           double thresh, const double* mb_total, int64_t* counts, double* s_hat,
                           void* stream);

/* ---- U_hat_r = Lop (Ku x N) . XL_r[idx_r, :] (N x K)  -> Uhat: R x Ku x K   (bootstrap_permutation.py:617).
 * xl_stride = 0: one latent matrix XL shared by all resamples; otherwise XL_r = XL + r*xl_stride
 * (multiblock Tdistrib, :654-656, :665-666).  idx may be NULL (identity).                            */
int plsb200_uhat_f64(const double* XL, int64_t xl_stride, int N, int K, const double* Lop, int Ku,
                     const int32_t* idx, int R, double* Uhat, void* stream);

/* ---- K1 fast mode: G = X X^T on the tcgen05 tensor cores (kind::tf32, 3xTF32 split), N <= 320 (else
 * PLSB200_EUNSUPPORTED: use plsb200_gram_f64).  gram_tf32_split writes the operand image (TF32 hi/lo planes of X,
 * [block of 16 voxels][hi|lo][row][16 voxels] in the K-major SWIZZLE_64B tile order; gram_tf32_image_bytes bytes);
 * gram_tf32 forms G (N x N, both triangles) from it; accumulate != 0 adds to G (X given as several voxel ranges).
 * p = the voxel count the image was built for.  Relative error of the diagonal ~3e-6 (FP32 accumulation in tensor
 * memory drained every 512 voxels into round-to-nearest FP32 sums, FP64 across CTAs).  Replaces the N x p work of
 * every permutation (plspy/core/bootstrap_permutation.py:323-452) like plsb200_gram_f64.                        */
size_t plsb200_gram_tf32_image_bytes(int N, int64_t p);
int plsb200_gram_tf32_split(const double* X, int N, int64_t p, int64_t ldx, void* image, void* stream);
int plsb200_gram_tf32_split_x32(const float* X, int N, int64_t p, int64_t ldx, void* image, void* stream);
size_t plsb200_gram_tf32_workspace(int N, int64_t p);
int plsb200_gram_tf32(const void* image, int N, int64_t p, double* G, int accumulate, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ---- K4: bootstrap salience moments ---------------------------------------------------------------
 * The batched GEMM  VS[v, (r,k)] = sum_i X[i, v] . C_r[i, k]  over all R resamples, with
 * sum_r (VS - pivot) and sum_r (VS - pivot)^2 accumulated in registers; nothing of size p x K x R is
 * written (the reference materialises right_sv_sampled, bootstrap_permutation.py:497,626,695).
 *
 * Step 1 packs the coefficients C_r = scatter(E, idx_r) into the DMMA B-fragment order the kernel
 * streams through shared memory (`coef`, size from plsb200_boot_coef_bytes).
 * Step 2 runs the GEMM+moment kernel.  pivot (p x K) may be NULL (= 0).  sum, sumsq: p x K, overwritten.
 * Supported shapes: K <= 24 per call (split wider problems by column), any N.                     */
size_t plsb200_boot_coef_bytes(int N, int K, int R);
int plsb200_boot_coef_pack_f64(const double* E, int N, int K, const int32_t* idx, int R, double* coef,
                               void* stream);
size_t plsb200_boot_moments_f64_workspace(int N, int64_t p, int K, int R);
int plsb200_boot_moments_f64(const double* X, int N, int64_t p, int64_t ldx, const double* coef, int K,
                             int R, const double* pivot, double* sum, double* sumsq,
                             void* workspace, size_t workspace_bytes, void* stream);
int plsb200_boot_moments_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* coef, int K,
                                 int R, const double* pivot, double* sum, double* sumsq,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* Factored collapsed bootstrap (task methods; DESIGN.md section 3): J pseudo-resamples with the coefficients
 * c_j[n,k] = E[n,k] . L[sid[n], j] (L: ns x J row-major, sid: N subjects) packed for plsb200_boot_moments_f64 /
 * _x32_f64, which then run with R = J and pivot = NULL: their `sumsq` is q[v,k] = sum_j (x_v^T c_jk)^2.  Any N:
 * the pack writes the layout boot_moments reads (the register-resident kernel's for N <= 320, the output-stationary
 * kernel's for N > 320 or with PLSB200_EXACT=os).  The size query returns 0 (and the pack PLSB200_EUNSUPPORTED) for
 * K > 24.                                                                                                       */
size_t plsb200_boot_factor_coef_bytes(int N, int K, int J);
int plsb200_boot_factor_pack_f64(const double* E, int N, int K, const double* L, int J, const int32_t* sid,
                                 double* coef, void* stream);

/* ---- K4 collapsed (task methods, exact FP64): the bootstrap variance as a quadratic form ------------------
 * Each salience is linear in the draw, so R . Var_r(VS_r[v,k]) = x_v^T S_k x_v with S_k = R . Cov_r(c_rk) (N x N).
 *   q[v,k] = x_v^T S_k x_v   (p x K, overwritten)
 * Step 1 packs S ([K][N][N], row-major, k slowest) into the B-fragment order of the bootstrap GEMM
 * (`coef`, plsb200_boot_quad_coef_bytes bytes); step 2 evaluates the p x K quadratic forms on the FP64 tensor cores.
 * Feeding (sum = 0, sumsq = q) to plsb200_boot_finalize_f64 gives the bootstrap standard errors.
 * Supported shapes: N <= 320 and K <= 24 per call (split wider problems by column), else PLSB200_EUNSUPPORTED
 * (the size queries return 0).                                                                                  */
size_t plsb200_boot_quad_coef_bytes(int N, int K);
int plsb200_boot_quad_coef_pack_f64(const double* S, int N, int K, double* coef, void* stream);
size_t plsb200_boot_quad_f64_workspace(int N, int64_t p, int K);
int plsb200_boot_quad_f64(const double* X, int N, int64_t p, int64_t ldx, const double* coef, int K, double* q,
                          void* workspace, size_t workspace_bytes, void* stream);
int plsb200_boot_quad_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* coef, int K, double* q,
                              void* workspace, size_t workspace_bytes, void* stream);
/* The factor of the draw-count covariance.  layout (int32, 2N + ns): base[n] = first row of n's cell, sid[n] = subject of
 * row n, row0[s] = row of subject s in the first condition of its group.
 * boot_counts_f64: for every draw r of idx (R x N) sets *bad |= 1 unless each row keeps its cell and follows the
 * first condition's subject map (bad may be NULL); with counts != NULL writes counts[s * ldc + r] = m_r[s] - 1 (draws of
 * subject s) and counts[ns * ldc + r] = 1 -- their Gram matrix (plsb200_gram_f64) holds sum_r (m_r - 1)(m_r - 1)^T and,
 * in its last column, s1 = sum_r (m_r - 1).
 * boot_factor_f64: one CTA.  From that (ns + 1)-square Gram matrix Mg, M = Mg[:ns,:ns] - s1 s1^T / R_total, and L
 * (ns x J, J = ns - G, row-major) with L L^T = M: Cholesky of M without the last subject of each group (gstart: G + 1
 * subject offsets), a dropped subject's row = minus the sum of its group's other rows; non-positive pivots give zero
 * columns.  workspace: plsb200_boot_factor_f64_workspace bytes.                                                 */
int plsb200_boot_counts_f64(const int32_t* idx, int N, int R, const int32_t* layout, int ns, double* counts,
                            int64_t ldc, int32_t* bad, void* stream);
size_t plsb200_boot_factor_f64_workspace(int ns, int G);
int plsb200_boot_factor_f64(const double* Mg, int ns, int64_t R_total, const int32_t* gstart, int G, double* L,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ---- K4 fast mode: the same moments on the tcgen05 tensor cores with the 3xTF32 split ---------------------
 * (x = xh + xl, c = ch + cl, each TF32-exact; xh.cl + xl.ch + xh.ch accumulated in FP32 in tensor memory, the
 * moments in FP64).  Relative error of a salience ~1e-6; std_errs / boot_ratios agree with the FP64 path to
 * ~1e-6 (north-star tolerance for the fast mode: 1e-4).  Any N; 1 <= K <= 24 per call.
 * tf32_split_x: X -> `ximage` (plsb200_tf32_ximage_bytes), the TF32 hi/lo planes of X laid out as the
 *   shared-memory tiles the MMA reads; done once per analysis.
 * boot_coef_pack_tf32: coefficients C_r = scatter(E, idx_r) -> `coef` (plsb200_boot_coef_bytes_tf32).
 * boot_moments_tf32: sum_r (VS_r - pivot), sum_r (VS_r - pivot)^2 (p x K each, overwritten).              */
size_t plsb200_tf32_ximage_bytes(int N, int64_t p);
int plsb200_tf32_split_x(const double* X, int N, int64_t p, int64_t ldx, void* ximage, void* stream);
int plsb200_tf32_split_x32(const float* X, int N, int64_t p, int64_t ldx, void* ximage, void* stream);
size_t plsb200_boot_coef_bytes_tf32(int N, int K, int R);
int plsb200_boot_coef_pack_tf32(const double* E, int N, int K, const int32_t* idx, int R, void* coef, void* stream);
size_t plsb200_boot_moments_tf32_workspace(int N, int64_t p, int K, int R);
int plsb200_boot_moments_tf32(const void* ximage, int N, int64_t p, const void* coef, int K, int R,
                              const double* pivot, double* sum, double* sumsq, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---- std_errs / boot_ratios from the moments (bootstrap_permutation.py:695-703) --------------------
 * mean = pivot + sum/R ; std_errs = sqrt(max(sumsq/R - (sum/R)^2, 0)) (population std, ddof = 0);
 * boot_ratios = numer / std_errs  with numer = V*s (no contrast) or V (contrast), p x K.            */
int plsb200_boot_finalize_f64(const double* sum, const double* sumsq, int64_t p, int K, int64_t R_total,
                              const double* numer, double* std_errs, double* boot_ratios, void* stream);

/* ---- population std over the first axis of a (R x M) matrix -> M values (np.std(..., axis=0),
 * bootstrap_permutation.py:715,723,732)                                                             */
int plsb200_colstd_f64(const double* A, int R, int64_t M, double* out, void* stream);

/* ---- percentile interval over the resample axis (plspy/core/resample.py:171-222 `confidence_interval`, MATLAB
 * prctile convention: sorted sample k at 100 (k + 0.5) / B per cent, linear interpolation, clamped to the extremes).
 * Series s has its B samples at samples[r * stride_sample + s * stride_series] (strides in elements), so a
 * (B x m x n) stack is stride_sample = m n, stride_series = 1.  q_lo / q_hi are fractions in [0, 1]; lower / upper
 * receive nseries values each.  B <= 16384 sorts in shared memory; longer series need
 * plsb200_percentile_f64_workspace(B) bytes of scratch.                                                      */
size_t plsb200_percentile_f64_workspace(int B);
int plsb200_percentile_f64(const double* samples, int B, int64_t nseries, int64_t stride_sample,
                           int64_t stride_series, double q_lo, double q_hi, double* lower, double* upper,
                           void* workspace, size_t workspace_bytes, void* stream);
/* the bias-corrected percentile interval (Efron) of the same series: orig[s] is the original value theta of series s,
 * prop[s] = #{r : sample_r <= theta} / B, z0 = Phi^-1(prop), and the bounds are taken as above at the levels
 * Phi(2 z0 + Phi^-1(q_lo)) and Phi(2 z0 + Phi^-1(q_hi)) (q = 0 / 1: the minimum / maximum).  prop 0 or 1 gives NaN
 * bounds; a NaN theta gives NaN bounds and prop.  Workspace: plsb200_percentile_f64_workspace(B).                    */
int plsb200_percentile_bc_f64(const double* samples, int B, int64_t nseries, int64_t stride_sample,
                              int64_t stride_series, const double* orig, double q_lo, double q_hi, double* lower,
                              double* upper, double* prop, void* workspace, size_t workspace_bytes, void* stream);
/* the bias-corrected and accelerated interval (BCa, Efron 1987) of the same series: prop and z0 as in the BC interval,
 * accel[s] the acceleration a of series s, w = z0 + Phi^-1(q), and the bounds taken at the levels
 * Phi(z0 + w / (1 - a w)).  q = 0 / 1 give the minimum / maximum; the bound is NaN where 1 - a w <= 0 (or a is NaN),
 * where prop is 0 or 1, and for a NaN theta (whose prop is NaN).  a = 0 gives the BC bounds.
 * Workspace: plsb200_percentile_f64_workspace(B).                                                                   */
int plsb200_percentile_bca_f64(const double* samples, int B, int64_t nseries, int64_t stride_sample,
                               int64_t stride_series, const double* orig, const double* accel, double q_lo,
                               double q_hi, double* lower, double* upper, double* prop, void* workspace,
                               size_t workspace_bytes, void* stream);
/* the stratified jackknife acceleration of nseries series S[s][j] (J contiguous samples each, s-major), the samples
 * in G groups [goff[g], goff[g+1]) (goff: G + 1 int32 in device memory, goff[0] = 0, goff[G] = J, every group
 * non-empty).  With d_j = S[s][j] - theta[s], m_g the mean of d over group g (n_g samples) and
 * l_j = (n_g - 1)(m_g - d_j):  accel[s] = (1/6) sum_g n_g^-3 sum l^3 / (sum_g n_g^-2 sum l^2)^(3/2), 0 where the
 * denominator is 0 (NaN where it is NaN).  theta is only a pivot: a does not depend on it.                       */
int plsb200_jack_accel_f64(const double* S, int64_t nseries, int J, const int32_t* goff, int G, const double* theta,
                           double* accel, void* stream);

/* ---- explicit saliences for a small batch: VS[r] = X^T . C_r  (R x p x K), for callers that ask for
 * boot_debug_dict["right_sv_sampled"] on problems small enough to hold it.                          */
int plsb200_salience_f64(const double* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                         const int32_t* idx, int R, double* VS, void* stream);
int plsb200_salience_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                             const int32_t* idx, int R, double* VS, void* stream);
/* the same saliences series-major, VS[v][k][r] (p x K x R): the R samples of an element are contiguous, which is the
 * layout plsb200_percentile_f64 sorts fastest (stride_sample = 1, stride_series = R); p <= 65535 * 128 per call.   */
int plsb200_salience_series_f64(const double* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                                const int32_t* idx, int R, double* VS, void* stream);
int plsb200_salience_series_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* E, int K,
                                    const int32_t* idx, int R, double* VS, void* stream);
/* saliences over explicit per-sample coefficients, series-major: VS[v][k][j] = sum_i X[i, v] . C[j][i][k] (C: J x N x K,
 * VS: p x K x J), the leave-one-subject-out jackknife of the saliences (C zero on the removed rows).  X is read in
 * place through ldx, so a voxel window is X + v0; p <= 65535 * 128 per call, N K <= 25600.                      */
int plsb200_salience_coef_series_f64(const double* X, int N, int64_t p, int64_t ldx, const double* C, int K, int J,
                                     double* VS, void* stream);
int plsb200_salience_coef_series_x32_f64(const float* X, int N, int64_t p, int64_t ldx, const double* C, int K, int J,
                                         double* VS, void* stream);

/* ---- K5: behaviour PLS (rb / csb) -----------------------------------------------------------------
 * Cells = (group, condition) blocks of consecutive rows, given as ncell+1 int32 offsets `cell_start`.
 *
 * cell_standardize: Xc = X - block means, Z = Xc / (block sd * sqrt(n)) (0 where sd == 0): the X half of
 *   `_compute_corr` (class_functions.py:221-238), done once per analysis.  Xc, Z: N x p dense (Z may be NULL).
 * nspace_coef: like plsb200_nspace_f64 but with an explicit coefficient matrix per resample
 *   (C: R x N x K): d2[r,k] = C_r[:,k]^T G C_r[:,k].  With G = Z Z^T this is the permuted behaviour PLS
 *   singular-value estimate (bootstrap_permutation.py:395-405, 429-437; only Y is permuted).
 * rb_coef: per resample, Ynew = Y[idx] (idx may be NULL = identity), z-scored inside every block;
 *   Q[r] (N x Kc) = pull-back of the design weights U (ncell*nb x Kc) to row space;
 *   scatter = 0: permutation (X rows stay), scatter = 1: bootstrap (X rows gathered by the same idx;
 *   W[r] (N) = multiplicity / block size).  Yz (R x N x nb, optional) = the z-scored resampled Y.
 * rb_boot: the p-space bootstrap pass for bootstraps [b0, b0+nbt): VS_b = R_b^T U with the per-voxel
 *   block std of the RESAMPLED rows (class_functions.py:219-245 as called at bootstrap_permutation.py:613);
 *   accumulates sum/sumsq of (VS - pivot) INTO sum/sumsq (p x K, caller zeroes before the first chunk) and
 *   writes T[b] = Xc . VS_b (N x K) and nrm2[b] = ||VS_b[:,k]||^2 for the LV correlations.
 *   The `_vs` variants also store VS_b itself (the reference's right_sv_sampled[b], before the pivot is subtracted)
 *   into VS, resample-major like T: VS[b * p * K + v * K + k] for b in [b0, b0+nbt), p x K per bootstrap.  The
 *   plain entry points are the `_vs` ones with VS = NULL (nothing stored).
 * rb_lvcorr: LVcorr[b] = _compute_corr(X_new @ V_hat, Y_new) (ncell*nb x K)  (bootstrap_permutation.py:636-642). */
int plsb200_cell_standardize_f64(const double* X, int N, int64_t p, int64_t ldx, const int32_t* cell_start,
                                 int ncell, double* Xc, double* Z, void* stream);
/* The N-space pass on the FP64 tensor cores (N <= 320, K <= 24): same outputs as plsb200_nspace_f64 from the PACKED
 * coefficients of plsb200_boot_coef_pack_f64 (the tensor the exact bootstrap GEMM streams, so one pack serves both):
 * H = G^T [C_1 | C_2 | ...] as a DMMA GEMM with G as the register-resident operand, d2 and T = Lmat H diag(1/sqrt(d2))
 * from its epilogue.  T may be NULL (then Lmat NULL, Kt 0).  The workspace query returns 0 when the shape is not
 * supported (use plsb200_nspace_f64).                                                                            */
size_t plsb200_nspace_dmma_f64_workspace(int N, int K, int Kt, int R);
int plsb200_nspace_dmma_f64(const double* G, int N, const double* Lmat, int Kt, const double* coef, int K, int R,
                            double* d2, double* T, void* workspace, size_t workspace_bytes, void* stream);
int plsb200_nspace_coef_f64(const double* G, int N, const double* C, int K, int R, const double* Lmat, int Kt,
                            double* d2, double* T, void* stream);
/* B[r] = C_r^T G C_r (R x K x K) for explicit coefficients: the Gram matrix of a resampled behaviour / multiblock
 * cross-block matrix (rows = columns of C_r), input of the per-permutation SVD mode (rotate_method = 0) through
 * plsb200_sym_eig_f64.  N x K must fit one shared-memory chunk (2 N K doubles <= 200 KB).                       */
int plsb200_nspace_coef_gram_f64(const double* G, int N, const double* C, int K, int R, double* d2, double* B,
                                 void* stream);
int plsb200_rb_coef_f64(const double* Y, int N, int nb, const int32_t* idx, int R, const int32_t* cell_start,
                        int ncell, const double* U, int Kc, int scatter, double* Q, double* W, double* Yz,
                        void* stream);
size_t plsb200_rb_boot_f64_workspace(int N, int64_t p, int K, int nbt);
 /* (the data matrix of rb_boot may be given as two row segments: rows [0, n1) = Xc (row stride p), rows [n1, N) = Xc2
  * (row stride ld2); Xc2 == NULL: all N rows in Xc.  The multiblock bootstrap passes [Xcb; X] this way.)          */
int plsb200_rb_boot_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2, const double* Q,
                        const double* W, int K, int b0,
                        int nbt, const int32_t* cell_start, int ncell, int unit_cells, const double* pivot,
                        double* sum, double* sumsq, double* T, double* nrm2, void* workspace,
                        size_t workspace_bytes, void* stream);
int plsb200_rb_boot_vs_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2, const double* Q,
                           const double* W, int K, int b0,
                           int nbt, const int32_t* cell_start, int ncell, int unit_cells, const double* pivot,
                           double* sum, double* sumsq, double* T, double* nrm2, double* VS, void* workspace,
                           size_t workspace_bytes, void* stream);
/* rb_boot on the FP64 tensor path (DMMA): same contract as plsb200_rb_boot_f64 except that the block offsets are
 * read on the HOST (`cell_start_host`), T may be NULL (squared norms only: first pass of the multiblock bootstrap)
 * and designs whose blocks, each padded to a multiple of 4 rows, exceed 384 rows are not supported: the workspace
 * query then returns 0 and the caller uses plsb200_rb_boot_f64.  Phase 1 keeps X fragments register-resident and
 * streams packed coefficients like the K4 kernel; the latent products T = Xc . VS are a split-K DMMA GEMM.     */
size_t plsb200_rb_boot_dmma_f64_workspace(int N, int64_t p, int K, int nbt, const int32_t* cell_start_host,
                                          int ncell, int unit_cells, int want_t);
int plsb200_rb_boot_dmma_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2,
                             const double* Q, const double* W, int K, int b0,
                             int nbt, const int32_t* cell_start_host, int ncell, int unit_cells, const double* pivot,
                             double* sum, double* sumsq, double* T, double* nrm2, void* workspace,
                             size_t workspace_bytes, void* stream);
int plsb200_rb_boot_dmma_vs_f64(const double* Xc, int N, int64_t p, const double* Xc2, int n1, int64_t ld2,
                                const double* Q, const double* W, int K, int b0,
                                int nbt, const int32_t* cell_start_host, int ncell, int unit_cells, const double* pivot,
                                double* sum, double* sumsq, double* T, double* nrm2, double* VS, void* workspace,
                                size_t workspace_bytes, void* stream);
/* rb_salience: the export-only pass of rb_boot over the voxel window [v0, v1): VS[b][v - v0][k] (nbt x (v1 - v0) x K,
 * resample-major, the reference's right_sv_sampled[b, v0:v1]) for the bootstraps [0, nbt) of Q / W, bit-identical to
 * the VS of the `_vs` entry points; no moments, norms or latent products.  The first row segment Xc has the row stride
 * ld1 (the second, if any, ld2 >= v1), so a window is read in place.
 * The DMMA path packs the coefficients of all nbt bootstraps once (plsb200_rb_salience_dmma_pack_f64 into the
 * workspace) and every window's launch reads them; its workspace query returns 0 for a design the DMMA kernels do not
 * hold, as plsb200_rb_boot_dmma_f64_workspace does, and the caller uses plsb200_rb_salience_f64 (cell_start in device
 * memory, no workspace).                                                                                          */
size_t plsb200_rb_salience_dmma_f64_workspace(int N, int K, int nbt, const int32_t* cell_start_host, int ncell,
                                             int unit_cells);
int plsb200_rb_salience_dmma_pack_f64(const double* Q, const double* W, int N, int K, int nbt,
                                      const int32_t* cell_start_host, int ncell, int unit_cells, void* workspace,
                                      size_t workspace_bytes, void* stream);
int plsb200_rb_salience_dmma_f64(const double* Xc, int N, int64_t ld1, const double* Xc2, int n1, int64_t ld2,
                                 int64_t v0, int64_t v1, int K, int nbt, const int32_t* cell_start_host, int ncell,
                                 int unit_cells, double* VS, const void* workspace, size_t workspace_bytes, void* stream);
int plsb200_rb_salience_f64(const double* Xc, int N, int64_t ld1, const double* Xc2, int n1, int64_t ld2, int64_t v0,
                            int64_t v1, const double* Q, const double* W, int K, int nbt, const int32_t* cell_start,
                            int ncell, int unit_cells, double* VS, void* stream);
/* multiblock glue (class_functions.py:454-516): the last `unit_cells` blocks of rb_boot are plain linear rows
 * (task part of the multiblock matrix, no standardisation).
 * scatter_coef: C[r] (N x K) = scatter(E, idx_r) written out explicitly.
 * coef_project: C2[r] (N x K) = C1[r] (N x M) . diag(1/sqrt(d2[r])) . Uc (M x K): row-normalise the M multiblock
 *   rows (d2 = their squared norms) and project on the design weights.                                */
int plsb200_scatter_coef_f64(const double* E, int N, int K, const int32_t* idx, int R, double* C, void* stream);
int plsb200_coef_project_f64(const double* C1, int N, int M, const double* d2, const double* Uc, int K, int R,
                             double* C2, void* stream);
int plsb200_rb_lvcorr_f64(const double* T, const double* nrm2, const double* Yz, const int32_t* idx, int N, int nb,
                          int K, int R, const int32_t* cell_start, int ncell, double* LVcorr, void* stream);

/* ---- split-half Gram blocks in p-space (behaviour / multiblock family) -----------------------------
 * For splits [s0, s0+ns): half h of split s is a list of nmax positions -> data rows `ids[s][h][pos]`, cut
 * into `ncell` blocks by the position offsets `cells[h][0..ncell]` (the same for every split); rows of
 * standardised blocks come from Xstd, those of the trailing `unit_cells` blocks from Xlin (both N x p dense).
 * Q[s][h][pos][k] are the per-position coefficients of the K rows of the half's cross-block matrix.
 * Output S3[s] = [S11 | S12 | S22] (3 x K x K): M1 M1^T, M1 M2^T, M2 M2^T.  K <= 24.
 * (split_half_resampling.py:198-262, 315-383, 615-683, 734-802)                                       */
size_t plsb200_half_gram_f64_workspace(int64_t p, int K, int ns);
int plsb200_half_gram_f64(const double* Xstd, const double* Xlin, int64_t p, const int32_t* ids, const double* Q,
                          const int32_t* cells, int ncell, int unit_cells, int nmax, int K, int s0, int ns,
                          double* S3, void* workspace, size_t workspace_bytes, void* stream);

/* Windowed version of the same quantity (half_gram.cu; preferred, K <= 32): instead of `cells`, each half carries
 * `nseg` segments  segs[h][s] = {pos_begin, pos_end, col0, width, unit, qoff}  (device, int32 x 6): the positions
 * [pos_begin, pos_end) form one block (standardised over its member rows unless `unit`), and only the columns
 * [col0, col0 + width), width <= 8, of Q are non-zero for them.  Inside the kernel a half's window coefficients
 * are packed, wq = width rounded up to 1, 2, 4, 8 doubles per position; `qoff` is the (even) offset of the segment
 * in that packing and `nq` (even) its total length in doubles.  Q keeps the dense S x 2 x nmax x K layout; columns
 * outside the windows are not read.  Phase 1 costs `width` FMAs per position instead of K, the 2K x 2K Gram of a
 * voxel tile runs on DMMA.                                                                                    */
size_t plsb200_half_gram_win_f64_workspace(int64_t p, int K, int ns);
int plsb200_half_gram_win_f64(const double* Xstd, const double* Xlin, int64_t p, const int32_t* ids, const double* Q,
                              const int32_t* segs, int nseg, int nq, int nmax, int K, int s0, int ns, double* S3,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- K3: batched symmetric eigensolver, one-sided (Hestenes) Jacobi.  K <= 32: one warp per K x K matrix, columns
 * in registers, shuffle-based rotations.  32 < K <= 112: one CTA per matrix, columns in shared memory, the K/2
 * disjoint pairs of a tournament round rotated by K/2 warps in parallel.  Replaces np.linalg.svd of the K x p
 * half-sample cross-block matrices (class_functions.py:122 as called from
 * split_half_resampling.py:194,207,255,311,612-613,...) through their K x K Gram matrices.
 * A: B x K x K symmetric PSD.  evals: B x K descending.  evecs: B x K x K row-major, eigenvectors in COLUMNS.
 * status (B int32, may be NULL): 0 = converged, 1 = sweep limit reached (results must not be used).
 * K > 112: PLSB200_EUNSUPPORTED.                                                                      */
int plsb200_sym_eig_f64(const double* A, int K, int B, double* evals, double* evecs, int32_t* status, void* stream);

/* ---- Gram blocks of S split-half resamples through G (task methods).
 * Half h of split s consists of the rows idx_h[s, 0..n_h) of X (null splits: rows of the permuted X,
 * i.e. composed indices); its cross-block matrix is M_h = A_h (K x n_h) . X[idx_h].  Outputs
 * S11 = M1 M1^T, S12 = M1 M2^T, S22 = M2 M2^T, each S x K x K.
 * (split_half_resampling.py:172-196, 289-313, 590-613, 709-732)                                    */
int plsb200_split_gram_f64(const double* G, int N, const int32_t* idx1, int n1, const int32_t* idx2, int n2,
                           int S, const double* A1, const double* A2, int K, double* S11, double* S12,
                           double* S22, void* stream);

/* ---- split-half outputs from the Gram blocks (SVD methods; K <= 112).  With S11 = U1 diag(s1^2) U1^T,
 * S22 = U2 diag(s2^2) U2^T (singular values descending):
 *   s_train (S x K)     = s1                                   (split_half_resampling.py:195)
 *   s_test  (S x K x K) = V1^T M2^T U1 = diag(1/s1) U1^T S12 U1 (:196)
 *   u_repro (S x K x K) = V1^T V2 = diag(1/s1) U1^T S12 U2 diag(1/s2)   (:682)
 *   v_repro (S x K x K) = U1^T U2                              (:683)
 *   s2      (S x K)     = s2
 * Any output pointer may be NULL.  Rows/columns belonging to zero singular values are written as 0
 * (LAPACK returns an arbitrary orthonormal completion there).  Signs of singular vectors are not
 * those of LAPACK: compare up to the sign of each latent variable.
 * status (S int32, may be NULL): 1 where one of the two eigensolves of split s did not converge.
 * K > 32 needs a workspace of plsb200_split_svd_f64_workspace(K, S) bytes (the eigenpairs of S11 and S22).  */
size_t plsb200_split_svd_f64_workspace(int K, int S);
int plsb200_split_svd_f64(const double* S11, const double* S12, const double* S22, int K, int S,
                          double* s_train, double* s_test, double* u_repro, double* v_repro, double* s2,
                          int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* ---- host-side resampling index generator (no GPU work) -------------------------------------------------
 * Continues numpy's legacy global MT19937 stream -- `key` = the 624 state words, `*pos` = the position, both as
 * returned by np.random.get_state() and updated in place -- with numpy's own algorithms (masked-rejection
 * random_interval, RandomState.shuffle, RandomState.choice), so the index matrices are bit-identical to what
 * the reference draws through resample_without_replacement / resample_with_replacement
 * (plspy/core/resample.py:44-79, 125-160; call order SURVEY.md App. B) at ~100x the speed of the numpy calls.
 * cond_order: G x C int32 (subjects per group and condition; must be constant within a group, else
 * PLSB200_EUNSUPPORTED and the caller falls back to numpy).
 *  task_permutations: count x N task-method permutation index vectors; beh_rows > 0 adds, after every draw, one
 *    np.random.permutation(beh_rows) for the multiblock behaviour block (bootstrap_permutation.py:342-347).
 *  bootstrap_draws: count x N bootstrap index vectors; cond_order2 != NULL adds the independent behaviour-block
 *    draw of the multiblock methods (bootstrap_permutation.py:545-554).
 *  row_permutations: count x n, np.random.permutation(n) each (behaviour PLS, :337-340).
 *  split_draws: the draws of one split-half routine (plspy/core/split_half_resampling.py:136, 271, 282 and :555,
 *    692, 703): `count` real splits of one permutation(group_sizes[g]) per group -> out_real (count x sum of sizes,
 *    groups side by side), then `count` null splits of permutation(nsub) -> out_null_subj (count x nsub) followed by
 *    permutation(n_rows) -> out_null_rows (count x n_rows).                                                  */
int plsb200_host_task_permutations(uint32_t* key, int32_t* pos, const int32_t* cond_order, int G, int C,
                                   int beh_rows, int count, int32_t* out_task, int32_t* out_beh);
int plsb200_host_bootstrap_draws(uint32_t* key, int32_t* pos, const int32_t* cond_order, int G, int C,
                                 const int32_t* cond_order2, int C2, int count, int32_t* out, int32_t* out2);
int plsb200_host_row_permutations(uint32_t* key, int32_t* pos, int n, int count, int32_t* out);
int plsb200_host_split_draws(uint32_t* key, int32_t* pos, const int32_t* group_sizes, int G, int nsub, int n_rows,
                             int count, int32_t* out_real, int32_t* out_null_subj, int32_t* out_null_rows);

#ifdef __cplusplus
}
#endif
#endif /* PLSB200_H */
