/* vittles_b200 - C ABI of the B200-native sensitivity hot path.
 *
 * The reference (rgiordan/vittles) is pure Python: it has no FFI or plugin
 * registry.  Its seam is the solver-closure protocol `solve(v) -> H^{-1} v`
 * (vittles/solver_lib.py:22-30) plus the constructors exported from
 * vittles/__init__.py:1-8.  This header is the boundary a maintainer would
 * bind (ctypes stub in INTEGRATION.md) to move the arithmetic behind those
 * Python entry points onto a B200.  Each function cites the reference code it
 * replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to float64 unless stated otherwise;
 *     matrices are row-major with an explicit leading dimension (elements);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous with
 *     respect to the host unless stated otherwise;
 *   - the return value is 0 on success or a VT_ERR_* code; the message of the
 *     last failure on the calling thread is returned by vt_last_error();
 *   - the library never allocates device memory: workspaces are sized by the
 *     *_workspace_bytes queries and owned by the caller, and it keeps no state
 *     between calls.  (One exception: vt_potrf with four or more block
 *     columns runs its large trailing updates on a helper stream - created
 *     lazily once per host thread and device, fenced against `stream` by
 *     events, and joined before the call returns.)
 */
#ifndef VITTLES_B200_H
#define VITTLES_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VT_OK 0
#define VT_ERR_CUDA 1            /* CUDA runtime / launch failure            */
#define VT_ERR_INVALID 2         /* bad argument -> ValueError upstream      */
#define VT_ERR_NOT_PD 3          /* non-positive pivot -> LinAlgError        */
#define VT_ERR_NO_CONVERGENCE 4  /* CG hit maxiter -> UserWarning upstream   */

#define VT_GLM_LOGISTIC 0
#define VT_GLM_POISSON 1
#define VT_GLM_GAUSSIAN 2

#define VT_OP_KC 0 /* operand element (r,k) at p[r*ld + k]  (k contiguous) */
#define VT_OP_KS 1 /* operand element (r,k) at p[k*ld + r]  (k strided)    */

const char* vt_last_error(void);
int vt_abi_version(void);
/* Number of kernels this library has launched in the process so far. */
int64_t vt_launch_count(void);
/* SM count and compute capability of the current device. */
int vt_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Runs a register-resident DMMA loop for about `seconds` and returns the
 * achieved FP64 tensor TFLOP/s: the roofline denominator bench.py reports
 * (MEASURED_PEAKS.json has no FP64 entry).  Synchronous. */
int vt_fp64_peak_probe(double seconds, double* tflops, void* stream);
/* Runs a bare tcgen05.mma.kind::i8 loop (M = 128, N = n_tile in 16..256, K = 32;
 * operands resident in shared memory, no loads) for about `seconds` and
 * returns the achieved dense INT8 TOP/s and the SM clocks per 128 x n_tile x 32
 * instruction (may be NULL): the roofline denominator of the
 * error-free-slicing engine (MEASURED_PEAKS.json has no INT8 entry).  Synchronous. */
int vt_i8_peak_probe(double seconds, int n_tile, double* tops, double* clocks_per_mma, void* stream);

/* ---- FP64 tensor-core GEMM engine ---------------------------------------
 * C(m,n) = alpha * rowscale[m] * colscale[n] * sum_k kscale[k] A(m,k) B(n,k) + beta * C(m,n)
 * (scale vectors may be NULL; kscale requires both operands in VT_OP_KS).
 * lower != 0: only the lower triangle of a square C is produced; mirror != 0
 * additionally writes the transposed entries (exactly symmetric result).
 * `tile` selects the CTA tile edge (128: throughput configuration, 64: short-K
 * / few-tile / ragged problems; 0: chosen from the shape).
 * Replaces the numpy `@` / einsum GEMMs at sensitivity_lib.py:67,76,247 and
 * lr_cov_lib.py:172 and is the engine under every routine below.            */
size_t vt_dgemm_workspace_bytes(int M, int N, int K, int lower, int tile);
int vt_dgemm(int M, int N, int K, double alpha, const double* A, int64_t lda, int amode, const double* B,
             int64_t ldb, int bmode, double beta, double* C, int64_t ldc, const double* kscale,
             const double* colscale, const double* rowscale, int lower, int mirror, int tile, void* workspace,
             size_t workspace_bytes, void* stream);

/* ---- Hessian assembly ----------------------------------------------------
 * H = X^T diag(s) X + l2 * I for X (N x D).  Replaces
 * autograd.hessian(objective)(theta, w) for GLM objectives
 * (sensitivity_lib.py:381-383, lr_cov_lib.py:102).  Deterministic split-K.   */
size_t vt_syrk_workspace_bytes(int64_t N, int D);
int vt_syrk_weighted(const double* X, int64_t ldx, int64_t N, int D, const double* s, double l2, double* H,
                     int64_t ldh, void* workspace, size_t workspace_bytes, void* stream);

/* ---- GLM passes over X (HBM bound, one read of X each) --------------------
 * vt_glm_stats: z = X theta, resid = b'(z) - y, s = w b''(z),
 *               grad = X^T (w resid) + l2 theta   (sensitivity_lib.py:354 grad;
 *               the optimum check at :203-215).  Outputs may be NULL.
 * vt_glm_hvp:   out = X^T (s .* (X v)) + ridge v  - the mat_times_vec handed
 *               to get_cg_solver (solver_lib.py:76-79,91).
 * vt_glm_dirderiv: out = X^T (w .* b^{(q+1)}(z) .* prod_j X dirs_j), the
 *               closed form of the nested JVPs of
 *               ForwardModeDerivativeArray.eval_directional_derivative
 *               (sensitivity_lib.py:788-807) for q eta-directions.           */
size_t vt_glm_workspace_bytes(int D);
int vt_glm_stats(const double* X, int64_t ldx, int64_t N, int D, const double* theta, const double* y,
                 const double* w, int family, double* z, double* resid, double* s, double* grad, double l2,
                 void* workspace, size_t workspace_bytes, void* stream);
/* vt_glm_stats that also writes sq[n] = sqrt(s_n) and colmax[c] = the bit pattern of max_n sq_n |x_nc| (D <= 2048;
 * workspace of 2 x vt_glm_workspace_bytes): the per-feature scales of the INT8 Hessian assembly (vt_syrk_ozaki)
 * come out of the statistics pass instead of a sweep of their own. */
int vt_glm_stats_colmax(const double* X, int64_t ldx, int64_t N, int D, const double* theta, const double* y,
                        const double* w, int family, double* z, double* resid, double* s, double* grad, double l2,
                        double* sq, uint64_t* colmax, void* workspace, size_t workspace_bytes, void* stream);
/* q <= 4 Hessian-vector products in ONE pass over X: out (q x D) = V X^T diag(s) X + ridge V, V (q x D)
 * row-major - the shared mat_times_vec of a multi-right-hand-side CG (D <= 2048 for q > 1). */
size_t vt_glm_hvp_multi_workspace_bytes(int D, int q);
int vt_glm_hvp_multi(const double* X, int64_t ldx, int64_t N, int D, const double* s, const double* V, int q,
                     double ridge, double* out, void* workspace, size_t workspace_bytes, void* stream);
int vt_glm_hvp(const double* X, int64_t ldx, int64_t N, int D, const double* s, const double* v, double ridge,
               double* out, void* workspace, size_t workspace_bytes, void* stream);
size_t vt_glm_dirderiv_workspace_bytes(int64_t N, int D);
int vt_glm_dirderiv(const double* X, int64_t ldx, int64_t N, int D, const double* z, const double* w, int family,
                    const double* dirs, int q, double* out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Per-observation influence on quantities of interest -----------------
 * out[k * ldo + n] = alpha * c[n] * (x_n . V[k, :]) for k < K, n < N: with c = resid, V = rows of H^{-1} A^T and
 * alpha = -1, row k of out is a_k^T S, the influence of every observation on the quantity of interest a_k, without
 * forming S (D x N).  One pass over X (ldx >= D), K values written per row, no workspace; V (K x D) row-major and
 * contiguous, out (K x N) row-major with ldo >= N.  K <= vt_glm_influence_max_directions(D): 8 up to D = 2048, 2 up
 * to 4096, 1 up to 8192, 0 beyond (D > 8192 is refused with VT_ERR_INVALID).  Bitwise reproducible.              */
int vt_glm_influence_max_directions(int D);
int vt_glm_influence(const double* X, int64_t ldx, int64_t N, int D, const double* c, const double* V, int K,
                     double alpha, double* out, int64_t ldo, void* stream);

/* ---- Dense Cholesky solver -------------------------------------------------
 * vt_potrf / vt_potrs replace scipy.linalg.cho_factor / cho_solve behind
 * get_dense_cholesky_solver (solver_lib.py:27,29).  A is overwritten by its
 * lower factor; `dinv` (vt_potrf_dinv_doubles(D) doubles) receives the inverted
 * 128x128 diagonal blocks used by the solve (followed by a D x 128 scratch
 * panel of the factorisation); *info (device int32) is 0 or the
 * 1-based column of the first non-positive pivot (LinAlgError upstream).
 * vt_potrs solves in place for a row-major D x K right-hand side.            */
size_t vt_potrf_dinv_doubles(int D);
int vt_potrf(double* A, int64_t lda, int D, double* dinv, int32_t* info, void* stream);
int vt_potrs(const double* L, int64_t ldl, int D, const double* dinv, double* B, int64_t ldb, int K, void* stream);
/* One half of vt_potrs, in place: B <- L^{-1} B (transpose = 0) or L^{-T} B
 * (transpose = 1).  Forward then backward gives the bits of vt_potrs.        */
int vt_trsm_lower(const double* L, int64_t ldl, int D, const double* dinv, double* B, int64_t ldb, int K, int transpose,
                  void* stream);

/* ---- Quadratic forms of the inverse Hessian ---------------------------------
 * out[n] = |Linv x_n|^2 = x_n^T H^{-1} x_n for H = L L^T, Linv = L^{-1} (D x D,
 * lower triangular: zero above the diagonal), x_n the rows of X (N x D): the
 * leverage terms of approximate leave-one-out cross-validation.  A sum of
 * squares, so no cancellation; nothing of size D x N is written.
 * vt_quad_forms runs on the FP64 DMMA engine (U = X_c Linv^T per chunk of rows,
 * then the row sums of squares); vt_quad_forms_ozaki on the INT8 slicing
 * engine (the chunks of vt_ij_apply_ozaki, squares summed in the GEMM's
 * epilogue, row block tm of Linv meeting its k-blocks 0 .. tm only).  Both sum
 * in a fixed order: two calls give the same bits.                           */
size_t vt_quad_forms_workspace_bytes(int64_t N, int D);
int vt_quad_forms(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D, double* out,
                  void* workspace, size_t workspace_bytes, void* stream);
size_t vt_quad_forms_ozaki_workspace_bytes(int64_t N, int D, int nslices);
int vt_quad_forms_ozaki(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D, double* out,
                        int nslices, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Leave-one-group-out predictors -----------------------------------------
 * Groups are runs of consecutive rows: group g is rows starts[g] .. starts[g+1]-1
 * (starts: G + 1 int64, strictly increasing from 0 to N, consecutive entries at
 * most 32 apart; the caller checks this).  For a group R, Q = X_R H^{-1} X_R^T
 * = U_R^T U_R with U = Linv X^T (Linv as for vt_quad_forms), t = Q u_R, and
 *   h[n]     = Q_nn = x_n^T H^{-1} x_n
 *   method 0 (IJ):          zpred_R = z_R + t
 *   method 1 (Newton step): zpred_R = z_R + t + Q S^1/2 M^{-1} S^1/2 t,
 *                           M = I - S^1/2 Q S^1/2, S = diag(s_R)
 * NaN on every row of a group when a pivot of the Cholesky factor of M, squared,
 * is <= 2^-40.  vt_group_loo runs U on the DMMA engine (rows x D per chunk),
 * vt_group_loo_ozaki on the INT8 slicing engine (the chunks of
 * vt_ij_apply_ozaki); both then form each group's Q in one kernel.  Chunks
 * overlap by 32 rows, so no group is split; nothing of size D x N is written.
 * Both sum in a fixed order: two calls give the same bits.                   */
size_t vt_group_loo_workspace_bytes(int64_t N, int D);
int vt_group_loo(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D,
                 const int64_t* starts, int64_t G, const double* s, const double* u, const double* z, int method,
                 double* zpred, double* h, void* workspace, size_t workspace_bytes, void* stream);
size_t vt_group_loo_ozaki_workspace_bytes(int64_t N, int D, int nslices);
int vt_group_loo_ozaki(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D,
                       const int64_t* starts, int64_t G, const double* s, const double* u, const double* z, int method,
                       double* zpred, double* h, int nslices, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Infinitesimal-jackknife apply ----------------------------------------
 * S (D x N) = -Hinv (D x D) * G^T, column n of G^T being resid[n] * x_n, fused
 * so that the cross-Hessian G^T is never materialised.  Replaces
 * `_sens_mat = -hess_solver(cross_hess)` (sensitivity_lib.py:226) for
 * lambda := per-observation weights.                                        */
int vt_ij_apply(const double* Hinv, int64_t ldh, const double* X, int64_t ldx, int64_t N, int D,
                const double* resid, double* S, int64_t lds, void* stream);

/* ---- Optional reduced-precision path: TF32 on tcgen05 / TMEM / TMA -----------
 * The north_star's "optional FP32/TF32 path" for the two contractions.  FP64
 * (above) is the default and the only path the rtol 1e-8 parity bar applies to;
 * these entry points are used only when the caller asks for precision 'tf32'
 * (one TF32 product, ~1e-3 of the operand scale) or 'tf32x3' (three-term hi/lo
 * split, ~1e-6).  split = 1 | 3 selects between them.
 * vt_tf32_convert: hi = tf32(scale_r * x) stored as FP32 (+ lo = tf32 of the
 *   remainder if lo != NULL); scale_r = rowscale[r] or sqrt(rowscale[r]);
 *   ldo % 4 == 0, pad columns are zero-filled.
 * vt_tf32_gemm: C (FP64) = alpha * rowscale[m] * colscale[n] * sum_k A(m,k) B(n,k)
 *   on tcgen05.mma.kind::tf32 with FP32 accumulation in TMEM, flushed to FP64
 *   every 4096 k; operand modes as for vt_dgemm (both operands the same mode).
 * vt_ij_apply_tf32 / vt_syrk_tf32: the two hot contractions with FP64 inputs
 *   and outputs; the observations are converted chunk by chunk inside.        */
size_t vt_tf32_gemm_workspace_bytes(int M, int N, int64_t K, int split);
int vt_tf32_convert(const double* X, int64_t ldx, int64_t rows, int cols, const double* rowscale, int sqrt_scale,
                    float* hi, float* lo, int64_t ldo, void* stream);
int vt_tf32_gemm(int M, int N, int64_t K, double alpha, const float* A_hi, const float* A_lo, int64_t lda, int amode,
                 const float* B_hi, const float* B_lo, int64_t ldb, int bmode, double* C, int64_t ldc,
                 const double* colscale, const double* rowscale, void* workspace, size_t workspace_bytes,
                 void* stream);
size_t vt_ij_apply_tf32_workspace_bytes(int64_t N, int D, int split);
int vt_ij_apply_tf32(const double* Hinv, int64_t ldh, const double* X, int64_t ldx, int64_t N, int D,
                     const double* resid, double* S, int64_t lds, int split, void* workspace,
                     size_t workspace_bytes, void* stream);
size_t vt_syrk_tf32_workspace_bytes(int64_t N, int D, int split);
int vt_syrk_tf32(const double* X, int64_t ldx, int64_t N, int D, const double* s, double l2, double* H, int64_t ldh,
                 int split, void* workspace, size_t workspace_bytes, void* stream);

/* ---- FP64-grade contraction on the INT8 tensor cores (error-free slicing) ------
 * An additional engine for the H^{-1} G^T apply (precision 'f64_ozaki'): every
 * row of both operands is scaled by a power of two and cut into `nslices`
 * (5..7) balanced base-256 digits in [-128, 127] (vt_ozaki_slice: out[s][r][k]
 * int8, scale_out[r] = 2^e_r * fold[r]); the nslices (nslices + 1) / 2
 * significant digit products run exactly on tcgen05.mma.kind::i8 with INT32
 * accumulators in TMEM and are recombined in INT64 / FP64 in the epilogue
 * (vt_ozaki_gemm, K <= 16384).  With 7 slices (54 bits) the result is within
 * ~1e-14 of sigma_m tau_n K (the row scales), inside the rtol 1e-8 parity bar
 * of the FP64 path.  vt_ij_apply_ozaki is vt_ij_apply on this engine; the
 * observations are sliced chunk by chunk by converter warps inside the GEMM
 * kernel.  Every slicer, in the GEMM kernel or standing alone, forms the
 * digits with integer instructions only, from the bit patterns (FP64
 * instructions starve while the tensor pipe is saturated), so every digit
 * is formed the same way.  vt_ozaki_slice_t writes the Hessian's operand:
 * digits of sq[n] * X[n][i] TRANSPOSED, out[s][i][n], one scale per feature
 * from colmax[i] (the bit pattern of max_n |sq[n] X[n][i]|).               */
int vt_ozaki_slice(const double* X, int64_t ldx, int64_t rows, int cols, int8_t* out, int64_t ldo, int64_t slice_stride,
                   int nslices, double* scale_out, const double* fold, void* stream);
int vt_ozaki_slice_t(const double* X, int64_t ldx, int64_t rows, int cols, const double* sq, const uint64_t* colmax,
                     int8_t* out, int64_t ldo, int64_t slice_stride, int nslices, double* scale_out, void* stream);
int vt_ozaki_gemm(int M, int N, int K, const int8_t* A, int64_t lda, int64_t a_slice_stride, const int8_t* B,
                  int64_t ldb, int64_t b_slice_stride, int nslices, double alpha, const double* rowscale,
                  const double* colscale, double* C, int64_t ldc, void* stream);
/* vt_syrk_ozaki is vt_syrk_weighted (s >= 0) on the same engine: the contraction runs over the
 * observations, so the digits of sqrt(s_n) x_ni are written transposed with one power-of-two
 * scale per feature and per chunk of observations, and the chunks' lower-triangular Gram tiles
 * (split-K parts of <= 16384 observations: the INT32 bound) are accumulated in FP64.
 * sq / colmax (both NULL, or both given): sqrt(s_n) and the column maxima of sqrt(s_n) |x_ni| as
 * written by vt_glm_stats_colmax - the sweep over X that would compute them is then skipped.   */
size_t vt_syrk_ozaki_workspace_bytes(int64_t N, int D, int nslices);
int vt_syrk_ozaki(const double* X, int64_t ldx, int64_t N, int D, const double* s, double l2, double* H, int64_t ldh,
                  int nslices, const double* sq, const uint64_t* colmax, void* workspace, size_t workspace_bytes,
                  void* stream);
size_t vt_ij_apply_ozaki_workspace_bytes(int64_t N, int D, int nslices);
int vt_ij_apply_ozaki(const double* Hinv, int64_t ldh, const double* X, int64_t ldx, int64_t N, int D,
                      const double* resid, double* S, int64_t lds, int nslices, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ---- Prediction GEMV --------------------------------------------------------
 * y = alpha * A x + beta * y0 for row-major A (M x N), N long:
 * theta_hat + S (lam1 - lam0)   (sensitivity_lib.py:245-247).                */
size_t vt_gemv_workspace_bytes(int M, int64_t N);
int vt_gemv(const double* A, int64_t lda, int M, int64_t N, const double* x, double alpha, const double* y0,
            double beta, double* y, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Conjugate-gradient vector kernels, batched over K right-hand sides -------
 * Replaces scipy.sparse.linalg.cg behind get_cg_solver (solver_lib.py:91-97, legacy
 * stopping rule |r| < max(atol, rtol |b|)).  Vectors are rows of (K, D) arrays;
 * `state` is K x 8 device doubles {rho, rho_prev, p.q, |r|^2, |b|^2, tol, status,
 * matvecs}, status 1 = running, 0 = converged, 2 = stopped at maxiter.  One
 * iteration of all K columns is
 *   vt_cg_batch_update_p  ->  Q = mat_times_vec(P)  ->  vt_cg_batch_update_xr;
 * every column follows scipy's iteration on its own scalars and freezes (P row =
 * 0) once it has converged; the host reads `state` only to learn that all have.
 * update_p: Z (K x D, may be NULL) = preconditioned residuals M r computed by the
 * caller, else minv (D, may be NULL) = the diagonal of a Jacobi preconditioner.
 * keep_xr != 0 in init: X and R already hold x0 and b - A x0.                     */
int vt_cg_batch_init(int D, int K, const double* B, double* X, double* R, double* state, double rtol, double atol,
                     int keep_xr, void* stream);
int vt_cg_batch_update_p(int D, int K, const double* R, const double* Z, const double* minv, double* P, double* state,
                         int maxiter, void* stream);
int vt_cg_batch_update_xr(int D, int K, const double* P, const double* Q, double* X, double* R, double* state,
                          void* stream);

/* ---- Block-arrow Hessians (SparseBlockHessian) ------------------------------
 * H = [blockdiag(B_g) C; C^T Hgg], B_g (M x M, M <= 32), C_g (M x Dg): the
 * structure sparse_hessian_lib.py:69-168 assembles entry by entry and
 * solver_lib.py:46-48 hands to SuperLU.  Factorisation on the GPU:
 *   L_g = chol(B_g) (vt_block_potrf_batched), Z_g = L_g^{-1} C_g
 *   (vt_block_trsm_batched, in place), Schur = Hgg - Z^T Z (vt_syrk_weighted on
 *   the (G*M) x Dg matrix Z) and vt_potrf of the Schur complement; the solve
 *   uses vt_block_solve_batched (mode 0: L^{-1}, 1: L^{-T}), vt_tall_colsum
 *   (Z^T u) and vt_tall_gemv (Z x).  *info: 0 or 1 + index of a non-PD block.
 * vt_gmm_blocks assembles B_g, C_g, the responsibilities r (N x K), the local
 * gradient and the per-observation objective terms in closed form for the
 * Gaussian-mixture mean-field VB objective (benchmark config 3); any output
 * pointer may be NULL.                                                       */
int vt_block_potrf_batched(double* blocks, int64_t G, int M, int32_t* info, void* stream);
int vt_block_trsm_batched(const double* Lb, double* C, int64_t G, int M, int Dg, void* stream);
/* C_g <- L_g^{-T} C_g in place: the backward half of a multi-right-hand-side block solve (C: G x M x K). */
int vt_block_trsmt_batched(const double* Lb, double* C, int64_t G, int M, int Dg, void* stream);
int vt_block_solve_batched(const double* Lb, double* b, int64_t G, int M, int mode, void* stream);
int vt_tall_gemv(const double* Z, int64_t R, int Dg, const double* x, double alpha, double* y, double beta,
                 void* stream);
size_t vt_tall_colsum_workspace_bytes(int Dg);
int vt_tall_colsum(const double* Z, int64_t R, int Dg, const double* u, double alpha, const double* y0, double beta,
                   double* out, void* workspace, size_t workspace_bytes, void* stream);
int vt_gmm_blocks(const double* X, int64_t N, int d, int K, const double* m, const double* rho,
                  const double* log_pi, double* blocks, double* cross, double* rmat, double* grad_rho,
                  double* obj_terms, void* stream);

/* ---- Synthetic data (bench and tests) ---------------------------------------
 * Counter-based, reproducible for any row range (oracle twin:
 * oracle/models.py synth_design / synth_uniform).                            */
int vt_synth_design(double* X, int64_t ldx, int64_t row0, int64_t nrows, int ncols, uint64_t seed, double scale,
                    void* stream);
int vt_synth_uniform(double* u, int64_t row0, int64_t nrows, uint64_t seed, void* stream);
int vt_synth_bernoulli(double* y, const double* z, int64_t row0, int64_t nrows, uint64_t seed, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VITTLES_B200_H */
