// Host-side launchers of the GLM-family kernels (glm.cu).
#pragma once
#include "common.cuh"

namespace vt {

enum GlmFamily : int { GLM_LOGISTIC = 0, GLM_POISSON = 1, GLM_GAUSSIAN = 2 };
constexpr int GLM_MAX_BDERIV = 8;   // highest derivative order of b(z) supported

size_t glm_workspace_bytes(int D);

// z = X theta; resid = b'(z) - y; s = w b''(z); grad = X^T (w resid) + l2 theta.
// Any of z/resid/s/grad may be null.  colmax != null (D <= 2048, workspace 2 x glm_workspace_bytes): the same pass
// also writes sq[n] = sqrt(s_n) and colmax[c] = bit pattern of max_n sq_n |x_nc| - the inputs of syrk_ozaki.
int glm_stats(const double* X, long ldx, long N, int D, const double* theta, const double* y, const double* w,
              int family, double* z, double* resid, double* s, double* grad, double l2, double* sq,
              unsigned long long* colmax, double* workspace, size_t workspace_bytes, cudaStream_t stream);

// out = X^T (s .* (X v)) + ridge * v
int glm_hvp(const double* X, long ldx, long N, int D, const double* s, const double* v, double ridge, double* out,
            double* workspace, size_t workspace_bytes, cudaStream_t stream);

// out (q x D) = V X^T diag(s) X + ridge V for q <= 4 directions (rows of V) in ONE pass over X
size_t glm_hvp_multi_workspace_bytes(int D, int q);
int glm_hvp_multi(const double* X, long ldx, long N, int D, const double* s, const double* V, int q, double ridge,
                  double* out, double* workspace, size_t workspace_bytes, cudaStream_t stream);

// out = X^T ( w .* b^{(q+1)}(z) .* prod_j (X dirs_j) ),  dirs is (q, D) row-major
size_t glm_dirderiv_workspace_bytes(long N, int D);
int glm_dirderiv(const double* X, long ldx, long N, int D, const double* z, const double* w, int family,
                 const double* dirs, int q, double* out, double* workspace, size_t workspace_bytes,
                 cudaStream_t stream);

// out[j * ldo + n] = alpha * c[n] * (x_n . V[j, :]) for j < q, n < N (V (q, D) row-major): one pass over X that
// writes q values per row and no column sums.  q <= glm_influence_max_directions(D) (0 for D > 8192).
constexpr int GLM_INFLUENCE_MAXQ = 8;
int glm_influence_max_directions(int D);
int glm_influence(const double* X, long ldx, long N, int D, const double* c, const double* V, int q, double alpha,
                  double* out, long ldo, cudaStream_t stream);

size_t gemv_workspace_bytes(int M, long N);
// y = alpha * A x + beta * y0, A (M x N) row-major with leading dimension lda
int gemv_rows(const double* A, long lda, int M, long N, const double* x, double alpha, const double* y0, double beta,
              double* y, double* workspace, size_t workspace_bytes, cudaStream_t stream);

// K conjugate-gradient iterations side by side (rows of (K, D) arrays; state is K x 8 doubles), see glm.cu
int cg_batch_init(int D, int K, const double* B, double* X, double* R, double* state, double rtol, double atol,
                  int keep_xr, cudaStream_t stream);
int cg_batch_update_p(int D, int K, const double* R, const double* Z, const double* minv, double* P, double* state,
                      int maxiter, cudaStream_t stream);
int cg_batch_update_xr(int D, int K, const double* P, const double* Q, double* X, double* R, double* state,
                       cudaStream_t stream);

}  // namespace vt
