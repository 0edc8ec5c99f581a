// Dense FP64 Cholesky factor / solve launchers (chol.cu).
#pragma once
#include "common.cuh"

namespace vt {

constexpr int CHOL_NB = 128;

// Number of doubles of the inverted-diagonal-block buffer for a D x D factor.
size_t chol_dinv_doubles(int D);

// In-place lower Cholesky of the row-major D x D matrix A (only the lower
// triangle is read and written).  *info (device int) is 0 on success or the
// 1-based column of the first non-positive pivot.  Asynchronous on `stream`.
int chol_potrf(double* A, long lda, int D, double* dinv, int* info, cudaStream_t stream);

// Solve (L L^T) X = B in place for the row-major D x K right-hand side B.
int chol_potrs(const double* L, long ldl, int D, const double* dinv, double* B, long ldb, int K, cudaStream_t stream);
// One pass of that solve, in place: B <- L^{-1} B (transpose = 0) or B <- L^{-T} B (transpose = 1).
int chol_trsm_lower(const double* L, long ldl, int D, const double* dinv, double* B, long ldb, int K, int transpose,
                    cudaStream_t stream);

}  // namespace vt
