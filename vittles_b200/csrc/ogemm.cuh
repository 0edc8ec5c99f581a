// FP64-grade GEMM on the INT8 tensor cores (tcgen05.mma.kind::i8) by error-free
// slicing - the "Ozaki scheme" - with balanced base-256 digits:
//
//   x_rk = sigma_r 2^-6 sum_{s=0..S-1} d_s[r][k] 2^{-8s} + O(sigma_r 2^{-(8S-1)}),   d_s in [-128, 127] (int8),
//   sigma_r = 2^e_r > max_k |x_rk| >= sigma_r / 2
//
// Every digit product and every K-sum is exact in INT32, so
//
//   sum_k a_mk b_nk = sigma_m tau_n 2^-12 sum_{s+t < S} 2^{-8(s+t)} (A_s B_t^T)_mn  +  O(S K 2^{-8S+2} sigma_m tau_n)
//
// needs S(S+1)/2 INT8 GEMMs whose results are combined in INT64 and FP64 in the
// epilogue.  S = 7 (54 bits per operand; 28 products) reproduces FP64 DMMA results to
// ~1e-14 of max|C| at several times the throughput bound of the FP64 pipe (INT8 dense
// peak 4.5 POP/s nominal vs 37 TFLOP/s); S = 6 (46 bits, 21 products) ~1e-12.
// Products whose digits sum to the same power of two share one TMEM accumulator
// (S accumulators of 64 columns), and because the B slices of a tile are contiguous in
// shared memory one tcgen05.mma with N = 64 (S - s) evaluates all products of A slice s.
#pragma once
#include "common.cuh"

namespace vt {

constexpr int OZAKI_MIN_SLICES = 5;
constexpr int OZAKI_MAX_SLICES = 7;
constexpr int OZAKI_MAX_K = 16384;      // (K + 128) * 128^2 * S < 2^31

// digits of every row of X (rows x cols, FP64): out[s][r][k] (int8, row pitch ldo bytes, a multiple of 16; pad bytes
// are zero), scale_out[r] = sigma_r (* fold[r] if fold != nullptr).
int ozaki_slice(const double* X, long ldx, long rows, int cols, int8_t* out, long ldo, long slice_stride, int nslices,
                double* scale_out, const double* fold, cudaStream_t stream);
// out[s][feature][observation] of sq_n x_ni with one scale per feature from colmax (bit patterns of the maxima).
int ozaki_slice_t(const double* X, long ldx, long rows, int cols, const double* sq, const unsigned long long* colmax,
                  int8_t* out, long ldo, long slice_stride, int nslices, double* scale_out, cudaStream_t stream);

// C (M x N, FP64) = alpha * rowscale[m] * colscale[n] * 2^-12 sum_{s+t<S} 2^{-8(s+t)} (A_s B_t^T)(m,n)
int ogemm_launch(int M, int N, int K, const int8_t* A, long lda, long a_slice_stride, const int8_t* B, long ldb,
                 long b_slice_stride, int nslices, double alpha, const double* rowscale, const double* colscale, double* C,
                 long ldc, cudaStream_t stream);

unsigned long long* ogemm_timing_buffer_public();   // development aid, see ogemm.cu

// Bare tcgen05.mma.kind::i8 loop (no loads) for about `seconds`: achieved dense INT8 TOP/s with instructions
// of N = n_tile, and SM clocks per 128 x n_tile x 32 instruction.  The denominator of the engine's roofline.
int i8_peak_probe(double seconds, int n_tile, double* tops, double* clocks_per_mma, cudaStream_t stream);

// S (D x N) = -Hinv diag(resid) X^T with FP64-grade accuracy on the INT8 tensor cores.
size_t ij_apply_ozaki_workspace_bytes(long N, int D, int nslices);
int ij_apply_ozaki(const double* Hinv, long ldh, const double* X, long ldx, long N, int D, const double* resid,
                   double* S, long lds, int nslices, void* workspace, size_t workspace_bytes, cudaStream_t stream);

// out[n] = |Linv x_n|^2 for every row x_n of X (N x D), Linv (D x D) lower triangular (zero above the diagonal:
// row block tm of Linv meets the k-blocks 0 .. tm only).  The chunks of ij_apply_ozaki; the epilogue squares each
// element of Linv X_c^T and sums the squares of every column over the rows of a warp, and a finish kernel adds
// the 4 ceil(D / 128) partials of a column in a fixed order.  Nothing of size D x N is written.
size_t quad_forms_ozaki_workspace_bytes(long N, int D, int nslices);
int quad_forms_ozaki(const double* Linv, long ldl, const double* X, long ldx, long N, int D, double* out, int nslices,
                     void* workspace, size_t workspace_bytes, cudaStream_t stream);

// Leave-one-group-out predictors and h_n (grouploo.cuh): per chunk of ij_apply_ozaki rows U = Linv X_c^T (D x ch,
// stored by the GEMM) over the full K range, then the per-group Gram and solve.  The chunks overlap by
// GROUP_LOO_OVERLAP rows so that every group lies whole in one of them.
size_t group_loo_ozaki_workspace_bytes(long N, int D, int nslices);
int group_loo_ozaki(const double* Linv, long ldl, const double* X, long ldx, long N, int D, const int64_t* starts,
                    long G, const double* s, const double* u, const double* z, int method, double* zpred, double* h,
                    int nslices, void* workspace, size_t workspace_bytes, cudaStream_t stream);

// H (D x D) = X^T diag(s) X (s >= 0) with FP64-grade accuracy on the INT8 tensor cores: per chunk of
// observations the digits of sqrt(s_n) x_ni are written transposed with one power-of-two scale per
// feature, the lower tiles of the chunk's Gram matrix run as split-K parts of at most 16384
// observations (INT32 bound) and are accumulated in FP64.
size_t syrk_ozaki_workspace_bytes(long N, int D, int nslices);
// sq_in / colmax_in (both or neither): sqrt(s_n) and the bit patterns of max_n sqrt(s_n) |x_ni| when the statistics
// pass has produced them already (glm_stats with colmax) - the sweep over X that computes them is then skipped.
int syrk_ozaki(const double* X, long ldx, long N, int D, const double* s, double* H, long ldh, int nslices,
               const double* sq_in, const unsigned long long* colmax_in, void* workspace, size_t workspace_bytes,
               cudaStream_t stream);

}  // namespace vt
