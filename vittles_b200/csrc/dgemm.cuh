// FP64 tensor-core GEMM engine shared by every dense contraction on the
// sensitivity hot path (weighted SYRK for the Hessian, the H^{-1} G^T apply,
// Cholesky trailing updates, triangular-solve updates, J1 H^{-1} J2^T).
//
// Design (B200, sm_100a):
//   * FP64 tensor math on sm_100a is the warp-level DMMA.8x8x4 (tcgen05 has no
//     f64 kind).  Measured peak: 128 flop/clk/SM = 37.2 TFLOP/s for DMMA and
//     DFMA alike (profiles/fp64_peak_r01.jsonl); DMMA needs 1/16 of the issue
//     slots and 1/4 of the operand reads, which is what lets two warps per
//     SMSP saturate the pipe.
//   * CTA tile 128x128x16, 8 warps as 2(M) x 4(N), warp tile 64x32 -> 32 DMMA
//     per 12 LDS.64 per k4 step; 128 accumulator registers per thread.
//     A second configuration (64x64x16, 4 warps as 2 x 2, two CTAs per SM)
//     serves short-K / few-tile problems (Cholesky panels and trailing updates,
//     triangular-solve steps) and outputs that 128-wide tiles cover wastefully
//     (e.g. the 320 x 320 Schur complement of config 3).
//   * Operands staged by 16-byte cp.async into a 4-stage ring.  Two operand
//     layouts: KC (k contiguous in memory, smem [row][16+4]) and KS (k strided,
//     i.e. the row index contiguous, smem [k][128+4]).  Both paddings are
//     = 4 (mod 16) doubles, which makes the DMMA fragment reads (lane ->
//     row g = lane>>2, k t = lane&3) bank-conflict free per half warp.
//   * Persistent CTAs (one per SM) walk a flat stream of (tile, k-iteration)
//     units; the cp.async ring runs ahead ACROSS tile boundaries so the
//     epilogue of one tile overlaps the loads of the next.
//   * Optional split-K ("parts"): partial tiles go to a workspace and are
//     summed in a fixed order by splitk_reduce_kernel -> bitwise reproducible.
#pragma once
#include "common.cuh"

namespace vt {

enum OpMode : int { KC = 0, KS = 1 };

constexpr int BK = 16;
constexpr int LDKC = BK + 4;    // 20 doubles; the KS leading dimension is (tile + 4) doubles
constexpr int STAGES = 4;
constexpr int TILE_BIG = 128, TILE_SMALL = 64;   // CTA tile edge of the two kernel configurations

struct GemmParams {
  int M, N, K;
  const double* A; long lda; int amode;   // KC: A(m,k) = A[m*lda+k];  KS: A(m,k) = A[k*lda+m]
  const double* B; long ldb; int bmode;   // KC: B(n,k) = B[n*ldb+k];  KS: B(n,k) = B[k*ldb+n]
  double* C; long ldc;                    // C(m,n) = C[m*ldc+n]
  double alpha, beta;                     // C = alpha * rs[m] * cs[n] * sum_k ks[k] A(m,k) B(n,k) + beta * C
  const double* kscale;
  const double* colscale;
  const double* rowscale;
  int lower;       // only tiles with tile_m >= tile_n (square outputs)
  int mirror;      // lower only: also write C(n,m) = C(m,n) (symmetric result)
  int parts;       // split-K factor (>= 1); 0 = choose automatically
  int tile;        // CTA tile edge: TILE_BIG, TILE_SMALL, or 0 = choose automatically
  int spare_sms;   // leave this many SMs without a CTA of the persistent grid (room for a concurrent kernel)
  double* workspace; size_t workspace_bytes;
  // derived (filled by gemm_launch)
  int tiles_m, tiles_n, ntiles, kiters, a_vec, b_vec, c_vec;
};

// Fills the derived fields, picks `parts` if 0 and launches on `stream`.
int gemm_launch(GemmParams p, cudaStream_t stream);
// Workspace needed by gemm_launch for automatic split-K of this shape.
size_t gemm_workspace_bytes(int M, int N, int K, int lower, int tile);
// Tile edge chosen for a shape when GemmParams::tile == 0.
int gemm_pick_tile(int M, int N, int K, int lower);
int gemm_pick_parts(int ntiles, int kiters, int tile, size_t workspace_bytes);
int gemm_ctas_per_sm(int tile);

// out[n] = |Linv x_n|^2 for the rows of X (N x D): per chunk of rows U = X_c Linv^T on this engine, then the sum of
// squares of every row of U in a fixed order.
size_t quad_forms_workspace_bytes(long N, int D);
int quad_forms(const double* Linv, long ldl, const double* X, long ldx, long N, int D, double* out, void* workspace,
               size_t workspace_bytes, cudaStream_t stream);

// Leave-one-group-out predictors and h_n (grouploo.cuh) with U = X_c Linv^T per chunk of rows on this engine; the
// chunks overlap by GROUP_LOO_OVERLAP rows so that every group lies whole in one of them.
size_t group_loo_workspace_bytes(long N, int D);
int group_loo(const double* Linv, long ldl, const double* X, long ldx, long N, int D, const int64_t* starts, long G,
              const double* s, const double* u, const double* z, int method, double* zpred, double* h, void* workspace,
              size_t workspace_bytes, cudaStream_t stream);

}  // namespace vt
