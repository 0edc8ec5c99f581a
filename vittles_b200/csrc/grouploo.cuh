// Leave-one-group-out predictors from one chunk of U = Linv X^T (Linv = L^{-1}, H = L L^T).
//
// For a group g of m <= 32 consecutive rows R: Q = U_R^T U_R = X_R H^{-1} X_R^T (m x m), t = Q u_R and
//   h_n      = Q_nn                                   (x_n^T H^{-1} x_n)
//   IJ:  z_R + t                                      (X_R of theta_hat + H^{-1} sum_{n in R} u_n x_n)
//   NS:  z_R + t + Q S^1/2 M^{-1} S^1/2 t,  M = I - S^1/2 Q S^1/2,  S = diag(s_R)
// The Newton-step form is z_R + X_R H_{-R}^{-1} X_R^T u_R by Woodbury: one Newton step from theta_hat on the
// objective without the group.  A group whose M has a Cholesky pivot (squared) <= 2^-40 gets NaN on all its rows.
#pragma once
#include "common.cuh"

namespace vt {

constexpr int GROUP_LOO_MAXM = 32;            // rows per group
constexpr int GROUP_LOO_IJ = 0, GROUP_LOO_NS = 1;

// One launch over the chunk of rows [r0, r0 + rows) of U, element (row r, feature i) at U[(r - r0) sr + i sf]
// (the INT8 engine's D x rows store: sr = 1, sf = pitch; the DMMA engine's rows x D: sr = pitch, sf = 1).  Handles
// the groups whose start lies in [lo, hi): every row of those groups must lie in the chunk.  starts (G + 1 entries,
// strictly increasing from 0 to N, at most GROUP_LOO_MAXM apart), s, u, z, zpred and h are indexed by global row.
// Sums run in a fixed order (no atomics): two calls give the same bits.
struct GroupLooChunk {
  const double* U;
  long sr, sf, r0, rows;
  int D;
  const int64_t* starts;
  long G, lo, hi;
  const double *s, *u, *z;
  int method;
  double *zpred, *h;
};
int group_loo_chunk(const GroupLooChunk& c, cudaStream_t stream);

// Rows a chunk overlaps the next one by, so that no group of at most GROUP_LOO_MAXM rows is split: chunk c spans
// [c p, c p + ch) with stride p = ch - GROUP_LOO_OVERLAP and handles the groups that start in [c p, (c + 1) p) (the
// last chunk: every group from c p on).
constexpr long GROUP_LOO_OVERLAP = GROUP_LOO_MAXM;

}  // namespace vt
