// Batched small-block kernels for block-arrow Hessians
//
//     H = [ blockdiag(B_1..B_G)   C ]     B_g (M x M) SPD,  C_g (M x Dg),  Hgg (Dg x Dg)
//         [ C^T                 Hgg ]
//
// produced by SparseBlockHessian (reference: sparse_hessian_lib.py:69-168) and
// solved upstream by SuperLU (solver_lib.py:46-48).  Here:
//   block_potrf : L_g = chol(B_g)                  one warp per block, rows in registers
//   block_trsm  : Z_g = L_g^{-1} C_g  (in place)   thread = (block, column), L_g in shared memory
//   block_solve : y_g = L_g^{-1} b_g / L_g^{-T} b_g
//   tall_gemv   : y = beta*y + alpha * Z x         Z (R x Dg), R ~ G*M huge, Dg short
//   tall_colsum : out = Z^T u                      deterministic two-stage reduction
// The Schur complement Hgg - Z^T Z is a SYRK over the (G*M) x Dg matrix Z and
// runs on the FP64 tensor-core engine (vt_syrk_weighted); the dense global solve
// is vt_potrf / vt_potrs.  All of these are HBM bound (M ~ 20): the design goal
// is one coalesced read and one coalesced write of every block.
//
// gmm_blocks assembles B_g, C_g and diag(Hgg) in closed form for the
// Gaussian-mixture mean-field VB objective of benchmark config 3.
#include "blockchol.cuh"

namespace vt {

namespace {

constexpr int MAXM = BLOCK_MAXM;   // 32

// ---------------------------------------------------------------- potrf ----
// 4 warps per CTA, one block per warp at a time.  The block is staged through
// shared memory (coalesced global traffic); lane i then owns row i in registers,
// the pivot column is broadcast with shuffles, and every pivot costs one rsqrt
// and no division (the serial chain of a 19 x 19 block is ~19 x 150 clocks).
template <int MT>
__global__ void __launch_bounds__(128) block_potrf_kernel(double* blocks, long G, int M, int* info) {
  __shared__ double sm[4][MT * (MT + 1)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* a = sm[warp];
  const int ld = M + 1;
  for (long g = (long)blockIdx.x * 4 + warp; g < G; g += (long)gridDim.x * 4) {
    double* B = blocks + g * M * M;
    for (int e = lane; e < M * M; e += 32) a[(e / M) * ld + (e % M)] = B[e];
    __syncwarp();
    double r[MT];
#pragma unroll
    for (int k = 0; k < MT; ++k) r[k] = (lane < M && k <= lane) ? a[lane * ld + k] : 0.0;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < MT; ++j) {
      if (j < M) {
        double d = __shfl_sync(0xffffffffu, r[j], j);
        if (!(d > 0.0)) { bad = true; d = 1.0; }
        const double rs = rsqrt(d);
        const double l = (lane > j) ? r[j] * rs : (lane == j ? d * rs : 0.0);
        r[j] = l;
#pragma unroll
        for (int k = j + 1; k < MT; ++k) {
          const double lk = __shfl_sync(0xffffffffu, l, k);
          r[k] = fma(-l, lk, r[k]);
        }
      }
    }
    if (bad && lane == 0) atomicCAS(info, 0, (int)(g < 2147483647L ? g + 1 : 2147483647L));
    __syncwarp();
#pragma unroll
    for (int k = 0; k < MT; ++k)
      if (lane < M && k < M) a[lane * ld + k] = (k <= lane) ? r[k] : 0.0;
    __syncwarp();
    for (int e = lane; e < M * M; e += 32) B[e] = a[(e / M) * ld + (e % M)];
    __syncwarp();
  }
}

// ----------------------------------------------------------------- trsm ----
// Z = L^{-1} C in place.  A CTA takes TRSM_BPC consecutive blocks at a time;
// work items are (block, column) pairs flattened over the threads, so that the
// global accesses of a warp are contiguous along the column index and every
// thread has all M loads of its column in flight before the substitution
// starts (HBM bound: 16 M Dg bytes per block).
constexpr int TRSM_BPC = 4;
constexpr int TRSM_MINB = 3;           // resident CTAs per SM for blocks of up to 24 rows
template <int MT, bool TR>
__global__ void __launch_bounds__(256, MT <= 24 ? TRSM_MINB : 1) block_trsm_kernel(const double* __restrict__ Lb, double* __restrict__ C, long G,
                                                         int M, int Dg) {
  __shared__ double sl[TRSM_BPC][MT * MT];
  __shared__ double sinv[TRSM_BPC][MT];
  const int MM = M * M;
  for (long g0 = (long)blockIdx.x * TRSM_BPC; g0 < G; g0 += (long)gridDim.x * TRSM_BPC) {
    const int nb = (int)(G - g0 < TRSM_BPC ? G - g0 : TRSM_BPC);
    __syncthreads();
    for (int e = threadIdx.x; e < nb * MM; e += blockDim.x) sl[e / MM][e % MM] = Lb[g0 * MM + e];
    __syncthreads();
    if (threadIdx.x < nb * M) {
      const int b = threadIdx.x / M, i = threadIdx.x % M;
      sinv[b][i] = 1.0 / sl[b][i * M + i];
    }
    __syncthreads();
    for (int item = threadIdx.x; item < nb * Dg; item += blockDim.x) {
      const int b = item / Dg, c = item - b * Dg;
      double* Cg = C + (g0 + b) * (long)M * Dg + c;
      const double* L = sl[b];
      double z[MT];
#pragma unroll
      for (int i = 0; i < MT; ++i)
        if (i < M) z[i] = Cg[(long)i * Dg];
      if constexpr (!TR) {
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          if (i < M) {
            double s = z[i];
#pragma unroll
            for (int k = 0; k < i; ++k) s = fma(-L[i * M + k], z[k], s);
            z[i] = s * sinv[b][i];
          }
        }
      } else {                                   // L^T z' = z: backward substitution down the columns of L
#pragma unroll
        for (int i = MT - 1; i >= 0; --i) {
          if (i < M) {
            double s = z[i];
#pragma unroll
            for (int k = i + 1; k < MT; ++k)
              if (k < M) s = fma(-L[k * M + i], z[k], s);
            z[i] = s * sinv[b][i];
          }
        }
      }
#pragma unroll
      for (int i = 0; i < MT; ++i)
        if (i < M) Cg[(long)i * Dg] = z[i];
    }
  }
}

// ---------------------------------------------------------- vector solves ----
// mode 0: b <- L^{-1} b ; mode 1: b <- L^{-T} b ; one warp per block (lane = row).
__global__ void __launch_bounds__(128) block_solve_kernel(const double* __restrict__ Lb, double* b, long G, int M,
                                                          int mode) {
  __shared__ double sm[4][MAXM * (MAXM + 1)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* a = sm[warp];
  const int ld = M + 1;
  for (long g = (long)blockIdx.x * 4 + warp; g < G; g += (long)gridDim.x * 4) {
    for (int e = lane; e < M * M; e += 32) a[(e / M) * ld + (e % M)] = Lb[g * M * M + e];
    double x = lane < M ? b[g * M + lane] : 0.0;
    __syncwarp();
    if (mode == 0) {
      for (int j = 0; j < M; ++j) {
        const double xj = __shfl_sync(0xffffffffu, x, j) / a[j * ld + j];
        if (lane == j) x = xj;
        if (lane > j && lane < M) x = fma(-a[lane * ld + j], xj, x);
      }
    } else {
      for (int j = M - 1; j >= 0; --j) {
        const double xj = __shfl_sync(0xffffffffu, x, j) / a[j * ld + j];
        if (lane == j) x = xj;
        if (lane < j) x = fma(-a[j * ld + lane], xj, x);
      }
    }
    if (lane < M) b[g * M + lane] = x;
    __syncwarp();
  }
}

// ------------------------------------------------------------- tall gemv ----
// y[r] = beta * y[r] + alpha * sum_c Z[r][c] x[c]; 8 lanes per row.
__global__ void __launch_bounds__(256) tall_gemv_kernel(const double* __restrict__ Z, long R, int Dg,
                                                        const double* __restrict__ x, double alpha, double* y,
                                                        double beta) {
  extern __shared__ double sx[];
  for (int c = threadIdx.x; c < Dg; c += blockDim.x) sx[c] = x[c];
  __syncthreads();
  const int sub = threadIdx.x & 7;
  for (long r = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 3; r < R; r += ((long)gridDim.x * blockDim.x) >> 3) {
    const double* zr = Z + r * Dg;
    double s = 0.0;
    for (int c = sub; c < Dg; c += 8) s = fma(zr[c], sx[c], s);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (sub == 0) y[r] = (beta == 0.0 ? 0.0 : beta * y[r]) + alpha * s;
  }
}

// ------------------------------------------------------------ tall colsum ----
// partial[cta][c] = sum over the CTA's rows of u[r] * Z[r][c]
constexpr int COLSUM_ROWS = 64;
// The block is as wide as the matrix (up to 1024 columns per sweep: a 256-thread block left 3/4 of its threads idle
// on the last 64 of 320 columns), and eight loads per thread are in flight (four accumulators, fixed order).
__global__ void __launch_bounds__(1024) tall_colsum_kernel(const double* __restrict__ Z, long R, int Dg,
                                                           const double* __restrict__ u, double* partial) {
  for (int c0 = 0; c0 < Dg; c0 += blockDim.x) {
    const int c = c0 + threadIdx.x;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    for (long rb = (long)blockIdx.x * COLSUM_ROWS; rb < R; rb += (long)gridDim.x * COLSUM_ROWS) {
      const long rend = rb + COLSUM_ROWS < R ? rb + COLSUM_ROWS : R;
      if (c < Dg) {
        long r = rb;
        for (; r + 8 <= rend; r += 8) {
          double z[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) z[k] = Z[(r + k) * Dg + c];
          a0 = fma(u[r], z[0], a0); a1 = fma(u[r + 1], z[1], a1); a2 = fma(u[r + 2], z[2], a2); a3 = fma(u[r + 3], z[3], a3);
          a0 = fma(u[r + 4], z[4], a0); a1 = fma(u[r + 5], z[5], a1); a2 = fma(u[r + 6], z[6], a2); a3 = fma(u[r + 7], z[7], a3);
        }
        for (; r < rend; ++r) a0 = fma(u[r], Z[r * Dg + c], a0);
      }
    }
    if (c < Dg) partial[(long)blockIdx.x * Dg + c] = (a0 + a1) + (a2 + a3);
  }
}

__global__ void colsum_finish_kernel(const double* partial, int ncta, int Dg, double alpha, const double* y0,
                                     double beta, double* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Dg) return;
  double s = 0.0;
  for (int k = 0; k < ncta; ++k) s += partial[(long)k * Dg + c];
  out[c] = alpha * s + (y0 ? beta * y0[c] : 0.0);
}

// -------------------------------------------------------------- GMM-VB ----
// One CTA per observation.  x = (m (K x d), rho_n (K-1 free logits)), logits l = [rho_n, 0]:
//   r = softmax(l),  c_k = 0.5 |x_n - m_k|^2 - log pi_k,  a_k = c_k + log r_k,  abar = sum r_k a_k
//   q_k = 1 - r_k,  delta_k = a_k - abar
//   B[j][l] = r_j d_jl (delta_j + 1) - r_j r_l (delta_j + delta_l + 1)                   j,l < K-1
//   C[j][k*d + t] = r_j (d_jk - r_k) (m_k[t] - x_n[t])                                   j < K-1, k < K
//   rsum[k] += r_k  (diagonal of the global block; reduced by the caller)
//   grad_rho[j] = r_j delta_j,  obj = abar
// A fitted mixture with separated clusters has logit gaps of tens to hundreds, so r_dom ~ 1 for the dominant
// component dom (the lowest lane holding the largest logit), and B_dom,dom, r_dom (1 - r_dom) and delta_dom are
// (1 - r_dom)-small.  Formed as written they are differences of O(1) numbers (1 - r rounds to 0 past a gap of ~37)
// and B comes out indefinite.  They are formed instead from sums over the other components, which do not cancel:
//   q_dom = r_dom sum_{i != dom} e_i  (e_k = e^(l_k - l_dom), r_dom = 1 / tot),  q_k = 1 - r_k for k != dom
//   (r_k <= 1/2 there),  delta_j = (a_j - a_dom) - sum_{i != dom} r_i (a_i - a_dom),
//   a_i - a_dom = (c_i - c_dom) + (l_i - l_dom),
//   B_jj = r_j q_j + r_j delta_j (q_j - r_j),  B_jl = -r_j r_l (delta_j + delta_l + 1),  C coefficient r_j q_j at j = k
// 8 CTAs per SM (the grid cap of gmm_blocks) need <= 32 registers a thread.
__global__ void __launch_bounds__(256, 8) gmm_blocks_kernel(const double* __restrict__ X, long N, int d, int K,
                                                         const double* __restrict__ m, const double* __restrict__ rho,
                                                         const double* __restrict__ log_pi, double* blocks,
                                                         double* cross, double* rmat, double* grad_rho,
                                                         double* obj_terms) {
  extern __shared__ double sm[];
  double* sr = sm;            // K: r
  double* sq = sm + K;        // K: q = 1 - r
  double* sa = sm + 2 * K;    // K: c, then delta
  double* sx = sm + 3 * K;    // d
  const int M = K - 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long n = blockIdx.x; n < N; n += gridDim.x) {
    __syncthreads();
    for (int t = threadIdx.x; t < d; t += blockDim.x) sx[t] = X[n * d + t];
    __syncthreads();
    // squared distances: warp w handles components w, w+8, ...
    for (int k = warp; k < K; k += 8) {
      double s = 0.0;
      for (int t = lane; t < d; t += 32) { const double df = sx[t] - m[(long)k * d + t]; s = fma(df, df, s); }
      s = warp_sum(s);
      if (lane == 0) sa[k] = 0.5 * s - log_pi[k];
    }
    __syncthreads();
    if (warp == 0) {
      // softmax over [rho, 0], q and delta, by one warp (K <= 32)
      double z = lane < M ? rho[n * M + lane] : (lane == M ? 0.0 : -1e300);
      double mx = z;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      z -= mx;                                                          // l - l_dom
      const double e = lane < K ? exp(z) : 0.0;
      const int dom = __ffs(__ballot_sync(0xffffffffu, z == 0.0)) - 1;
      const double tot = warp_sum(e);
      const double rest = warp_sum(lane == dom ? 0.0 : e);
      if (lane < K) { const double r = e / tot; sr[lane] = r; sq[lane] = lane == dom ? rest * r : 1.0 - r; }
      const double logr = z - log(tot);
      __syncwarp();
      const double r = lane < K ? sr[lane] : 0.0;
      if (lane < K && rmat) rmat[n * K + lane] = r;
      const double c = lane < K ? sa[lane] : 0.0;
      const double abar = warp_sum(r * (c + logr));
      const double da = (c - __shfl_sync(0xffffffffu, c, dom)) + z;     // a - a_dom
      const double dev = da - warp_sum(lane != dom ? r * da : 0.0);
      if (lane < K) sa[lane] = dev;
      if (lane < M && grad_rho) grad_rho[n * M + lane] = r * dev;
      if (lane == 0 && obj_terms) obj_terms[n] = abar;
    }
    __syncthreads();
    if (blocks) {
      for (int e = threadIdx.x; e < M * M; e += blockDim.x) {
        const int j = e / M, l = e % M;
        const double v = j == l ? sr[j] * sq[j] + sr[j] * sa[j] * (sq[j] - sr[j])
                                : -sr[j] * sr[l] * (sa[j] + sa[l] + 1.0);
        blocks[n * (long)M * M + e] = v;
      }
    }
    if (cross) {
      // thread = global column c = (k, t); one coalesced row of C_n per j
      const int Dg = K * d;
      double* Cn = cross + n * (long)M * Dg;
      for (int c = threadIdx.x; c < Dg; c += blockDim.x) {
        const int k = c / d, t = c - k * d;
        const double dm = m[(long)k * d + t] - sx[t];
        const double diag = sr[k] * sq[k] * dm, off = -sr[k] * dm;      // r_k q_k dm at j = k, -r_j r_k dm elsewhere
        double* p = Cn + c;
        for (int j = 0; j < M; ++j, p += Dg) *p = j == k ? diag : sr[j] * off;
      }
    }
  }
}

int grid_for(long work, int per_cta, int max_ctas_per_sm) {
  long g = (work + per_cta - 1) / per_cta;
  const long cap = (long)num_sms() * max_ctas_per_sm;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

}  // namespace

int block_potrf(double* blocks, long G, int M, int* info, cudaStream_t stream) {
  VT_REQUIRE(blocks && info && G >= 1 && M >= 1 && M <= MAXM, "block_potrf: need 1 <= M <= %d", MAXM);
  VT_CUDA(cudaMemsetAsync(info, 0, sizeof(int), stream));
  const int grid = grid_for(G, 4, 4);
  if (M <= 8) block_potrf_kernel<8><<<grid, 128, 0, stream>>>(blocks, G, M, info);
  else if (M <= 16) block_potrf_kernel<16><<<grid, 128, 0, stream>>>(blocks, G, M, info);
  else if (M <= 24) block_potrf_kernel<24><<<grid, 128, 0, stream>>>(blocks, G, M, info);
  else block_potrf_kernel<32><<<grid, 128, 0, stream>>>(blocks, G, M, info);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

int block_trsm(const double* Lb, double* C, long G, int M, int Dg, int transpose, cudaStream_t stream) {
  VT_REQUIRE(Lb && C && G >= 1 && M >= 1 && M <= MAXM && Dg >= 1, "block_trsm: bad arguments");
  const int grid = grid_for(G, TRSM_BPC, 3);
#define VT_TRSM(MT)                                                                      \
  do {                                                                                   \
    if (transpose) block_trsm_kernel<MT, true><<<grid, 256, 0, stream>>>(Lb, C, G, M, Dg);  \
    else block_trsm_kernel<MT, false><<<grid, 256, 0, stream>>>(Lb, C, G, M, Dg);           \
  } while (0)
  if (M <= 8) VT_TRSM(8);
  else if (M <= 16) VT_TRSM(16);
  else if (M <= 20) VT_TRSM(20);
  else if (M <= 24) VT_TRSM(24);
  else VT_TRSM(32);
#undef VT_TRSM
  VT_LAUNCH_CHECK();
  return VT_OK;
}

int block_solve(const double* Lb, double* b, long G, int M, int mode, cudaStream_t stream) {
  VT_REQUIRE(Lb && b && G >= 1 && M >= 1 && M <= MAXM && (mode == 0 || mode == 1), "block_solve: bad arguments");
  block_solve_kernel<<<grid_for(G, 4, 6), 128, 0, stream>>>(Lb, b, G, M, mode);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

int tall_gemv(const double* Z, long R, int Dg, const double* x, double alpha, double* y, double beta,
              cudaStream_t stream) {
  VT_REQUIRE(Z && x && y && R >= 1 && Dg >= 1 && Dg <= 6000, "tall_gemv: bad arguments");
  tall_gemv_kernel<<<grid_for(R, 32, 8), 256, Dg * 8, stream>>>(Z, R, Dg, x, alpha, y, beta);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

size_t tall_colsum_workspace_bytes(int Dg) { return (size_t)num_sms() * 8 * Dg * 8; }

int tall_colsum(const double* Z, long R, int Dg, const double* u, double alpha, const double* y0, double beta,
                double* out, double* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Z && u && out && R >= 1 && Dg >= 1, "tall_colsum: bad arguments");
  const int threads = Dg >= 1024 ? 1024 : (Dg + 31) / 32 * 32;
  const int grid = grid_for(R, COLSUM_ROWS, threads > 512 ? 2 : (threads > 256 ? 4 : 8));
  VT_REQUIRE(workspace && workspace_bytes >= (size_t)grid * Dg * 8, "tall_colsum: workspace too small");
  tall_colsum_kernel<<<grid, threads, 0, stream>>>(Z, R, Dg, u, workspace);
  VT_LAUNCH_CHECK();
  colsum_finish_kernel<<<(Dg + 255) / 256, 256, 0, stream>>>(workspace, grid, Dg, alpha, y0, beta, out);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

int gmm_blocks(const double* X, long N, int d, int K, const double* m, const double* rho, const double* log_pi,
               double* blocks, double* cross, double* rmat, double* grad_rho, double* obj_terms,
               cudaStream_t stream) {
  VT_REQUIRE(X && m && rho && log_pi && N >= 1 && d >= 1 && K >= 2 && K <= 32, "gmm_blocks: need 2 <= K <= 32");
  const size_t smem = (size_t)(3 * K + d) * 8;
  gmm_blocks_kernel<<<grid_for(N, 1, 8), 256, smem, stream>>>(X, N, d, K, m, rho, log_pi, blocks, cross, rmat,
                                                               grad_rho, obj_terms);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

}  // namespace vt
