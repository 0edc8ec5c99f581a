// Fused single-pass  out = X^T u,  u_n = f_n(x_n . v_0, ..., x_n . v_{Q-1})
// over a row-major design matrix X (N x D).  One read of X from HBM serves both
// the row dot products and the transposed accumulation, so the kernel is bound
// by HBM at 8*N*D bytes (SURVEY.md section 8d).  Instances:
//   * GLM statistics + gradient      (Q=1, v=theta; writes z, resid, s)
//   * Hessian-vector product         (Q=1; u = s_n * t)            -> CG solver
//   * Q Hessian-vector products      (Q=NOUT<=4; u_j = s_n * t_j)  -> multi-RHS CG: one read of X for Q columns
//   * Taylor directional derivatives (Q=m; u = c_n * prod_j t_j)   -> dirderiv
//   * per-row outputs only           (NOUT=0, Q<=8; out_jn = op.store(n, j, t_j)) -> observation influence
//
// Structure (B200): persistent CTAs, two per SM, 256 threads.  A block of
// R = 8/CPT rows (32 KB for D = 512*CPT) is staged in shared memory by ONE
// bulk-TMA copy (cp.async.bulk ... mbarrier::complete_tx; SASS UBLKCP) into a
// 3-deep ring, so up to 192 KB per SM are in flight with one issuing thread per
// CTA.  Thread t owns columns {2t, 2t+1} + 512*i: it pulls its 16 double2
// of the block into registers once, uses them for the partial dot products
// (warp-shuffle reduction, then an 8-way cross-warp sum) and again for the
// rank-R update of its private column accumulators.  Per-CTA column sums go to a
// workspace and are added in a fixed order by xtfx_reduce_kernel (bitwise
// reproducible, no atomics).
#pragma once
#include "common.cuh"

namespace vt {

constexpr int XT_THREADS = 256;
constexpr int XT_NBUF = 3;
constexpr int XT_MAXQ = 4;

struct XtfxParams {
  const double* X; long ldx; long N; int D;
  const double* V;        // Q x D directions, row-major, contiguous
  double* partial;        // [grid][NOUT][Dp] column sums per CTA (null: skip the transposed pass)
  double* partial_max;    // CMAX kernels: [grid][Dp] column maxima of q_n |x_nc| per CTA (q_n from op.stats2)
  int Dp;                 // D rounded up to even
  int bulk;               // 1: rows can be staged with cp.async.bulk
  int contiguous;         // 1: ldx == D, a block of rows is one contiguous copy
};

// ---- mbarrier / bulk-copy PTX -------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

inline size_t xtfx_smem_bytes(int Dp, int R, int Q) {
  return (size_t)XT_NBUF * R * Dp * 8 + (size_t)(8 * R * Q + R * Q + R) * 8 + XT_NBUF * 8 + 128;
}

// R rows per block, CPT double2 columns per thread: R*CPT = 8 gives 32 KB blocks at
// D = 512*CPT, a 96 KB ring and two CTAs per SM, so that the block-wide syncs and
// the serial row-functor step of one CTA overlap the other's arithmetic (one
// CTA per SM left stats at 62% and the HVP at 79% of HBM peak, profiles/r01).
// NOUT = 1: one output vector, u_n = op(n, t, aux).  NOUT = Q > 1: Q output vectors, op.multi(n, t, aux, u) fills
// u_j - the accumulators of all Q outputs live in registers, so the CTA count per SM drops to one.
// CMAX: additionally keep max_n q_n |x_nc| per column, q_n the second value of op.stats2 (the column scales of the
// INT8 slicing engine's Hessian assembly come out of the statistics pass instead of a sweep of their own).  Only
// the binade of the maximum matters (the scale is the next power of two), so the maximum is taken over the HIGH
// words of the products as unsigned integers - sign 0, exponent, top 20 bits of the significand: one integer
// instruction per element, the exponent of the result is exact, and Inf / NaN (exponent all ones) are above every
// finite value, so a non-finite product poisons its column as the engine's own sweep does.
__device__ __forceinline__ uint32_t xt_himax(uint32_t m, double v) {
  const uint32_t h = (uint32_t)__double2hiint(v);
  return h > m ? h : m;
}
// NOUT = 0: no transposed pass at all - the row functor stores the Q dot products of each row (op.store(n, j, t_j)).
// The directions then take the registers the accumulators would, so two CTAs fit an SM only while Q * CPT <= 8.
template <int Q, int CPT, int R, int NOUT>
constexpr int xt_ctas_per_sm() {
  return (R * CPT <= 8 && (NOUT == 1 || (NOUT == 0 && Q * CPT <= 8))) ? 2 : 1;
}

// Sum over the warp of each of the Q values s[0..Q-1] by a transpose-reduce: every step halves the values a lane
// holds, the lanes of the pair exchanging the halves they drop (Q/2 + Q/4 + ... shuffles, then a plain butterfly over
// the remaining lanes), instead of Q separate 5-step reductions.  Afterwards lane l holds the sum of value
// j = l / (32 / QP) (QP = Q rounded up to a power of two).  Each lane adds its values in a fixed order, so the result
// is bitwise reproducible.
__host__ __device__ constexpr int xt_pow2_ceil(int q) { return q <= 1 ? 1 : 2 * xt_pow2_ceil((q + 1) / 2); }

template <int Q>
__device__ __forceinline__ double xt_transpose_reduce(double (&s)[Q], int lane) {
  static_assert(Q >= 1 && Q <= 32, "one value per lane at most");
  constexpr int QP = xt_pow2_ceil(Q);
  double v[QP];
#pragma unroll
  for (int j = 0; j < QP; ++j) v[j] = j < Q ? s[j] : 0.0;
#pragma unroll
  for (int m = QP, o = 16; o >= 1; o >>= 1) {
    if (m > 1) {
      const bool upper = (lane & o) != 0;        // this lane keeps the upper half of its values
#pragma unroll
      for (int j = 0; j < m / 2; ++j) {
        const double keep = upper ? v[j + m / 2] : v[j];
        const double send = upper ? v[j] : v[j + m / 2];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
      }
      m /= 2;
    } else {
      v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
    }
  }
  return v[0];
}

template <class RowOp, int Q, int CPT, int R, int NOUT = 1, bool CMAX = false>
__global__ void __launch_bounds__(XT_THREADS, (xt_ctas_per_sm<Q, CPT, R, NOUT>())) xtfx_kernel(const XtfxParams p, const RowOp op) {
  extern __shared__ __align__(128) unsigned char xt_raw[];
  const int Dp = p.Dp;
  double* bufs = reinterpret_cast<double*>(xt_raw);
  double* s_part = bufs + (size_t)XT_NBUF * R * Dp;   // [8][R][Q]
  double* s_u = s_part + 8 * R * Q;                    // [R][NOUT]
  double* s_q = s_u + R * Q;                           // [R] (CMAX)
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_q + R);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long nblocks = (p.N + R - 1) / R;
  const long my_first = blockIdx.x;
  const long stride = gridDim.x;

  if (tid == 0) {
#pragma unroll
    for (int b = 0; b < XT_NBUF; ++b) mbar_init(&bars[b], 1);
    fence_barrier_init();
  }
  __syncthreads();

  auto issue = [&](long blk, int buf) {   // thread 0 only
    const long row0 = blk * R;
    const int rows = (int)min((long)R, p.N - row0);
    double* dst = bufs + (size_t)buf * R * Dp;
    const uint32_t row_bytes = (uint32_t)p.D * 8u;
    mbar_expect_tx(&bars[buf], row_bytes * rows);
    if (p.contiguous) {
      bulk_g2s(dst, p.X + row0 * p.ldx, row_bytes * rows, &bars[buf]);
    } else {
      for (int r = 0; r < rows; ++r) bulk_g2s(dst + (size_t)r * Dp, p.X + (row0 + r) * p.ldx, row_bytes, &bars[buf]);
    }
  };

  // direction vectors for this thread's columns, kept in registers
  double2 v[Q][CPT];
#pragma unroll
  for (int j = 0; j < Q; ++j)
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
      const int c = 2 * tid + 512 * i;
      v[j][i].x = (c < p.D) ? p.V[(long)j * p.D + c] : 0.0;
      v[j][i].y = (c + 1 < p.D) ? p.V[(long)j * p.D + c + 1] : 0.0;
    }
  constexpr int NACC = NOUT > 0 ? NOUT : 1;
  double2 acc[NACC][CPT];
#pragma unroll
  for (int o = 0; o < NACC; ++o)
#pragma unroll
    for (int i = 0; i < CPT; ++i) acc[o][i] = make_double2(0.0, 0.0);
  uint32_t cmx[CMAX ? 2 * CPT : 1];
#pragma unroll
  for (int i = 0; i < (CMAX ? 2 * CPT : 1); ++i) cmx[i] = 0u;

  if (p.bulk && tid == 0) {
    for (int s = 0; s < XT_NBUF; ++s) {
      const long blk = my_first + s * stride;
      if (blk < nblocks) issue(blk, s);
    }
  }

  long it = 0;
  for (long blk = my_first; blk < nblocks; blk += stride, ++it) {
    const int buf = (int)(it % XT_NBUF);
    const long row0 = blk * R;
    const int rows = (int)min((long)R, p.N - row0);
    double* xs = bufs + (size_t)buf * R * Dp;
    if (p.bulk) {
      mbar_wait(&bars[buf], (uint32_t)((it / XT_NBUF) & 1));
    } else {
      // generic staging (odd D or unaligned rows): coalesced loads, zero padding
      for (int e = tid; e < R * Dp; e += XT_THREADS) {
        const int r = e / Dp, c = e - r * Dp;
        xs[e] = (r < rows && c < p.D) ? p.X[(row0 + r) * p.ldx + c] : 0.0;
      }
      __syncthreads();
    }
    // per-row operands of the row functor (y, w, z, s ...): issue the global loads
    // now so that their latency overlaps the dot products instead of sitting in
    // the serial functor step
    // (NOUT = 0: thread tid stores output tid / R of row tid % R)
    constexpr int NAUX = NOUT == 0 ? R * Q : R;
    typename RowOp::Aux aux;
    if (tid < NAUX && tid % R < rows) aux = op.load(row0 + tid % R);
    double2 x[R][CPT];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int i = 0; i < CPT; ++i) {
        const int c = 2 * tid + 512 * i;
        x[r][i] = (r < rows && c < Dp) ? *reinterpret_cast<const double2*>(xs + (size_t)r * Dp + c)
                                       : make_double2(0.0, 0.0);
        if (c + 1 >= p.D) x[r][i].y = 0.0;   // padded column of an odd-D matrix (bulk never used then)
      }
    __syncthreads();   // every thread holds its slice: the buffer may be refilled
    if (p.bulk && tid == 0) {
      const long nb = blk + XT_NBUF * stride;
      if (nb < nblocks) issue(nb, buf);
    }
    // ---- phase 1: row dot products --------------------------------------
    if constexpr (NOUT == 0) {
      constexpr int LPV = 32 / xt_pow2_ceil(Q);                  // lanes that end up holding the same direction's sum
#pragma unroll
      for (int r = 0; r < R; ++r) {
        double s[Q];
#pragma unroll
        for (int j = 0; j < Q; ++j) {
          s[j] = 0.0;
#pragma unroll
          for (int i = 0; i < CPT; ++i) s[j] = fma(x[r][i].x, v[j][i].x, fma(x[r][i].y, v[j][i].y, s[j]));
        }
        const double t = xt_transpose_reduce<Q>(s, lane);
        const int j = lane / LPV;
        if (lane % LPV == 0 && j < Q) s_part[(warp * R + r) * Q + j] = t;
      }
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < Q; ++j) {
          double s = 0.0;
#pragma unroll
          for (int i = 0; i < CPT; ++i) s = fma(x[r][i].x, v[j][i].x, fma(x[r][i].y, v[j][i].y, s));
          s = warp_sum(s);
          if (lane == 0) s_part[(warp * R + r) * Q + j] = s;
        }
    }
    __syncthreads();
    if constexpr (NOUT == 0) {
      // R * Q threads, one output each: consecutive threads store consecutive rows of one direction
      if (tid < R * Q) {
        const int r = tid % R, j = tid / R;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += s_part[(w * R + r) * Q + j];
        if (r < rows) op.store(row0 + r, j, s, aux);
      }
    } else if (tid < R) {
      double t[Q];
#pragma unroll
      for (int j = 0; j < Q; ++j) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += s_part[(w * R + tid) * Q + j];
        t[j] = s;
      }
      if constexpr (CMAX) {
        double uq[2] = {0.0, 0.0};
        if (tid < rows) op.stats2(row0 + tid, t, aux, uq);
        s_u[tid] = uq[0];
        s_q[tid] = uq[1];
      } else if constexpr (NOUT == 1) {
        s_u[tid] = (tid < rows) ? op(row0 + tid, t, aux) : 0.0;
      } else {
        double u[NOUT];
#pragma unroll
        for (int o = 0; o < NOUT; ++o) u[o] = 0.0;
        if (tid < rows) op.multi(row0 + tid, t, aux, u);
#pragma unroll
        for (int o = 0; o < NOUT; ++o) s_u[tid * NOUT + o] = u[o];
      }
    }
    if (NOUT > 0 && p.partial) {
      __syncthreads();
      // ---- phase 2: rank-R update of the column sums --------------------
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
          const double u = s_u[r * NOUT + o];
#pragma unroll
          for (int i = 0; i < CPT; ++i) {
            acc[o][i].x = fma(u, x[r][i].x, acc[o][i].x);
            acc[o][i].y = fma(u, x[r][i].y, acc[o][i].y);
          }
        }
      if constexpr (CMAX) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const double q = s_q[r];
#pragma unroll
          for (int i = 0; i < CPT; ++i) {
            cmx[2 * i] = xt_himax(cmx[2 * i], q * fabs(x[r][i].x));
            cmx[2 * i + 1] = xt_himax(cmx[2 * i + 1], q * fabs(x[r][i].y));
          }
        }
      }
    }
    // s_part / s_u are rewritten only after the next block's first barrier
  }
  if (NOUT > 0 && p.partial) {
#pragma unroll
    for (int o = 0; o < NOUT; ++o)
#pragma unroll
      for (int i = 0; i < CPT; ++i) {
        const int c = 2 * tid + 512 * i;
        if (c < Dp) *reinterpret_cast<double2*>(p.partial + ((size_t)blockIdx.x * NOUT + o) * Dp + c) = acc[o][i];
      }
    if constexpr (CMAX) {
#pragma unroll
      for (int i = 0; i < CPT; ++i) {
        const int c = 2 * tid + 512 * i;
        if (c < Dp)
          *reinterpret_cast<double2*>(p.partial_max + (size_t)blockIdx.x * Dp + c) =
              make_double2(__hiloint2double((int)cmx[2 * i], 0), __hiloint2double((int)cmx[2 * i + 1], 0));
      }
    }
  }
}

// out[c] = alpha * sum_cta partial[cta * stride + c] + beta_vec * addvec[c]
__global__ void xtfx_reduce_kernel(const double* partial, int ncta, int stride, int D, double* out, double alpha,
                                   const double* addvec, double beta_vec);

}  // namespace vt
