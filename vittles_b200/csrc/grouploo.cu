// Per-group Gram of U and the leave-one-group-out predictors (see grouploo.cuh).
//
// A block of GL_THREADS threads owns the groups that start in GL_SPAN consecutive rows [b0, b0 + GL_SPAN); their rows
// lie in [b0, b0 + GL_SPAN + 31) and thread t takes row b0 + t (at most 31 of the GL_THREADS threads go idle at either
// end).  Tiles of GL_KT features x GL_THREADS rows of U are staged in shared memory; thread t accumulates row t of
// its group's Q (m values, one FMA and one shared-memory load each: the threads of a group read the same word), in
// feature order.  For 'ns' the rows of M then go to shared memory and the threads of a group run the right-looking
// Cholesky of M and the two triangular solves together, one barrier per step.
#include "grouploo.cuh"

namespace vt {
namespace {

constexpr int GL_THREADS = 256;
constexpr int GL_SPAN = GL_THREADS - GROUP_LOO_MAXM;             // group starts per block
constexpr int GL_TW = GL_THREADS + GROUP_LOO_MAXM + 1;           // tile pitch: columns t0 + k < GL_THREADS + 32 stay
                                                                 // inside; odd, so the transposed fill is 2-way only
constexpr int GL_MP = GROUP_LOO_MAXM + 1;                        // pitch of a row of M
constexpr int GL_BUF = GL_THREADS * GL_MP;                       // doubles: M, or a tile of U
constexpr int GL_KT = GL_BUF / GL_TW;                            // features per tile (29)
constexpr size_t GL_SMEM = (size_t)(GL_BUF + 3 * GL_THREADS) * 8 + (size_t)(GL_SPAN + 1 + GL_THREADS + 8) * 4;

__device__ __forceinline__ long lower_bound_i64(const int64_t* a, long n, long key) {
  long lo = 0, hi = n;
  while (lo < hi) {
    const long mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(GL_THREADS, 2) group_loo_kernel(const GroupLooChunk a) {
  extern __shared__ double gl_smem[];
  double* buf = gl_smem;                                         // tile [GL_KT][GL_TW], later M [GL_THREADS][GL_MP]
  double* ssq = buf + GL_BUF;                                    // sqrt(s) of the window's rows
  double* sv = ssq + GL_THREADS;                                 // S^1/2 t, then the forward solve
  double* sy = sv + GL_THREADS;                                  // M^{-1} S^1/2 t
  int* sst = reinterpret_cast<int*>(sy + GL_THREADS);            // starts of the owned groups, minus b0
  int* sbad = sst + GL_SPAN + 1;                                 // per group (at its first thread): a pivot failed
  int* smax = sbad + GL_THREADS;
  __shared__ long sg[2];

  const int t = threadIdx.x;
  const long b0 = a.lo + (long)blockIdx.x * GL_SPAN;
  const long b1 = (b0 + GL_SPAN < a.hi) ? b0 + GL_SPAN : a.hi;
  if (t == 0) {
    sg[0] = lower_bound_i64(a.starts, a.G + 1, b0);
    sg[1] = lower_bound_i64(a.starts, a.G + 1, b1);
  }
  __syncthreads();
  const long g0 = sg[0];
  const int ng = (int)(sg[1] - g0);                              // owned groups: [g0, g0 + ng)
  for (int k = t; k <= ng; k += GL_THREADS) sst[k] = (int)(a.starts[g0 + k] - b0);
  sbad[t] = 0;
  __syncthreads();

  const int row_begin = sst[0], row_end = sst[ng];               // window columns of the owned rows
  const bool owned = ng > 0 && t >= row_begin && t < row_end;
  int tb = 0, m = 0;                                             // this row's group: window columns [tb, tb + m)
  if (owned) {
    int lo = 0, hi = ng;                                         // the last k with sst[k] <= t
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (sst[mid] <= t) lo = mid; else hi = mid;
    }
    tb = sst[lo];
    m = sst[lo + 1] - tb;
  }
  const int ai = t - tb;                                         // position in the group
  {
    const int mw = __reduce_max_sync(0xffffffffu, (unsigned)m);
    if ((t & 31) == 0) smax[t >> 5] = mw;
  }
  __syncthreads();
  int kmax = 0;
#pragma unroll
  for (int w = 0; w < GL_THREADS / 32; ++w) kmax = smax[w] > kmax ? smax[w] : kmax;

  // ---- Gram: acc[k] = sum_i U[i][row] U[i][tb + k], features in order ----
  double acc[GROUP_LOO_MAXM];
#pragma unroll
  for (int k = 0; k < GROUP_LOO_MAXM; ++k) acc[k] = 0.0;
  const long rloc0 = b0 - a.r0;                                  // chunk row of window column 0
  const long cmax = a.rows - rloc0;                              // window columns inside the chunk
  const int c_hi = (long)row_end < cmax ? row_end : (int)cmax;
  for (int i0 = 0; i0 < a.D; i0 += GL_KT) {
    const int kt = (a.D - i0 < GL_KT) ? a.D - i0 : GL_KT;
    __syncthreads();
    if (a.sr == 1) {                                             // rows contiguous: a feature's row segment per pass
      for (int e = t; e < GL_KT * GL_TW; e += GL_THREADS) {
        const int i = e / GL_TW, c = e - i * GL_TW;
        buf[e] = (i < kt && c >= row_begin && c < c_hi) ? a.U[(rloc0 + c) + (long)(i0 + i) * a.sf] : 0.0;
      }
    } else {                                                     // features contiguous: GL_KT of a row per pass
      for (int e = t; e < GL_KT * GL_TW; e += GL_THREADS) {
        const int c = e / GL_KT, i = e - c * GL_KT;
        buf[i * GL_TW + c] = (i < kt && c >= row_begin && c < c_hi) ? a.U[(rloc0 + c) * a.sr + (long)(i0 + i) * a.sf]
                                                                    : 0.0;
      }
    }
    __syncthreads();
    if (owned) {
      for (int i = 0; i < kt; ++i) {
        const double* row = buf + i * GL_TW;
        const double ur = row[t];
#pragma unroll
        for (int k = 0; k < GROUP_LOO_MAXM; ++k) {
          if (k >= kmax) break;
          acc[k] = fma(ur, row[tb + k], acc[k]);
        }
      }
    }
  }

  // ---- h = Q_aa, t = Q u ----
  const long r = b0 + t;
  const long gs = b0 + tb;                                       // global first row of the group
  double hq = 0.0, tq = 0.0;
  if (owned) {
#pragma unroll
    for (int k = 0; k < GROUP_LOO_MAXM; ++k) {
      if (k >= m) break;
      if (k == ai) hq = acc[k];
      tq = fma(acc[k], a.u[gs + k], tq);
    }
  }
  if (a.method == GROUP_LOO_IJ) {
    if (owned) {
      a.h[r] = hq;
      a.zpred[r] = a.z[r] + tq;
    }
    return;
  }

  // ---- 'ns': M = I - S^1/2 Q S^1/2 (lower triangle, row per thread), factored in place ----
  __syncthreads();                                               // the tile buffer becomes M
  double* Ma = buf + t * GL_MP;
  const double sa = owned ? sqrt(a.s[r]) : 0.0;
  ssq[t] = sa;
  __syncthreads();
  if (owned) {
#pragma unroll
    for (int k = 0; k < GROUP_LOO_MAXM; ++k) {
      if (k > ai) break;
      Ma[k] = (k == ai ? 1.0 : 0.0) - sa * acc[k] * ssq[tb + k];
    }
  }
  sv[t] = sa * tq;
  __syncthreads();
  // Step j: the pivot p_j = M^(j)[j][j]; rows a > j subtract M^(j)[a][j] / p_j times row j from columns j + 1 .. a
  // and from the right-hand side (the forward solve L w = S^1/2 t of M = L diag(p) L^T rides along).  Column j is
  // read, never written, during step j.
  for (int j = 0; j < kmax; ++j) {
    if (owned && j < m) {
      const double* Mj = buf + (tb + j) * GL_MP;
      if (ai == j) {
        if (!(Mj[j] > 0x1p-40)) sbad[tb] = 1;
      } else if (ai > j) {
        const double l = Ma[j] / Mj[j];
        for (int b = j + 1; b <= ai; ++b) Ma[b] = fma(-l, buf[(tb + b) * GL_MP + j], Ma[b]);
        sv[t] = fma(-l, sv[tb + j], sv[t]);
      }
    }
    __syncthreads();
  }
  // Backward: y_a = (w_a - sum_{b > a} M^(a)[b][a] y_b) / p_a, b from the last row down.
  for (int j = kmax - 1; j >= 0; --j) {
    if (owned && ai == j) sy[t] = sv[t] / Ma[j];
    __syncthreads();
    if (owned && ai < j && j < m) sv[t] = fma(-buf[(tb + j) * GL_MP + ai], sy[tb + j], sv[t]);
  }
  __syncthreads();
  if (owned) {
    double q = 0.0;                                              // (Q S^1/2 y)_a
#pragma unroll
    for (int k = 0; k < GROUP_LOO_MAXM; ++k) {
      if (k >= m) break;
      q = fma(acc[k], ssq[tb + k] * sy[tb + k], q);
    }
    a.h[r] = hq;
    a.zpred[r] = sbad[tb] ? __longlong_as_double(0x7ff8000000000000LL) : (a.z[r] + tq) + q;
  }
}

}  // namespace

int group_loo_chunk(const GroupLooChunk& c, cudaStream_t stream) {
  if (c.hi <= c.lo) return VT_OK;
  VT_CUDA(cudaFuncSetAttribute(group_loo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GL_SMEM));
  const long blocks = (c.hi - c.lo + GL_SPAN - 1) / GL_SPAN;
  group_loo_kernel<<<(unsigned)blocks, GL_THREADS, GL_SMEM, stream>>>(c);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

}  // namespace vt
