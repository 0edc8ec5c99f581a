// GLM-family instances of the fused X^T f(X V) pass (xtfx.cuh), the dense
// prediction GEMV, and the conjugate-gradient vector kernels.
//
// Family: f(theta, w) = sum_n w_n [ b(z_n) - y_n z_n ],  z = X theta.
//   logistic: b = softplus,  poisson: b = exp,  gaussian: b = z^2/2.
// Reference call sites these kernels replace (closed forms of the autograd
// sweeps): gradient `sensitivity_lib.py:354`, Hessian-vector products behind
// `solver_lib.py:70-98` (get_cg_solver's mat_times_vec), nested JVPs
// `sensitivity_lib.py:440-492,788-807`, prediction GEMV `:245-247`.
#include "xtfx.cuh"
#include "glm.cuh"
#include <cmath>

namespace vt {

__global__ void xtfx_reduce_kernel(const double* partial, int ncta, int stride, int D, double* out, double alpha,
                                   const double* addvec, double beta_vec) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  double s = 0.0;
  for (int k = 0; k < ncta; ++k) s += partial[(size_t)k * stride + c];
  s *= alpha;
  if (addvec) s += beta_vec * addvec[c];
  out[c] = s;
}

namespace {

// b^{(k)}(z) for the logistic family is a degree-k polynomial in sigma(z):
// P_1 = s,  P_{k+1} = P_k'(s) * (s - s^2).  Coefficients are built on the host.
struct Poly {
  double c[GLM_MAX_BDERIV + 2];
  int deg;
};

static Poly logistic_poly(int k) {
  double cur[GLM_MAX_BDERIV + 2] = {0.0, 1.0};
  int deg = 1;
  for (int it = 1; it < k; ++it) {
    double der[GLM_MAX_BDERIV + 2] = {0};
    for (int i = 1; i <= deg; ++i) der[i - 1] = i * cur[i];
    double nxt[GLM_MAX_BDERIV + 2] = {0};
    for (int i = 0; i < deg; ++i) {
      nxt[i + 1] += der[i];
      nxt[i + 2] -= der[i];
    }
    deg += 1;
    for (int i = 0; i <= deg; ++i) cur[i] = nxt[i];
  }
  Poly p;
  p.deg = deg;
  for (int i = 0; i < GLM_MAX_BDERIV + 2; ++i) p.c[i] = i <= deg ? cur[i] : 0.0;
  return p;
}

__device__ __forceinline__ double sigmoid(double z) {
  // stable in both tails
  if (z >= 0) {
    const double e = exp(-z);
    return 1.0 / (1.0 + e);
  }
  const double e = exp(z);
  return e / (1.0 + e);
}

// k-th derivative of b at z (k >= 1)
__device__ __forceinline__ double b_deriv(int family, int k, double z, const Poly& poly) {
  if (family == GLM_LOGISTIC) {
    const double s = sigmoid(z);
    double r = poly.c[poly.deg];
    for (int i = poly.deg - 1; i >= 0; --i) r = fma(r, s, poly.c[i]);
    return r;
  }
  if (family == GLM_POISSON) return exp(z);
  return k == 1 ? z : (k == 2 ? 1.0 : 0.0);
}

struct StatsOp {
  const double* y; const double* w;
  double* z; double* resid; double* s;
  int family;
  double* sq;        // CMAX kernels: sqrt(s_n), kept for the slicing kernels of the INT8 Hessian assembly
  struct Aux { double y, w; };
  __device__ Aux load(long n) const { return Aux{y[n], w ? w[n] : 1.0}; }
  __device__ double eval(long n, const double* t, const Aux& a, double* s_out) const {
    const double zz = t[0];
    double mu, var;
    if (family == GLM_LOGISTIC) { mu = sigmoid(zz); var = mu * (1.0 - mu); }
    else if (family == GLM_POISSON) { mu = exp(zz); var = mu; }
    else { mu = zz; var = 1.0; }
    const double r = mu - a.y;
    if (z) z[n] = zz;
    if (resid) resid[n] = r;
    const double sv = a.w * var;
    if (s) s[n] = sv;
    *s_out = sv;
    return a.w * r;
  }
  __device__ double operator()(long n, const double* t, const Aux& a) const {
    double sv;
    return eval(n, t, a, &sv);
  }
  // uq[0] = w_n resid_n (the gradient weight), uq[1] = sqrt(s_n) (the weight of the column maxima)
  __device__ void stats2(long n, const double* t, const Aux& a, double* uq) const {
    double sv;
    uq[0] = eval(n, t, a, &sv);
    const double q = (sv == sv) ? sqrt(fmax(sv, 0.0)) : sv;        // a NaN weight stays NaN (fmax would drop it)
    if (sq) sq[n] = q;
    uq[1] = q;
  }
};

// colmax[c] = max over the CTAs, as the bit pattern of a non-negative double (orders like an unsigned integer; the
// quiet-NaN pattern is above every finite one) - the form the slicing kernels read
__global__ void xtfx_reduce_max_kernel(const double* partial_max, int ncta, int stride, int D,
                                       unsigned long long* colmax) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  unsigned long long m = 0ULL;
  for (int k = 0; k < ncta; ++k) {
    const unsigned long long v = (unsigned long long)__double_as_longlong(partial_max[(size_t)k * stride + c]);
    m = v > m ? v : m;
  }
  colmax[c] = m;
}

struct HvpOp {
  const double* s;
  struct Aux { double s; };
  __device__ Aux load(long n) const { return Aux{s[n]}; }
  __device__ double operator()(long n, const double* t, const Aux& a) const { return a.s * t[0]; }
};

// Q Hessian-vector products in one pass: u_j = s_n (x_n . v_j)
template <int Q>
struct HvpMultiOp {
  const double* s;
  struct Aux { double s; };
  __device__ Aux load(long n) const { return Aux{s[n]}; }
  __device__ double operator()(long n, const double* t, const Aux& a) const { return a.s * t[0]; }
  __device__ void multi(long n, const double* t, const Aux& a, double* u) const {
#pragma unroll
    for (int j = 0; j < Q; ++j) u[j] = a.s * t[j];
  }
};

// coef[n] = w_n * b^{(k)}(z_n): elementwise pre-pass of the directional derivative
__global__ void __launch_bounds__(256) glm_coef_kernel(const double* __restrict__ z, const double* __restrict__ w,
                                                       long N, int family, int k, const Poly poly, double* coef) {
  for (long n = (long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long)gridDim.x * blockDim.x)
    coef[n] = b_deriv(family, k, z[n], poly) * (w ? w[n] : 1.0);
}

template <int Q>
struct DirDerivOp {
  const double* coef;
  struct Aux { double c; };
  __device__ Aux load(long n) const { return Aux{coef[n]}; }
  __device__ double operator()(long n, const double* t, const Aux& a) const {
    double u = a.c;
#pragma unroll
    for (int j = 0; j < Q; ++j) u *= t[j];
    return u;
  }
};

// out[j * ldo + n] = alpha * c_n * (x_n . v_j): the per-observation influence of Q quantities of interest
struct InfluenceOp {
  const double* c;
  double* out;
  long ldo;
  double alpha;
  struct Aux { double c; };
  __device__ Aux load(long n) const { return Aux{c[n]}; }
  __device__ void store(long n, int j, double t, const Aux& a) const { out[(long)j * ldo + n] = alpha * (a.c * t); }
};

template <class RowOp, int Q, int CPT, int NOUT = 1, bool CMAX = false>
int launch_xtfx(const XtfxParams& p, const RowOp& op, cudaStream_t stream, int* grid_out) {
  constexpr int R = (CPT <= 8) ? 8 / CPT : 1;
  constexpr int CTAS_PER_SM = xt_ctas_per_sm<Q, CPT, R, NOUT>();
  const size_t smem = xtfx_smem_bytes(p.Dp, R, Q);
  VT_CUDA(cudaFuncSetAttribute(xtfx_kernel<RowOp, Q, CPT, R, NOUT, CMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long nblocks = (p.N + R - 1) / R;
  const long cap = (long)num_sms() * CTAS_PER_SM;
  const int grid = (int)(nblocks < cap ? nblocks : cap);
  xtfx_kernel<RowOp, Q, CPT, R, NOUT, CMAX><<<grid, XT_THREADS, smem, stream>>>(p, op);
  VT_LAUNCH_CHECK();
  *grid_out = grid;
  return VT_OK;
}

template <class RowOp, int Q, int NOUT = 1>
int dispatch_cpt(const XtfxParams& p, const RowOp& op, cudaStream_t stream, int* grid_out) {
  const int D = p.D;
  if (D <= 512) return launch_xtfx<RowOp, Q, 1, NOUT>(p, op, stream, grid_out);
  if (D <= 1024) return launch_xtfx<RowOp, Q, 2, NOUT>(p, op, stream, grid_out);
  if (D <= 2048) return launch_xtfx<RowOp, Q, 4, NOUT>(p, op, stream, grid_out);
  if constexpr (Q == 1) {
    if (D <= 4096) return launch_xtfx<RowOp, 1, 8>(p, op, stream, grid_out);
    if (D <= 8192) return launch_xtfx<RowOp, 1, 16>(p, op, stream, grid_out);
  }
  set_error("xtfx: D=%d with %d directions is not supported (D <= 2048, or <= 8192 for one direction)", D, Q);
  return VT_ERR_INVALID;
}

// statistics pass that also produces the column maxima (D <= 2048: the accumulators double)
int dispatch_stats_cmax(const XtfxParams& p, const StatsOp& op, cudaStream_t stream, int* grid_out) {
  const int D = p.D;
  if (D <= 512) return launch_xtfx<StatsOp, 1, 1, 1, true>(p, op, stream, grid_out);
  if (D <= 1024) return launch_xtfx<StatsOp, 1, 2, 1, true>(p, op, stream, grid_out);
  if (D <= 2048) return launch_xtfx<StatsOp, 1, 4, 1, true>(p, op, stream, grid_out);
  set_error("glm_stats: column maxima are fused for D <= 2048 only (D = %d)", D);
  return VT_ERR_INVALID;
}

int make_params(XtfxParams& p, const double* X, long ldx, long N, int D, const double* V, double* workspace,
                size_t workspace_bytes, bool need_partial) {
  VT_REQUIRE(X && V, "xtfx: null pointer");
  VT_REQUIRE(N >= 1 && D >= 1 && ldx >= D, "xtfx: bad shape N=%ld D=%d ldx=%ld", N, D, ldx);
  p.X = X; p.ldx = ldx; p.N = N; p.D = D; p.V = V;
  p.Dp = (D + 1) & ~1;
  p.contiguous = (ldx == D);
  p.bulk = (D % 2 == 0) && (reinterpret_cast<uintptr_t>(X) % 16 == 0) && (p.contiguous || ldx % 2 == 0);
  p.partial = nullptr;
  p.partial_max = nullptr;
  if (need_partial) {
    VT_REQUIRE(workspace && workspace_bytes >= glm_workspace_bytes(D),
               "xtfx: workspace too small: need %zu bytes", glm_workspace_bytes(D));
    p.partial = workspace;
  }
  return VT_OK;
}

}  // namespace

size_t glm_workspace_bytes(int D) { return (size_t)num_sms() * 2 * ((D + 1) & ~1) * 8; }

int glm_stats(const double* X, long ldx, long N, int D, const double* theta, const double* y, const double* w,
              int family, double* z, double* resid, double* s, double* grad, double l2, double* sq,
              unsigned long long* colmax, double* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(y, "glm_stats: y is null");
  VT_REQUIRE(family >= 0 && family <= 2, "glm_stats: unknown family %d", family);
  const bool cmax = colmax != nullptr;
  VT_REQUIRE(!cmax || (sq && D <= 2048), "glm_stats: fused column maxima need `sq` and D <= 2048");
  XtfxParams p;
  int st = make_params(p, X, ldx, N, D, theta, workspace, workspace_bytes, grad != nullptr || cmax);
  if (st != VT_OK) return st;
  StatsOp op{y, w, z, resid, s, family, cmax ? sq : nullptr};
  int grid = 0;
  if (cmax) {
    VT_REQUIRE(workspace_bytes >= 2 * glm_workspace_bytes(D), "glm_stats: workspace too small for the column maxima");
    p.partial_max = workspace + glm_workspace_bytes(D) / 8;
    st = dispatch_stats_cmax(p, op, stream, &grid);
  } else {
    st = dispatch_cpt<StatsOp, 1>(p, op, stream, &grid);
  }
  if (st != VT_OK) return st;
  if (grad) {
    xtfx_reduce_kernel<<<(D + 255) / 256, 256, 0, stream>>>(p.partial, grid, p.Dp, D, grad, 1.0, theta, l2);
    VT_LAUNCH_CHECK();
  }
  if (cmax) {
    xtfx_reduce_max_kernel<<<(D + 255) / 256, 256, 0, stream>>>(p.partial_max, grid, p.Dp, D, colmax);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

int glm_hvp(const double* X, long ldx, long N, int D, const double* s, const double* v, double ridge, double* out,
            double* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(s && out, "glm_hvp: null pointer");
  XtfxParams p;
  int st = make_params(p, X, ldx, N, D, v, workspace, workspace_bytes, true);
  if (st != VT_OK) return st;
  HvpOp op{s};
  int grid = 0;
  st = dispatch_cpt<HvpOp, 1>(p, op, stream, &grid);
  if (st != VT_OK) return st;
  xtfx_reduce_kernel<<<(D + 255) / 256, 256, 0, stream>>>(p.partial, grid, p.Dp, D, out, 1.0, v, ridge);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

// out (q x D) = V X^T diag(s) X + ridge V for q <= XT_MAXQ directions (rows of V): ONE read of X for all of them.
size_t glm_hvp_multi_workspace_bytes(int D, int q) { return glm_workspace_bytes(D) * (size_t)(q < 1 ? 1 : q); }

namespace {
template <int Q>
int hvp_multi_q(XtfxParams& p, const double* s, const double* V, double ridge, double* out, cudaStream_t stream) {
  HvpMultiOp<Q> op{s};
  int grid = 0;
  int st = dispatch_cpt<HvpMultiOp<Q>, Q, Q>(p, op, stream, &grid);
  if (st != VT_OK) return st;
  for (int j = 0; j < Q; ++j) {
    xtfx_reduce_kernel<<<(p.D + 255) / 256, 256, 0, stream>>>(p.partial + (size_t)j * p.Dp, grid, Q * p.Dp, p.D,
                                                              out + (size_t)j * p.D, 1.0, V + (size_t)j * p.D, ridge);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}
}  // namespace

int glm_hvp_multi(const double* X, long ldx, long N, int D, const double* s, const double* V, int q, double ridge,
                  double* out, double* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(s && out, "glm_hvp_multi: null pointer");
  VT_REQUIRE(q >= 1 && q <= XT_MAXQ, "glm_hvp_multi: 1..%d directions per pass, got %d", XT_MAXQ, q);
  VT_REQUIRE(D <= 2048 || q == 1, "glm_hvp_multi: D <= 2048 for more than one direction");
  VT_REQUIRE(workspace && workspace_bytes >= glm_hvp_multi_workspace_bytes(D, q), "glm_hvp_multi: workspace too small");
  if (q == 1) return glm_hvp(X, ldx, N, D, s, V, ridge, out, workspace, workspace_bytes, stream);
  XtfxParams p;
  int st = make_params(p, X, ldx, N, D, V, workspace, glm_workspace_bytes(D), true);
  if (st != VT_OK) return st;
  switch (q) {
    case 2: return hvp_multi_q<2>(p, s, V, ridge, out, stream);
    case 3: return hvp_multi_q<3>(p, s, V, ridge, out, stream);
    default: return hvp_multi_q<4>(p, s, V, ridge, out, stream);
  }
}

// Directions per influence pass: the Q x CPT direction registers of a thread bound Q (no spills, -Xptxas -v)
int glm_influence_max_directions(int D) {
  if (D < 1) return 0;
  if (D <= 2048) return GLM_INFLUENCE_MAXQ;
  if (D <= 4096) return 2;
  if (D <= 8192) return 1;
  return 0;
}

namespace {
template <int Q>
int influence_q(const XtfxParams& p, const InfluenceOp& op, cudaStream_t stream) {
  int grid = 0;
  const int D = p.D;
  if (D <= 512) return launch_xtfx<InfluenceOp, Q, 1, 0>(p, op, stream, &grid);
  if (D <= 1024) return launch_xtfx<InfluenceOp, Q, 2, 0>(p, op, stream, &grid);
  if (D <= 2048) return launch_xtfx<InfluenceOp, Q, 4, 0>(p, op, stream, &grid);
  if constexpr (Q <= 2) {
    if (D <= 4096) return launch_xtfx<InfluenceOp, Q, 8, 0>(p, op, stream, &grid);
  }
  if constexpr (Q == 1) {
    if (D <= 8192) return launch_xtfx<InfluenceOp, 1, 16, 0>(p, op, stream, &grid);
  }
  set_error("glm_influence: %d directions at D = %d exceed the per-pass limit", Q, D);
  return VT_ERR_INVALID;
}
}  // namespace

int glm_influence(const double* X, long ldx, long N, int D, const double* c, const double* V, int q, double alpha,
                  double* out, long ldo, cudaStream_t stream) {
  VT_REQUIRE(c && out, "glm_influence: null pointer");
  VT_REQUIRE(D >= 1 && D <= 8192, "glm_influence: D = %d is not supported (1 <= D <= 8192)", D);
  const int qmax = glm_influence_max_directions(D);
  VT_REQUIRE(q >= 1 && q <= qmax, "glm_influence: 1..%d directions per pass at D = %d, got %d", qmax, D, q);
  VT_REQUIRE(ldo >= N, "glm_influence: ldo = %ld < N = %ld", ldo, N);
  XtfxParams p;
  int st = make_params(p, X, ldx, N, D, V, nullptr, 0, false);
  if (st != VT_OK) return st;
  const InfluenceOp op{c, out, ldo, alpha};
  switch (q) {
    case 1: return influence_q<1>(p, op, stream);
    case 2: return influence_q<2>(p, op, stream);
    case 3: return influence_q<3>(p, op, stream);
    case 4: return influence_q<4>(p, op, stream);
    case 5: return influence_q<5>(p, op, stream);
    case 6: return influence_q<6>(p, op, stream);
    case 7: return influence_q<7>(p, op, stream);
    default: return influence_q<8>(p, op, stream);
  }
}

size_t glm_dirderiv_workspace_bytes(long N, int D) { return glm_workspace_bytes(D) + (size_t)N * 8; }

int glm_dirderiv(const double* X, long ldx, long N, int D, const double* z, const double* w, int family,
                 const double* dirs, int q, double* out, double* workspace, size_t workspace_bytes,
                 cudaStream_t stream) {
  VT_REQUIRE(z && out, "glm_dirderiv: null pointer");
  VT_REQUIRE(q >= 1 && q <= XT_MAXQ, "glm_dirderiv: number of directions must be 1..%d, got %d", XT_MAXQ, q);
  VT_REQUIRE(q + 1 <= GLM_MAX_BDERIV, "glm_dirderiv: derivative order too high");
  VT_REQUIRE(family >= 0 && family <= 2, "glm_dirderiv: unknown family %d", family);
  VT_REQUIRE(workspace && workspace_bytes >= glm_dirderiv_workspace_bytes(N, D),
             "glm_dirderiv: workspace too small: need %zu bytes", glm_dirderiv_workspace_bytes(N, D));
  XtfxParams p;
  int st = make_params(p, X, ldx, N, D, dirs, workspace, workspace_bytes, true);
  if (st != VT_OK) return st;
  double* coef = workspace + glm_workspace_bytes(D) / 8;
  const Poly poly = logistic_poly(q + 1);
  const long want = (N + 255) / 256;
  const int cgrid = (int)(want < (long)num_sms() * 8 ? want : (long)num_sms() * 8);
  glm_coef_kernel<<<cgrid, 256, 0, stream>>>(z, w, N, family, q + 1, poly, coef);
  VT_LAUNCH_CHECK();
  int grid = 0;
  switch (q) {
    case 1: { DirDerivOp<1> op{coef}; st = dispatch_cpt<DirDerivOp<1>, 1>(p, op, stream, &grid); break; }
    case 2: { DirDerivOp<2> op{coef}; st = dispatch_cpt<DirDerivOp<2>, 2>(p, op, stream, &grid); break; }
    case 3: { DirDerivOp<3> op{coef}; st = dispatch_cpt<DirDerivOp<3>, 3>(p, op, stream, &grid); break; }
    default: { DirDerivOp<4> op{coef}; st = dispatch_cpt<DirDerivOp<4>, 4>(p, op, stream, &grid); break; }
  }
  if (st != VT_OK) return st;
  xtfx_reduce_kernel<<<(D + 255) / 256, 256, 0, stream>>>(p.partial, grid, p.Dp, D, out, 1.0, nullptr, 0.0);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

// ---------------------------------------------------------------------------
// y = alpha * A x + beta * y0  for a row-major A (M x N) with N long: the
// prediction theta_hat + S (lam1 - lam0) (sensitivity_lib.py:245-247) with
// S = (D, N).  HBM-bound: one streaming read of A.  Each CTA owns a (row,
// column-chunk) pair; chunk sums are combined in a fixed order.
// ---------------------------------------------------------------------------
namespace {
constexpr int GEMV_THREADS = 256;
constexpr int GEMV_CHUNK = 256 * 2 * 16;   // columns per CTA pass (64 KB of A)

__global__ void __launch_bounds__(GEMV_THREADS) gemv_rows_kernel(const double* __restrict__ A, long lda, int M, long N,
                                                                  const double* __restrict__ x, double* partial,
                                                                  int nchunks) {
  const int row = blockIdx.y;
  const int chunk = blockIdx.x;
  const long c0 = (long)chunk * GEMV_CHUNK;
  const long c1 = min(N, c0 + GEMV_CHUNK);
  const double* a = A + (long)row * lda;
  const bool vec = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(x)) % 16 == 0);
  double s = 0.0;
  if (vec) {
    for (long c = c0 + 2 * threadIdx.x; c + 1 < c1; c += 2 * GEMV_THREADS) {
      const double2 av = ld_stream2(a + c);
      const double2 xv = *reinterpret_cast<const double2*>(x + c);
      s = fma(av.x, xv.x, fma(av.y, xv.y, s));
    }
    if (((c1 - c0) & 1) && threadIdx.x == 0) s = fma(a[c1 - 1], x[c1 - 1], s);
  } else {
    for (long c = c0 + threadIdx.x; c < c1; c += GEMV_THREADS) s = fma(a[c], x[c], s);
  }
  __shared__ double red[GEMV_THREADS / 32];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < GEMV_THREADS / 32; ++i) t += red[i];
    partial[(size_t)row * nchunks + chunk] = t;
  }
}

__global__ void gemv_finish_kernel(const double* partial, int M, int nchunks, double alpha, const double* y0,
                                   double beta, double* y) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= M) return;
  double s = 0.0;
  for (int k = 0; k < nchunks; ++k) s += partial[(size_t)row * nchunks + k];
  y[row] = alpha * s + (y0 ? beta * y0[row] : 0.0);
}
}  // namespace

size_t gemv_workspace_bytes(int M, long N) {
  const long nchunks = (N + GEMV_CHUNK - 1) / GEMV_CHUNK;
  return (size_t)M * nchunks * 8;
}

int gemv_rows(const double* A, long lda, int M, long N, const double* x, double alpha, const double* y0, double beta,
              double* y, double* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(A && x && y, "gemv: null pointer");
  VT_REQUIRE(M >= 1 && N >= 1 && lda >= N, "gemv: bad shape");
  VT_REQUIRE(M <= 65535, "gemv: at most 65535 rows");
  const long nchunks = (N + GEMV_CHUNK - 1) / GEMV_CHUNK;
  VT_REQUIRE(workspace && workspace_bytes >= gemv_workspace_bytes(M, N), "gemv: workspace too small");
  dim3 grid((unsigned)nchunks, (unsigned)M);
  gemv_rows_kernel<<<grid, GEMV_THREADS, 0, stream>>>(A, lda, M, N, x, workspace, (int)nchunks);
  VT_LAUNCH_CHECK();
  gemv_finish_kernel<<<(M + 255) / 256, 256, 0, stream>>>(workspace, M, (int)nchunks, alpha, y0, beta, y);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

// ---------------------------------------------------------------------------
// Conjugate-gradient vector kernels, batched over K right-hand sides.  Every column runs scipy's cg (the reference's
// solver, solver_lib.py:91-97, legacy stopping rule) step for step on its own scalars, so that each column stops at
// the iteration scipy would stop at; the columns only share the matrix-vector product (one fused pass over X for
// up to four of them).  All scalars stay on the device - the host never reads a residual norm:
//   state[k] = {rho, rho_prev, p.q, |r|^2, |b|^2, tol, status, matvecs}     status 1: running, 0: converged,
//                                                                           2: stopped at maxiter
//   cg_batch_update_p : if |r| < tol: status 0.  else z = M r (z given, or minv .* r, or r), rho = r.z,
//                       p = z + (rho / rho_prev) p.  Columns that are not running get p = 0.
//   cg_batch_update_xr: alpha = rho / (p.q);  x += alpha p;  r -= alpha q;  |r|^2
// Vectors are rows of (K, D) arrays.  One CTA of 1024 threads per column: D is at most a few thousand, so one block
// does the vector update and the deterministic reduction in one launch.
// ---------------------------------------------------------------------------
namespace {
__device__ double block_sum_1024(double v, double* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 32) {
    t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
    t = warp_sum(t);
  }
  __syncthreads();
  if (threadIdx.x == 0) red[0] = t;
  __syncthreads();
  t = red[0];
  __syncthreads();
  return t;
}

constexpr int CG_RHO = 0, CG_RHO_PREV = 1, CG_PQ = 2, CG_RNORM2 = 3, CG_BNORM2 = 4, CG_TOL = 5, CG_STATUS = 6, CG_ITERS = 7;

__global__ void __launch_bounds__(1024) cg_batch_init_kernel(int D, const double* B, double* X, double* R, double* state,
                                                             double rtol, double atol, int keep_xr) {
  __shared__ double red[32];
  const long off = (long)blockIdx.x * D;
  const double* b = B + off;
  double* x = X + off;
  double* r = R + off;
  double* st = state + 8L * blockIdx.x;
  double sb = 0.0, sr = 0.0;
  for (int i = threadIdx.x; i < D; i += blockDim.x) {
    const double bi = b[i];
    if (!keep_xr) { x[i] = 0.0; r[i] = bi; }
    const double ri = r[i];
    sb = fma(bi, bi, sb);
    sr = fma(ri, ri, sr);
  }
  sb = block_sum_1024(sb, red);
  sr = block_sum_1024(sr, red);
  if (threadIdx.x == 0) {
    const double bn = sqrt(sb);
    st[CG_RHO] = 0.0; st[CG_RHO_PREV] = 0.0; st[CG_PQ] = 0.0;
    st[CG_RNORM2] = sr; st[CG_BNORM2] = sb;
    st[CG_TOL] = fmax(atol, rtol * bn);
    st[CG_STATUS] = (sb == 0.0) ? 0.0 : 1.0;       // scipy: a zero right-hand side returns x = b at once
    st[CG_ITERS] = 0.0;
  }
  if (sb == 0.0 && !keep_xr) return;
  if (sb == 0.0)
    for (int i = threadIdx.x; i < D; i += blockDim.x) x[i] = 0.0;
}

__global__ void __launch_bounds__(1024) cg_batch_update_p_kernel(int D, const double* R, const double* Zin,
                                                                 const double* minv, double* P, double* state,
                                                                 int maxiter) {
  __shared__ double red[32];
  const long off = (long)blockIdx.x * D;
  const double* r = R + off;
  double* p = P + off;
  double* st = state + 8L * blockIdx.x;
  double status = st[CG_STATUS];
  const double iters = st[CG_ITERS];
  if (status == 1.0) {
    if (sqrt(st[CG_RNORM2]) < st[CG_TOL]) status = 0.0;
    else if (iters >= (double)maxiter) status = 2.0;
  }
  if (status != 1.0) {
    for (int i = threadIdx.x; i < D; i += blockDim.x) p[i] = 0.0;
    if (threadIdx.x == 0) st[CG_STATUS] = status;
    return;
  }
  const double* z = Zin ? Zin + off : nullptr;
  double rho;
  if (z || minv) {
    double s = 0.0;
    for (int i = threadIdx.x; i < D; i += blockDim.x) s = fma(r[i], z ? z[i] : minv[i] * r[i], s);
    rho = block_sum_1024(s, red);
  } else {
    rho = st[CG_RNORM2];
  }
  const bool first = iters == 0.0;
  const double beta = first ? 0.0 : rho / st[CG_RHO_PREV];
  for (int i = threadIdx.x; i < D; i += blockDim.x) {
    const double zi = z ? z[i] : (minv ? minv[i] * r[i] : r[i]);
    p[i] = first ? zi : fma(beta, p[i], zi);
  }
  if (threadIdx.x == 0) { st[CG_RHO] = rho; st[CG_ITERS] = iters + 1.0; }
}

__global__ void __launch_bounds__(1024) cg_batch_update_xr_kernel(int D, const double* P, const double* Q, double* X,
                                                                  double* R, double* state) {
  __shared__ double red[32];
  const long off = (long)blockIdx.x * D;
  double* st = state + 8L * blockIdx.x;
  if (st[CG_STATUS] != 1.0) return;
  const double* p = P + off;
  const double* q = Q + off;
  double* x = X + off;
  double* r = R + off;
  double s = 0.0;
  for (int i = threadIdx.x; i < D; i += blockDim.x) s = fma(p[i], q[i], s);
  const double pq = block_sum_1024(s, red);
  const double rho = st[CG_RHO];
  const double alpha = rho / pq;
  double rr = 0.0;
  for (int i = threadIdx.x; i < D; i += blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    const double ri = fma(-alpha, q[i], r[i]);
    r[i] = ri;
    rr = fma(ri, ri, rr);
  }
  rr = block_sum_1024(rr, red);
  if (threadIdx.x == 0) { st[CG_RHO_PREV] = rho; st[CG_PQ] = pq; st[CG_RNORM2] = rr; }
}
}  // namespace

int cg_batch_init(int D, int K, const double* B, double* X, double* R, double* state, double rtol, double atol,
                  int keep_xr, cudaStream_t stream) {
  VT_REQUIRE(D >= 1 && K >= 1 && B && X && R && state, "cg_batch_init: bad arguments");
  cg_batch_init_kernel<<<K, 1024, 0, stream>>>(D, B, X, R, state, rtol, atol, keep_xr);
  VT_LAUNCH_CHECK();
  return VT_OK;
}
int cg_batch_update_p(int D, int K, const double* R, const double* Z, const double* minv, double* P, double* state,
                      int maxiter, cudaStream_t stream) {
  VT_REQUIRE(D >= 1 && K >= 1 && R && P && state && maxiter >= 0, "cg_batch_update_p: bad arguments");
  cg_batch_update_p_kernel<<<K, 1024, 0, stream>>>(D, R, Z, minv, P, state, maxiter);
  VT_LAUNCH_CHECK();
  return VT_OK;
}
int cg_batch_update_xr(int D, int K, const double* P, const double* Q, double* X, double* R, double* state,
                       cudaStream_t stream) {
  VT_REQUIRE(D >= 1 && K >= 1 && P && Q && X && R && state, "cg_batch_update_xr: bad arguments");
  cg_batch_update_xr_kernel<<<K, 1024, 0, stream>>>(D, P, Q, X, R, state);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

}  // namespace vt
