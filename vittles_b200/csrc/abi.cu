// extern "C" entry points declared in include/vittles_b200.h.
#include "../../include/vittles_b200.h"
#include "blockchol.cuh"
#include "chol.cuh"
#include "common.cuh"
#include "dgemm.cuh"
#include "glm.cuh"
#include "synth.cuh"
#include "tgemm.cuh"
#include "ogemm.cuh"

namespace vt {
const char* last_error();

namespace {
__global__ void add_diag_kernel(double* H, long ldh, int D, double v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < D) H[(long)i * ldh + i] += v;
}

// Register-resident DMMA loop (same kernel as tools/fp64_peak.cu, variant
// dmma884_t16): 16 independent accumulator tiles per warp, 2 warps per SMSP.
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, double a, double b, int iters) {
  double c[16][2];
#pragma unroll
  for (int i = 0; i < 16; ++i) { c[i][0] = threadIdx.x; c[i][1] = i; }
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) dmma884(c[i][0], c[i][1], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += c[i][0] + c[i][1];
  if (s == 12345.678) out[0] = s;
}
}  // namespace
}  // namespace vt

using namespace vt;

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

const char* vt_last_error(void) { return vt::last_error(); }
int vt_abi_version(void) { return 2; }
int64_t vt_launch_count(void) { return (int64_t)vt::launch_count(); }

int vt_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  VT_CUDA(cudaGetDevice(&dev));
  if (sm_count) VT_CUDA(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev));
  if (cc_major) VT_CUDA(cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev));
  if (cc_minor) VT_CUDA(cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
  return VT_OK;
}

int vt_fp64_peak_probe(double seconds, double* tflops, void* stream) {
  VT_REQUIRE(tflops && seconds > 0, "fp64_peak_probe: bad arguments");
  double* out = nullptr;
  VT_CUDA(cudaMalloc(&out, 8));   // the one allocation in the library: 8 bytes, freed below
  cudaEvent_t e0, e1;
  VT_CUDA(cudaEventCreate(&e0));
  VT_CUDA(cudaEventCreate(&e1));
  const int grid = num_sms(), iters0 = 1 << 14;
  auto run = [&](int iters, float* ms) -> int {
    VT_CUDA(cudaEventRecord(e0, S(stream)));
    dmma_peak_kernel<<<grid, 256, 0, S(stream)>>>(out, 1.0000001, 1e-9, iters);
    VT_LAUNCH_CHECK();
    VT_CUDA(cudaEventRecord(e1, S(stream)));
    VT_CUDA(cudaEventSynchronize(e1));
    VT_CUDA(cudaEventElapsedTime(ms, e0, e1));
    return VT_OK;
  };
  float ms = 0.f;
  int st = run(iters0, &ms);          // warm-up + calibration
  if (st == VT_OK) st = run(iters0, &ms);
  if (st == VT_OK) {
    double want = seconds * 1e3 / (ms > 1e-3f ? ms : 1e-3f) * iters0;
    int iters = want > 2e9 ? 2000000000 : (int)want;
    if (iters < iters0) iters = iters0;
    st = run(iters, &ms);
    if (st == VT_OK) *tflops = 512.0 * 16.0 * 8.0 * (double)grid * (double)iters / (ms * 1e-3) / 1e12;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  return st;
}

int vt_i8_peak_probe(double seconds, int n_tile, double* tops, double* clocks_per_mma, void* stream) {
  return i8_peak_probe(seconds, n_tile, tops, clocks_per_mma, S(stream));
}

size_t vt_dgemm_workspace_bytes(int M, int N, int K, int lower, int tile) {
  return gemm_workspace_bytes(M, N, K, lower, tile);
}

int vt_dgemm(int M, int N, int K, double alpha, const double* A, int64_t lda, int amode, const double* B,
             int64_t ldb, int bmode, double beta, double* C, int64_t ldc, const double* kscale,
             const double* colscale, const double* rowscale, int lower, int mirror, int tile, void* workspace,
             size_t workspace_bytes, void* stream) {
  VT_REQUIRE((amode == KC || amode == KS) && (bmode == KC || bmode == KS), "dgemm: bad operand mode");
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.A = A; p.lda = lda; p.amode = amode;
  p.B = B; p.ldb = ldb; p.bmode = bmode;
  p.C = C; p.ldc = ldc;
  p.alpha = alpha; p.beta = beta;
  p.kscale = kscale; p.colscale = colscale; p.rowscale = rowscale;
  p.lower = lower; p.mirror = mirror;
  p.parts = 0;
  p.tile = tile;
  p.workspace = static_cast<double*>(workspace);
  p.workspace_bytes = workspace_bytes;
  return gemm_launch(p, S(stream));
}

size_t vt_syrk_workspace_bytes(int64_t N, int D) {
  return gemm_workspace_bytes(D, D, (int)(N > 2147483647LL ? 2147483647LL : N), 1, 0);
}

int vt_syrk_weighted(const double* X, int64_t ldx, int64_t N, int D, const double* s, double l2, double* H,
                     int64_t ldh, void* workspace, size_t workspace_bytes, void* stream) {
  VT_REQUIRE(X && H, "syrk_weighted: null pointer");
  VT_REQUIRE(N >= 1 && N <= 2147483647LL && D >= 1 && ldx >= D && ldh >= D, "syrk_weighted: bad shape");
  GemmParams p{};
  p.M = D; p.N = D; p.K = (int)N;
  p.A = X; p.lda = ldx; p.amode = KS;
  p.B = X; p.ldb = ldx; p.bmode = KS;
  p.C = H; p.ldc = ldh;
  p.alpha = 1.0; p.beta = 0.0;
  p.kscale = s;
  p.lower = 1; p.mirror = 1;
  p.parts = 0;
  p.workspace = static_cast<double*>(workspace);
  p.workspace_bytes = workspace_bytes;
  int st = gemm_launch(p, S(stream));
  if (st != VT_OK) return st;
  if (l2 != 0.0) {
    add_diag_kernel<<<(D + 255) / 256, 256, 0, S(stream)>>>(H, ldh, D, l2);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

size_t vt_glm_workspace_bytes(int D) { return glm_workspace_bytes(D); }

int vt_glm_stats(const double* X, int64_t ldx, int64_t N, int D, const double* theta, const double* y,
                 const double* w, int family, double* z, double* resid, double* s, double* grad, double l2,
                 void* workspace, size_t workspace_bytes, void* stream) {
  return glm_stats(X, ldx, N, D, theta, y, w, family, z, resid, s, grad, l2, nullptr, nullptr,
                   static_cast<double*>(workspace), workspace_bytes, S(stream));
}
int vt_glm_stats_colmax(const double* X, int64_t ldx, int64_t N, int D, const double* theta, const double* y,
                        const double* w, int family, double* z, double* resid, double* s, double* grad, double l2,
                        double* sq, uint64_t* colmax, void* workspace, size_t workspace_bytes, void* stream) {
  VT_REQUIRE(sq && colmax, "glm_stats_colmax: sq and colmax are required");
  return glm_stats(X, ldx, N, D, theta, y, w, family, z, resid, s, grad, l2, sq,
                   reinterpret_cast<unsigned long long*>(colmax), static_cast<double*>(workspace), workspace_bytes,
                   S(stream));
}

size_t vt_glm_hvp_multi_workspace_bytes(int D, int q) { return glm_hvp_multi_workspace_bytes(D, q); }
int vt_glm_hvp_multi(const double* X, int64_t ldx, int64_t N, int D, const double* s, const double* V, int q,
                     double ridge, double* out, void* workspace, size_t workspace_bytes, void* stream) {
  return glm_hvp_multi(X, ldx, N, D, s, V, q, ridge, out, static_cast<double*>(workspace), workspace_bytes, S(stream));
}
int vt_glm_hvp(const double* X, int64_t ldx, int64_t N, int D, const double* s, const double* v, double ridge,
               double* out, void* workspace, size_t workspace_bytes, void* stream) {
  return glm_hvp(X, ldx, N, D, s, v, ridge, out, static_cast<double*>(workspace), workspace_bytes, S(stream));
}

int vt_glm_influence_max_directions(int D) { return glm_influence_max_directions(D); }
int vt_glm_influence(const double* X, int64_t ldx, int64_t N, int D, const double* c, const double* V, int K,
                     double alpha, double* out, int64_t ldo, void* stream) {
  return glm_influence(X, ldx, N, D, c, V, K, alpha, out, ldo, S(stream));
}

size_t vt_glm_dirderiv_workspace_bytes(int64_t N, int D) { return glm_dirderiv_workspace_bytes(N, D); }

int vt_glm_dirderiv(const double* X, int64_t ldx, int64_t N, int D, const double* z, const double* w, int family,
                    const double* dirs, int q, double* out, void* workspace, size_t workspace_bytes, void* stream) {
  return glm_dirderiv(X, ldx, N, D, z, w, family, dirs, q, out, static_cast<double*>(workspace), workspace_bytes,
                      S(stream));
}

size_t vt_potrf_dinv_doubles(int D) { return chol_dinv_doubles(D); }

int vt_potrf(double* A, int64_t lda, int D, double* dinv, int32_t* info, void* stream) {
  return chol_potrf(A, lda, D, dinv, info, S(stream));
}

int vt_potrs(const double* L, int64_t ldl, int D, const double* dinv, double* B, int64_t ldb, int K, void* stream) {
  return chol_potrs(L, ldl, D, dinv, B, ldb, K, S(stream));
}

int vt_trsm_lower(const double* L, int64_t ldl, int D, const double* dinv, double* B, int64_t ldb, int K, int transpose,
                  void* stream) {
  return chol_trsm_lower(L, ldl, D, dinv, B, ldb, K, transpose, S(stream));
}

size_t vt_quad_forms_workspace_bytes(int64_t N, int D) { return quad_forms_workspace_bytes(N, D); }

int vt_quad_forms(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D, double* out,
                  void* workspace, size_t workspace_bytes, void* stream) {
  return quad_forms(Linv, ldl, X, ldx, N, D, out, workspace, workspace_bytes, S(stream));
}

int vt_ij_apply(const double* Hinv, int64_t ldh, const double* X, int64_t ldx, int64_t N, int D,
                const double* resid, double* Sout, int64_t lds, void* stream) {
  VT_REQUIRE(Hinv && X && resid && Sout, "ij_apply: null pointer");
  VT_REQUIRE(N >= 1 && N <= 2147483647LL && D >= 1 && ldh >= D && ldx >= D && lds >= N, "ij_apply: bad shape");
  GemmParams p{};
  p.M = D; p.N = (int)N; p.K = D;
  p.A = Hinv; p.lda = ldh; p.amode = KC;
  p.B = X; p.ldb = ldx; p.bmode = KC;
  p.C = Sout; p.ldc = lds;
  p.alpha = -1.0; p.beta = 0.0;
  p.colscale = resid;
  p.parts = 1;
  return gemm_launch(p, S(stream));
}

size_t vt_tf32_gemm_workspace_bytes(int M, int N, int64_t K, int split) { return tgemm_workspace_bytes(M, N, K, split); }

int vt_tf32_convert(const double* X, int64_t ldx, int64_t rows, int cols, const double* rowscale, int sqrt_scale,
                    float* hi, float* lo, int64_t ldo, void* stream) {
  return tf32_convert(X, ldx, rows, cols, rowscale, sqrt_scale, hi, lo, ldo, S(stream));
}

int vt_tf32_gemm(int M, int N, int64_t K, double alpha, const float* A_hi, const float* A_lo, int64_t lda, int amode,
                 const float* B_hi, const float* B_lo, int64_t ldb, int bmode, double* C, int64_t ldc,
                 const double* colscale, const double* rowscale, void* workspace, size_t workspace_bytes,
                 void* stream) {
  VT_REQUIRE((amode == KC || amode == KS) && (bmode == KC || bmode == KS), "tf32_gemm: bad operand mode");
  TGemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.A_hi = A_hi; p.A_lo = A_lo; p.lda = lda; p.amode = amode;
  p.B_hi = B_hi; p.B_lo = B_lo; p.ldb = ldb; p.bmode = bmode;
  p.C = C; p.ldc = ldc;
  p.alpha = alpha;
  p.colscale = colscale; p.rowscale = rowscale;
  p.parts = 0;
  p.workspace = static_cast<double*>(workspace);
  p.workspace_bytes = workspace_bytes;
  return tgemm_launch(p, S(stream));
}

size_t vt_ij_apply_tf32_workspace_bytes(int64_t N, int D, int split) { return ij_apply_tf32_workspace_bytes(N, D, split); }

int vt_ij_apply_tf32(const double* Hinv, int64_t ldh, const double* X, int64_t ldx, int64_t N, int D,
                     const double* resid, double* Sout, int64_t lds, int split, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return ij_apply_tf32(Hinv, ldh, X, ldx, N, D, resid, Sout, lds, split, workspace, workspace_bytes, S(stream));
}

size_t vt_syrk_tf32_workspace_bytes(int64_t N, int D, int split) { return syrk_tf32_workspace_bytes(N, D, split); }

int vt_syrk_tf32(const double* X, int64_t ldx, int64_t N, int D, const double* s, double l2, double* H, int64_t ldh,
                 int split, void* workspace, size_t workspace_bytes, void* stream) {
  int st = syrk_tf32(X, ldx, N, D, s, H, ldh, split, workspace, workspace_bytes, S(stream));
  if (st != VT_OK) return st;
  if (l2 != 0.0) {
    add_diag_kernel<<<(D + 255) / 256, 256, 0, S(stream)>>>(H, ldh, D, l2);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

int vt_ozaki_slice(const double* X, int64_t ldx, int64_t rows, int cols, int8_t* out, int64_t ldo, int64_t slice_stride,
                   int nslices, double* scale_out, const double* fold, void* stream) {
  return ozaki_slice(X, ldx, rows, cols, out, ldo, slice_stride, nslices, scale_out, fold, S(stream));
}

int vt_ozaki_slice_t(const double* X, int64_t ldx, int64_t rows, int cols, const double* sq, const uint64_t* colmax,
                     int8_t* out, int64_t ldo, int64_t slice_stride, int nslices, double* scale_out, void* stream) {
  return ozaki_slice_t(X, ldx, rows, cols, sq, reinterpret_cast<const unsigned long long*>(colmax), out, ldo, slice_stride,
                       nslices, scale_out, S(stream));
}

int vt_ozaki_gemm(int M, int N, int K, const int8_t* A, int64_t lda, int64_t a_slice_stride, const int8_t* B,
                  int64_t ldb, int64_t b_slice_stride, int nslices, double alpha, const double* rowscale,
                  const double* colscale, double* C, int64_t ldc, void* stream) {
  return ogemm_launch(M, N, K, A, lda, a_slice_stride, B, ldb, b_slice_stride, nslices, alpha, rowscale, colscale, C, ldc,
                      S(stream));
}

size_t vt_ij_apply_ozaki_workspace_bytes(int64_t N, int D, int nslices) {
  return ij_apply_ozaki_workspace_bytes(N, D, nslices);
}

int vt_ij_apply_ozaki(const double* Hinv, int64_t ldh, const double* X, int64_t ldx, int64_t N, int D,
                      const double* resid, double* Sout, int64_t lds, int nslices, void* workspace,
                      size_t workspace_bytes, void* stream) {
  return ij_apply_ozaki(Hinv, ldh, X, ldx, N, D, resid, Sout, lds, nslices, workspace, workspace_bytes, S(stream));
}

size_t vt_quad_forms_ozaki_workspace_bytes(int64_t N, int D, int nslices) {
  return quad_forms_ozaki_workspace_bytes(N, D, nslices);
}

int vt_quad_forms_ozaki(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D, double* out,
                        int nslices, void* workspace, size_t workspace_bytes, void* stream) {
  return quad_forms_ozaki(Linv, ldl, X, ldx, N, D, out, nslices, workspace, workspace_bytes, S(stream));
}

size_t vt_group_loo_workspace_bytes(int64_t N, int D) { return group_loo_workspace_bytes(N, D); }

int vt_group_loo(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D,
                 const int64_t* starts, int64_t G, const double* s, const double* u, const double* z, int method,
                 double* zpred, double* h, void* workspace, size_t workspace_bytes, void* stream) {
  return group_loo(Linv, ldl, X, ldx, N, D, starts, G, s, u, z, method, zpred, h, workspace, workspace_bytes,
                   S(stream));
}

size_t vt_group_loo_ozaki_workspace_bytes(int64_t N, int D, int nslices) {
  return group_loo_ozaki_workspace_bytes(N, D, nslices);
}

int vt_group_loo_ozaki(const double* Linv, int64_t ldl, const double* X, int64_t ldx, int64_t N, int D,
                       const int64_t* starts, int64_t G, const double* s, const double* u, const double* z, int method,
                       double* zpred, double* h, int nslices, void* workspace, size_t workspace_bytes, void* stream) {
  return group_loo_ozaki(Linv, ldl, X, ldx, N, D, starts, G, s, u, z, method, zpred, h, nslices, workspace,
                         workspace_bytes, S(stream));
}

size_t vt_syrk_ozaki_workspace_bytes(int64_t N, int D, int nslices) { return syrk_ozaki_workspace_bytes(N, D, nslices); }

int vt_syrk_ozaki(const double* X, int64_t ldx, int64_t N, int D, const double* s, double l2, double* H, int64_t ldh,
                  int nslices, const double* sq, const uint64_t* colmax, void* workspace, size_t workspace_bytes,
                  void* stream) {
  int st = syrk_ozaki(X, ldx, N, D, s, H, ldh, nslices, sq, reinterpret_cast<const unsigned long long*>(colmax),
                      workspace, workspace_bytes, S(stream));
  if (st != VT_OK) return st;
  if (l2 != 0.0) {
    add_diag_kernel<<<(D + 255) / 256, 256, 0, S(stream)>>>(H, ldh, D, l2);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

size_t vt_gemv_workspace_bytes(int M, int64_t N) { return gemv_workspace_bytes(M, N); }

int vt_gemv(const double* A, int64_t lda, int M, int64_t N, const double* x, double alpha, const double* y0,
            double beta, double* y, void* workspace, size_t workspace_bytes, void* stream) {
  return gemv_rows(A, lda, M, N, x, alpha, y0, beta, y, static_cast<double*>(workspace), workspace_bytes, S(stream));
}

int vt_cg_batch_init(int D, int K, const double* B, double* X, double* R, double* state, double rtol, double atol,
                     int keep_xr, void* stream) {
  return cg_batch_init(D, K, B, X, R, state, rtol, atol, keep_xr, S(stream));
}
int vt_cg_batch_update_p(int D, int K, const double* R, const double* Z, const double* minv, double* P, double* state,
                         int maxiter, void* stream) {
  return cg_batch_update_p(D, K, R, Z, minv, P, state, maxiter, S(stream));
}
int vt_cg_batch_update_xr(int D, int K, const double* P, const double* Q, double* X, double* R, double* state,
                          void* stream) {
  return cg_batch_update_xr(D, K, P, Q, X, R, state, S(stream));
}

int vt_block_potrf_batched(double* blocks, int64_t G, int M, int32_t* info, void* stream) {
  return block_potrf(blocks, G, M, info, S(stream));
}
int vt_block_trsm_batched(const double* Lb, double* C, int64_t G, int M, int Dg, void* stream) {
  return block_trsm(Lb, C, G, M, Dg, 0, S(stream));
}
int vt_block_trsmt_batched(const double* Lb, double* C, int64_t G, int M, int Dg, void* stream) {
  return block_trsm(Lb, C, G, M, Dg, 1, S(stream));
}
int vt_block_solve_batched(const double* Lb, double* b, int64_t G, int M, int mode, void* stream) {
  return block_solve(Lb, b, G, M, mode, S(stream));
}
int vt_tall_gemv(const double* Z, int64_t R, int Dg, const double* x, double alpha, double* y, double beta,
                 void* stream) {
  return tall_gemv(Z, R, Dg, x, alpha, y, beta, S(stream));
}
size_t vt_tall_colsum_workspace_bytes(int Dg) { return tall_colsum_workspace_bytes(Dg); }
int vt_tall_colsum(const double* Z, int64_t R, int Dg, const double* u, double alpha, const double* y0, double beta,
                   double* out, void* workspace, size_t workspace_bytes, void* stream) {
  return tall_colsum(Z, R, Dg, u, alpha, y0, beta, out, static_cast<double*>(workspace), workspace_bytes, S(stream));
}
int vt_gmm_blocks(const double* X, int64_t N, int d, int K, const double* m, const double* rho,
                  const double* log_pi, double* blocks, double* cross, double* rmat, double* grad_rho,
                  double* obj_terms, void* stream) {
  return gmm_blocks(X, N, d, K, m, rho, log_pi, blocks, cross, rmat, grad_rho, obj_terms, S(stream));
}

int vt_synth_design(double* X, int64_t ldx, int64_t row0, int64_t nrows, int ncols, uint64_t seed, double scale,
                    void* stream) {
  return synth_design(X, ldx, row0, nrows, ncols, seed, scale, S(stream));
}
int vt_synth_uniform(double* u, int64_t row0, int64_t nrows, uint64_t seed, void* stream) {
  return synth_uniform(u, row0, nrows, seed, S(stream));
}
int vt_synth_bernoulli(double* y, const double* z, int64_t row0, int64_t nrows, uint64_t seed, void* stream) {
  return synth_bernoulli(y, z, row0, nrows, seed, S(stream));
}

}  // extern "C"
