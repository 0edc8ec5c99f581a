// FP64 DMMA GEMM engine - see dgemm.cuh for the design notes.
#include "dgemm.cuh"
#include "grouploo.cuh"
#include <cstdlib>

namespace vt {

namespace {

struct Unit {
  int m0, n0;      // tile origin
  int kit0, nkit;  // k-iteration range of this unit
};

__device__ __forceinline__ void tile_coords(const GemmParams& p, int tile, int& tm, int& tn) {
  if (p.lower) {
    int i = (int)((sqrtf(8.f * (float)tile + 1.f) - 1.f) * 0.5f);
    while ((long)(i + 1) * (i + 2) / 2 <= tile) ++i;
    while ((long)i * (i + 1) / 2 > tile) --i;
    tm = i;
    tn = tile - i * (i + 1) / 2;
  } else {
    tm = tile % p.tiles_m;
    tn = tile / p.tiles_m;
  }
}

template <int TM>
__device__ __forceinline__ Unit decode_unit(const GemmParams& p, long u) {
  Unit r;
  const int tile = (int)(u % p.ntiles);
  const int part = (int)(u / p.ntiles);
  int tm, tn;
  tile_coords(p, tile, tm, tn);
  r.m0 = tm * TM;
  r.n0 = tn * TM;
  const int q = p.kiters / p.parts, rem = p.kiters % p.parts;
  r.kit0 = part * q + min(part, rem);
  r.nkit = q + (part < rem ? 1 : 0);
  return r;
}

// Kernel configuration: square CTA tile TM x TM (128: the throughput
// configuration; 64: twice the CTAs per SM and a quarter of the work per tile,
// for short-K / few-tile problems such as the Cholesky panels and for outputs
// that 128-wide tiles cover wastefully), the warp grid over it, whether the DMMA
// fragments are double buffered in registers, and the CTAs resident per SM.
template <int TM_, int WARPS_M_, int WARPS_N_, bool DBUF_, int CTAS_PER_SM_>
struct GemmCfg {
  static constexpr int TM = TM_;
  static constexpr int WARPS_M = WARPS_M_, WARPS_N = WARPS_N_;
  static constexpr int NTHREADS = WARPS_M_ * WARPS_N_ * 32;
  static constexpr int MT = TM_ / (WARPS_M_ * 8), NT = TM_ / (WARPS_N_ * 8);
  static constexpr int VC = (TM_ * BK / 2) / NTHREADS;   // 16-byte chunks per operand per thread per stage
  static constexpr bool DBUF = DBUF_;
  static constexpr int CTAS_PER_SM = CTAS_PER_SM_;
  static constexpr int LDKS = TM_ + 4;                   // = 4 (mod 16) for TM = 64, 128
  static constexpr int TILE_DOUBLES = TM_ * LDKC;        // >= BK * LDKS
  static constexpr int SMEM_BYTES = (2 * STAGES * TILE_DOUBLES + STAGES * BK) * 8;
};

// Copy one 16-byte chunk (VEC) or two 8-byte elements (!VEC: odd leading
// dimension or unaligned base) of an operand tile (TM rows x 16 k) into shared
// memory; `chunk` in [0, VC).  Straight-line and fully predicated (zero fill
// outside the matrix or when `live` is false) so that ptxas can interleave the
// copies with the DMMA stream: a runtime branch per chunk splits the hot loop
// into dozens of basic blocks and costs ~20% of the tensor pipe (r01 tuning).
template <int MODE, bool VEC, int NTHREADS, int TM>
__device__ __forceinline__ void issue_chunk(double* __restrict__ s, const double* __restrict__ gp, long ld, int r0,
                                            int R, int k0, int K, bool live, int tid, int chunk) {
  constexpr int LDKS = TM + 4;
  if (VEC) {
    const int c = tid + chunk * NTHREADS;
    int row, kc, sm_off;
    if (MODE == KC) { row = c >> 3; kc = (c & 7) * 2; sm_off = row * LDKC + kc; }
    else            { kc = c / (TM / 2); row = (c % (TM / 2)) * 2; sm_off = kc * LDKS + row; }
    const int gr = r0 + row, gk = k0 + kc;
    // contiguous direction: k for KC, row for KS
    const int left = (MODE == KC) ? (K - gk) : (R - gr);
    const bool other_ok = (MODE == KC) ? (gr < R) : (gk < K);
    const int bytes = (live && other_ok) ? min(max(left * 8, 0), 16) : 0;
    const long off = (MODE == KC) ? (long)gr * ld + gk : (long)gk * ld + gr;
    cp_async16(s + sm_off, bytes ? gp + off : gp, bytes);
  } else {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int e = tid + (2 * chunk + i) * NTHREADS;
      int row, kc, sm_off;
      if (MODE == KC) { row = e >> 4; kc = e & 15; sm_off = row * LDKC + kc; }
      else            { kc = e / TM; row = e % TM; sm_off = kc * LDKS + row; }
      const int gr = r0 + row, gk = k0 + kc;
      const bool ok = live && (gr < R) && (gk < K);
      const long off = (MODE == KC) ? (long)gr * ld + gk : (long)gk * ld + gr;
      cp_async8(s + sm_off, ok ? gp + off : gp, ok ? 8 : 0);
    }
  }
}

template <int AMODE, int BMODE, bool KSCALE, bool VEC, class CFG>
__global__ void __launch_bounds__(CFG::NTHREADS, CFG::CTAS_PER_SM) dgemm_kernel(const GemmParams p) {
  constexpr int MT = CFG::MT, NT = CFG::NT, NTHREADS = CFG::NTHREADS, VC = CFG::VC;
  constexpr int TM = CFG::TM, LDKS = CFG::LDKS, TILE_DOUBLES = CFG::TILE_DOUBLES;
  constexpr int WM = MT * 8, WN = NT * 8;
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;
  double* sB = smem + STAGES * TILE_DOUBLES;
  double* sS = smem + 2 * STAGES * TILE_DOUBLES;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, tig = lane & 3;
  const int wm0 = (warp / CFG::WARPS_N) * WM;
  const int wn0 = (warp % CFG::WARPS_N) * WN;

  // fragment base offsets inside a stage
  const int a_off = (AMODE == KC) ? (wm0 + g) * LDKC + tig : tig * LDKS + wm0 + g;
  const int b_off = (BMODE == KC) ? (wn0 + g) * LDKC + tig : tig * LDKS + wn0 + g;
  constexpr int A_MT = (AMODE == KC) ? 8 * LDKC : 8;
  constexpr int A_KK = (AMODE == KC) ? 4 : 4 * LDKS;
  constexpr int B_NT = (BMODE == KC) ? 8 * LDKC : 8;
  constexpr int B_KK = (BMODE == KC) ? 4 : 4 * LDKS;

  double acc[MT][NT][2];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const long total_units = (long)p.ntiles * p.parts;
  long lu = blockIdx.x;
  bool lvalid = lu < total_units;
  Unit lU = decode_unit<TM>(p, lvalid ? lu : 0);
  int lk = 0;
  long mu = lu;
  bool mvalid = lvalid;
  Unit mU = lU;
  int mk = 0;

  constexpr int KK = BK / 4;
  constexpr int SLOTS = 2 * VC;                      // copy slots per thread per stage: A chunks then B chunks
  constexpr int SPK = (SLOTS + KK - 2) / (KK - 1);   // slots per k4 step; the refill is spread over steps 0..KK-2
  // copy slots [first, last) of the refill of `stage` at the load cursor (straight-line, predicated)
  auto issue_slots = [&](int stage, int first, int last) {
    const int k0 = (lU.kit0 + lk) * BK;
#pragma unroll
    for (int sl = first; sl < last; ++sl) {
      if (sl < VC)
        issue_chunk<AMODE, VEC, NTHREADS, TM>(sA + stage * TILE_DOUBLES, p.A, p.lda, lU.m0, p.M, k0, p.K, lvalid, tid, sl);
      else if (sl < SLOTS)
        issue_chunk<BMODE, VEC, NTHREADS, TM>(sB + stage * TILE_DOUBLES, p.B, p.ldb, lU.n0, p.N, k0, p.K, lvalid, tid,
                                          sl - VC);
    }
  };
  // per-k scale vector of the stage, then close the cp.async group
  auto finish_refill = [&](int stage) {
    if (KSCALE && tid < BK) {
      const int k = (lU.kit0 + lk) * BK + tid;
      const bool ok = lvalid && k < p.K;
      cp_async8(sS + stage * BK + tid, ok ? p.kscale + k : p.kscale, ok ? 8 : 0);
    }
    cp_async_commit();
  };
  auto advance_load_cursor = [&]() {
    if (lvalid && ++lk == lU.nkit) {
      lk = 0;
      lu += gridDim.x;
      lvalid = lu < total_units;
      if (lvalid) lU = decode_unit<TM>(p, lu);
    }
  };

#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    issue_slots(s, 0, SLOTS);
    finish_refill(s);
    advance_load_cursor();
  }

  // Register (double) buffer for the DMMA fragments: the fragments of k4-step
  // kk+1 (or of the next stage's step 0) are loaded while the DMMAs of step kk
  // are in the tensor pipe.
  constexpr int NBUF = CFG::DBUF ? 2 : 1;
  double fa[NBUF][MT], fb[NBUF][NT], fs[NBUF];
  auto load_frags = [&](int buf, int stg, int kk) {
    const double* As = sA + stg * TILE_DOUBLES + a_off + kk * A_KK;
    const double* Bs = sB + stg * TILE_DOUBLES + b_off + kk * B_KK;
#pragma unroll
    for (int i = 0; i < MT; ++i) fa[buf][i] = As[i * A_MT];
#pragma unroll
    for (int j = 0; j < NT; ++j) fb[buf][j] = Bs[j * B_NT];
    if (KSCALE) fs[buf] = sS[stg * BK + kk * 4 + tig];
  };

  cp_async_wait<STAGES - 2>();
  __syncthreads();
  if (CFG::DBUF) load_frags(0, 0, 0);

  int stage = 0;
  while (mvalid) {
    const int refill_stage = (stage + STAGES - 1) % STAGES;
#pragma unroll
    for (int kk = 0; kk < KK; ++kk) {
      const int cur = CFG::DBUF ? (kk & 1) : 0, nxt = CFG::DBUF ? (cur ^ 1) : 0;
      if (!CFG::DBUF) load_frags(0, stage, kk);
      if (CFG::DBUF) {
        if (kk == KK - 1) {
          // the next stage must have landed (own copies) and be visible (barrier);
          // the barrier also certifies that every warp is done reading the stage
          // that the next iteration's refill will overwrite
          cp_async_wait<STAGES - 2>();
          __syncthreads();
          load_frags(nxt, (stage + 1) % STAGES, 0);
        } else {
          load_frags(nxt, stage, kk + 1);
        }
      }
      // refill of the stage consumed in the previous iteration, spread over
      // steps 0..KK-2 and placed after the fragment loads in program order
      if (kk < KK - 1) issue_slots(refill_stage, kk * SPK, (kk + 1) * SPK);
      if (kk == KK - 2) finish_refill(refill_stage);
      if (KSCALE) {
#pragma unroll
        for (int j = 0; j < NT; ++j) fb[cur][j] *= fs[cur];
      }
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[cur][i], fb[cur][j]);
    }
    if (!CFG::DBUF) {
      cp_async_wait<STAGES - 2>();
      __syncthreads();
    }
    advance_load_cursor();
    stage = (stage + 1) % STAGES;

    if (++mk == mU.nkit) {
      // ------------------------------------------------------ epilogue ----
      if (p.parts > 1) {
        double* ws = p.workspace + mu * (long)(TM * TM);
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
          for (int j = 0; j < NT; ++j) {
            const int r = wm0 + i * 8 + g, c = wn0 + j * 8 + 2 * tig;
            *reinterpret_cast<double2*>(ws + r * TM + c) = make_double2(acc[i][j][0], acc[i][j][1]);
          }
      } else {
        double cs[NT][2];
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          const int c = mU.n0 + wn0 + j * 8 + 2 * tig;
          cs[j][0] = (p.colscale && c < p.N) ? p.colscale[c] : 1.0;
          cs[j][1] = (p.colscale && c + 1 < p.N) ? p.colscale[c + 1] : 1.0;
        }
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          const int r = mU.m0 + wm0 + i * 8 + g;
          if (r < p.M) {
            const double rs = p.alpha * (p.rowscale ? p.rowscale[r] : 1.0);
#pragma unroll
            for (int j = 0; j < NT; ++j) {
              const int c = mU.n0 + wn0 + j * 8 + 2 * tig;
              if (c >= p.N) continue;
              double v0 = acc[i][j][0] * rs * cs[j][0];
              double v1 = acc[i][j][1] * rs * cs[j][1];
              double* cp = p.C + (long)r * p.ldc + c;
              const bool has1 = c + 1 < p.N;
              if (p.lower) {
                // keep only the lower triangle (exact symmetry comes from mirroring it)
                const bool k0 = r >= c, k1 = has1 && r >= c + 1;
                if (p.beta != 0.0) {
                  if (k0) v0 += p.beta * cp[0];
                  if (k1) v1 += p.beta * cp[1];
                }
                if (k0) cp[0] = v0;
                if (k1) cp[1] = v1;
                if (p.mirror) {
                  if (k0 && r != c) p.C[(long)c * p.ldc + r] = v0;
                  if (k1 && r != c + 1) p.C[(long)(c + 1) * p.ldc + r] = v1;
                }
              } else {
                if (p.beta != 0.0) {
                  v0 += p.beta * cp[0];
                  if (has1) v1 += p.beta * cp[1];
                }
                if (p.c_vec && has1) {
                  *reinterpret_cast<double2*>(cp) = make_double2(v0, v1);
                } else {
                  cp[0] = v0;
                  if (has1) cp[1] = v1;
                }
              }
            }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
      mk = 0;
      mu += gridDim.x;
      mvalid = mu < total_units;
      if (mvalid) mU = decode_unit<TM>(p, mu);
    }
  }
  cp_async_wait<0>();
}

// Sum split-K partials in a fixed order (bitwise reproducible) and apply the
// same scaling/beta/lower/mirror rules as the direct epilogue.
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const GemmParams p) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int T = p.tile;
  const long per_tile = (long)T * T;
  if (idx >= per_tile * p.ntiles) return;
  const int tile = (int)(idx / per_tile);
  const int e = (int)(idx % per_tile);
  int tm, tn;
  tile_coords(p, tile, tm, tn);
  const int r = tm * T + e / T, c = tn * T + e % T;
  if (r >= p.M || c >= p.N) return;
  if (p.lower && r < c) return;
  double s = 0.0;
  const double* ws = p.workspace + (long)tile * per_tile + e;
  for (int part = 0; part < p.parts; ++part) s += ws[(long)part * p.ntiles * per_tile];
  double v = s * p.alpha;
  if (p.rowscale) v *= p.rowscale[r];
  if (p.colscale) v *= p.colscale[c];
  double* cp = p.C + (long)r * p.ldc + c;
  if (p.beta != 0.0) v += p.beta * cp[0];
  cp[0] = v;
  if (p.lower && p.mirror && r != c) p.C[(long)c * p.ldc + r] = v;
}

template <int AMODE, int BMODE, bool KSCALE, bool VEC, class CFG>
int launch_cfg(const GemmParams& p, int grid, cudaStream_t stream) {
  // once per instantiation and device: the attribute call costs as much host time as the launch itself, and the
  // blocked Cholesky / triangular solves issue ~100 short GEMMs back to back
  static thread_local int configured_dev = -1;
  int dev = 0;
  VT_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    VT_CUDA(cudaFuncSetAttribute(dgemm_kernel<AMODE, BMODE, KSCALE, VEC, CFG>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, CFG::SMEM_BYTES));
    configured_dev = dev;
  }
  dgemm_kernel<AMODE, BMODE, KSCALE, VEC, CFG><<<grid, CFG::NTHREADS, CFG::SMEM_BYTES, stream>>>(p);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

using CfgBig = GemmCfg<TILE_BIG, 2, 4, true, 1>;
using CfgSmall = GemmCfg<TILE_SMALL, 2, 2, true, 2>;

int ctas_per_sm(int tile) { return tile == TILE_SMALL ? CfgSmall::CTAS_PER_SM : CfgBig::CTAS_PER_SM; }

template <int AMODE, int BMODE, bool KSCALE>
int launch_variant(const GemmParams& p, int grid, cudaStream_t stream) {
  const bool vec = p.a_vec && p.b_vec;
  if (p.tile == TILE_SMALL) {
    if (vec) return launch_cfg<AMODE, BMODE, KSCALE, true, CfgSmall>(p, grid, stream);
    return launch_cfg<AMODE, BMODE, KSCALE, false, CfgSmall>(p, grid, stream);
  }
  if (vec) return launch_cfg<AMODE, BMODE, KSCALE, true, CfgBig>(p, grid, stream);
  return launch_cfg<AMODE, BMODE, KSCALE, false, CfgBig>(p, grid, stream);
}

int count_tiles(int M, int N, int lower, int tile) {
  const int tm = (M + tile - 1) / tile, tn = (N + tile - 1) / tile;
  return lower ? tm * (tm + 1) / 2 : tm * tn;
}

}  // namespace

// 128-wide tiles are the throughput configuration (half the L2->smem traffic per
// flop).  64-wide tiles win when (a) the big tiles cannot occupy the machine
// even with split-K (short K: Cholesky panels, trailing updates, solve steps),
// or (b) they would execute >= 15% more flops than the small ones (ragged or
// narrow outputs, the diagonal tiles of a small SYRK).
int gemm_pick_tile(int M, int N, int K, int lower) {
  const int kiters = (K + BK - 1) / BK;
  const long nt_big = count_tiles(M, N, lower, TILE_BIG), nt_small = count_tiles(M, N, lower, TILE_SMALL);
  const long max_parts = kiters / 8 > 0 ? kiters / 8 : 1;
  if (nt_big * max_parts < num_sms()) return TILE_SMALL;
  const double exec_big = (double)nt_big * TILE_BIG * TILE_BIG, exec_small = (double)nt_small * TILE_SMALL * TILE_SMALL;
  return exec_big >= 1.15 * exec_small ? TILE_SMALL : TILE_BIG;
}

int gemm_pick_parts(int ntiles, int kiters, int tile, size_t workspace_bytes) {
  const int G = num_sms() * ctas_per_sm(tile);
  if (ntiles >= 4 * G) return 1;
  long pmax = kiters / 8;                                  // at least 8 k-iterations per unit
  const long by_ws = (long)(workspace_bytes / ((size_t)ntiles * tile * tile * 8));
  if (by_ws < pmax) pmax = by_ws;
  if (pmax > 4L * G) pmax = 4L * G;
  if (pmax < 2) return 1;
  int best = 1;
  double best_eff = 0.0;
  for (int P = 1; P <= pmax; ++P) {
    const long U = (long)ntiles * P;
    const double eff = (double)U / ((double)G * (double)((U + G - 1) / G));
    if (eff > best_eff + 1e-9) { best_eff = eff; best = P; }
    if (eff >= 0.985) break;
  }
  return best;
}

int gemm_ctas_per_sm(int tile) { return ctas_per_sm(tile); }

size_t gemm_workspace_bytes(int M, int N, int K, int lower, int tile) {
  if (tile == 0) tile = gemm_pick_tile(M, N, K, lower);
  const int ntiles = count_tiles(M, N, lower, tile);
  const int kiters = (K + BK - 1) / BK;
  const int P = gemm_pick_parts(ntiles, kiters, tile, (size_t)1 << 62);
  return P > 1 ? (size_t)ntiles * P * tile * tile * 8 : 0;
}

int gemm_launch(GemmParams p, cudaStream_t stream) {
  VT_REQUIRE(p.M >= 0 && p.N >= 0 && p.K >= 0, "gemm: negative dimension");
  if (p.M == 0 || p.N == 0) return VT_OK;
  VT_REQUIRE(p.A && p.B && p.C, "gemm: null operand");
  VT_REQUIRE(p.K > 0, "gemm: K must be positive");
  VT_REQUIRE(p.tile == 0 || p.tile == TILE_BIG || p.tile == TILE_SMALL, "gemm: tile must be 0, %d or %d", TILE_BIG,
             TILE_SMALL);
  if (p.lower) VT_REQUIRE(p.M == p.N, "gemm: lower-only output must be square");
  if (p.tile == 0) p.tile = gemm_pick_tile(p.M, p.N, p.K, p.lower);
  p.tiles_m = (p.M + p.tile - 1) / p.tile;
  p.tiles_n = (p.N + p.tile - 1) / p.tile;
  p.ntiles = p.lower ? p.tiles_m * (p.tiles_m + 1) / 2 : p.tiles_m * p.tiles_n;
  p.kiters = (p.K + BK - 1) / BK;
  p.a_vec = (p.lda % 2 == 0) && (reinterpret_cast<uintptr_t>(p.A) % 16 == 0);
  p.b_vec = (p.ldb % 2 == 0) && (reinterpret_cast<uintptr_t>(p.B) % 16 == 0);
  p.c_vec = (p.ldc % 2 == 0) && (reinterpret_cast<uintptr_t>(p.C) % 16 == 0);
  if (p.parts <= 0) p.parts = (p.workspace ? gemm_pick_parts(p.ntiles, p.kiters, p.tile, p.workspace_bytes) : 1);
  if (p.parts > p.kiters) p.parts = p.kiters;
  if (p.parts > 1)
    VT_REQUIRE(p.workspace && p.workspace_bytes >= (size_t)p.ntiles * p.parts * p.tile * p.tile * 8,
               "gemm: split-K workspace too small (%zu bytes for %d parts x %d tiles)", p.workspace_bytes,
               p.parts, p.ntiles);
  if (p.parts > 1)
    VT_REQUIRE(reinterpret_cast<uintptr_t>(p.workspace) % 16 == 0, "gemm: the split-K workspace must be 16-byte aligned");
  const long units = (long)p.ntiles * p.parts;
  const long slots = (long)num_sms() * ctas_per_sm(p.tile);
  long cap = slots - (long)p.spare_sms * ctas_per_sm(p.tile);
  if (cap < ctas_per_sm(p.tile)) cap = ctas_per_sm(p.tile);
  const int grid = (int)(units < cap ? units : cap);
  int st;
  if (p.kscale) {
    VT_REQUIRE(p.amode == KS && p.bmode == KS, "gemm: kscale is only implemented for KS x KS operands");
    st = launch_variant<KS, KS, true>(p, grid, stream);
  } else if (p.amode == KC && p.bmode == KC) {
    st = launch_variant<KC, KC, false>(p, grid, stream);
  } else if (p.amode == KC && p.bmode == KS) {
    st = launch_variant<KC, KS, false>(p, grid, stream);
  } else if (p.amode == KS && p.bmode == KC) {
    st = launch_variant<KS, KC, false>(p, grid, stream);
  } else {
    st = launch_variant<KS, KS, false>(p, grid, stream);
  }
  if (st != VT_OK) return st;
  if (p.parts > 1) {
    const long total = (long)p.ntiles * p.tile * p.tile;
    splitk_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

// ---- out[n] = |Linv x_n|^2 on the DMMA engine -------------------------------
namespace {
constexpr size_t QF_CHUNK_BYTES = (size_t)256 << 20;          // U of one chunk of rows

long quad_forms_chunk_rows(long N, int D) {
  long rows = (long)(QF_CHUNK_BYTES / ((size_t)D * 8));
  if (rows < 1) rows = 1;
  if (rows > 2147483647L) rows = 2147483647L;
  return rows < N ? rows : N;
}

// out[r] = sum_i U[r][i]^2: a warp per row, lane-strided partial sums and a fixed shuffle tree.
__global__ void __launch_bounds__(256) row_sumsq_kernel(const double* __restrict__ U, long ldu, long rows, int D,
                                                        double* __restrict__ out) {
  const long r = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const double* u = U + r * ldu;
  double acc = 0.0;
  for (int i = lane; i < D; i += 32) acc = fma(u[i], u[i], acc);
  acc = warp_sum(acc);
  if (lane == 0) out[r] = acc;
}
}  // namespace

size_t quad_forms_workspace_bytes(long N, int D) {
  return N > 0 && D > 0 ? (size_t)quad_forms_chunk_rows(N, D) * D * 8 : 0;
}

int quad_forms(const double* Linv, long ldl, const double* X, long ldx, long N, int D, double* out, void* workspace,
               size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Linv && X && out, "quad_forms: null pointer");
  VT_REQUIRE(D >= 1 && N >= 0 && ldl >= D && ldx >= D, "quad_forms: bad shape");
  if (N == 0) return VT_OK;
  VT_REQUIRE(workspace && workspace_bytes >= quad_forms_workspace_bytes(N, D), "quad_forms: workspace too small");
  const long ch = quad_forms_chunk_rows(N, D);
  double* U = static_cast<double*>(workspace);
  for (long r0 = 0; r0 < N; r0 += ch) {
    const long rows = (N - r0 < ch) ? N - r0 : ch;
    GemmParams p{};                                              // U = X_c Linv^T  (rows x D)
    p.M = (int)rows; p.N = D; p.K = D;
    p.A = X + r0 * ldx; p.lda = ldx; p.amode = KC;
    p.B = Linv; p.ldb = ldl; p.bmode = KC;
    p.C = U; p.ldc = D;
    p.alpha = 1.0; p.beta = 0.0;
    p.parts = 1;
    int st = gemm_launch(p, stream);
    if (st != VT_OK) return st;
    row_sumsq_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, stream>>>(U, D, rows, D, out + r0);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

// ---- leave-one-group-out on the DMMA engine ----------------------------------
size_t group_loo_workspace_bytes(long N, int D) { return quad_forms_workspace_bytes(N, D); }

int group_loo(const double* Linv, long ldl, const double* X, long ldx, long N, int D, const int64_t* starts, long G,
              const double* s, const double* u, const double* z, int method, double* zpred, double* h, void* workspace,
              size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Linv && X && starts && s && u && z && zpred && h, "group_loo: null pointer");
  VT_REQUIRE(D >= 1 && N >= 0 && G >= 0 && G <= N && ldl >= D && ldx >= D, "group_loo: bad shape");
  VT_REQUIRE(method == GROUP_LOO_IJ || method == GROUP_LOO_NS, "group_loo: method 0 (IJ) or 1 (Newton step)");
  if (N == 0) return VT_OK;
  VT_REQUIRE(workspace && workspace_bytes >= group_loo_workspace_bytes(N, D), "group_loo: workspace too small");
  const long ch = quad_forms_chunk_rows(N, D);
  VT_REQUIRE(ch == N || ch > GROUP_LOO_OVERLAP, "group_loo: D = %d leaves no room for whole groups in a chunk", D);
  const long stride = ch - GROUP_LOO_OVERLAP;
  double* U = static_cast<double*>(workspace);
  for (long r0 = 0;; r0 += stride) {
    const long rows = (N - r0 < ch) ? N - r0 : ch;
    const bool last = r0 + ch >= N;
    GemmParams p{};                                              // U = X_c Linv^T  (rows x D)
    p.M = (int)rows; p.N = D; p.K = D;
    p.A = X + r0 * ldx; p.lda = ldx; p.amode = KC;
    p.B = Linv; p.ldb = ldl; p.bmode = KC;
    p.C = U; p.ldc = D;
    p.alpha = 1.0; p.beta = 0.0;
    p.parts = 1;
    int st = gemm_launch(p, stream);
    if (st != VT_OK) return st;
    st = group_loo_chunk(GroupLooChunk{U, D, 1, r0, rows, D, starts, G, r0, last ? N : r0 + stride, s, u, z, method,
                                       zpred, h}, stream);
    if (st != VT_OK) return st;
    if (last) break;
  }
  return VT_OK;
}

}  // namespace vt
