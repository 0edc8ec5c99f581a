// TF32 GEMM engine on tcgen05 / TMEM / TMA - see tgemm.cuh for the design notes.
#include "tgemm.cuh"
#include "tc05.cuh"

namespace vt {

using namespace tc05;

namespace {

enum : int { T_KC = 0, T_KS = 1 };

constexpr int TBM = 128;               // CTA / UMMA tile rows (TMEM lanes)
constexpr int TBK = 32;                // fp32 elements per k-block: 128 bytes = one swizzle row
constexpr int UMMA_K = 8;              // k per tcgen05.mma.kind::tf32
constexpr int SEG_KBLOCKS = 128;       // at most 4096 k per FP32 accumulation segment (then flushed to FP64)
constexpr int T_THREADS = 192;         // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue

template <int BN_, int NSPLIT_>
struct TCfg {
  static constexpr int BN = BN_;
  static constexpr int NSPLIT = NSPLIT_;                      // 1: TF32, 3: TF32x3 (hi/lo operands)
  static constexpr int NOPS = NSPLIT_ == 1 ? 1 : 2;           // arrays per operand (hi [, lo])
  static constexpr int A_BYTES = TBM * TBK * 4;               // 16 KB
  static constexpr int B_BYTES = BN_ * TBK * 4;               // 32 KB (BN = 256) / 16 KB (BN = 128)
  static constexpr int STAGE_BYTES = NOPS * (A_BYTES + B_BYTES);
  static constexpr int STAGES = (196608 / STAGE_BYTES) < 6 ? (196608 / STAGE_BYTES) : 6;
  static constexpr int TMEM_COLS = 2 * BN_;                   // double-buffered accumulator
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
};

struct TKernelArgs {
  int M, N;
  int kblocks;             // ceil(K / TBK)
  int tiles_m, tiles_n, ntiles, parts, lower;
  long units;
  double* C; long ldc;
  double alpha;
  const double* colscale;
  const double* rowscale;
  double* ws;              // nullptr: scale and store to C; else raw FP64 partial tiles [unit][TBM][BN]
  int ws_add_first;        // ws mode: the first segment adds to the workspace instead of overwriting it
  int c_vec;               // C rows are 32-byte aligned (ldc % 4 == 0, base aligned)
};

// -------------------------------------------------------------- schedule ----
// Tiles are TBM x BN.  lower: only tiles that intersect the lower triangle of a
// square output (row block tm keeps column blocks 0 .. (tm*TBM + TBM-1) / BN).
__host__ __device__ inline int lower_cols(int tm, int tiles_n, int BN) {
  const int c = (tm * TBM + TBM - 1) / BN + 1;
  return c < tiles_n ? c : tiles_n;
}
__device__ __forceinline__ void decode_tile(const TKernelArgs& a, int BN, int tile, int& tm, int& tn) {
  if (!a.lower) {
    tm = tile % a.tiles_m;       // row blocks fastest: CTAs that run together share the B (column) panel in L2
    tn = tile / a.tiles_m;
  } else {
    int t = tile;
    for (tm = 0; tm < a.tiles_m - 1; ++tm) {
      const int c = lower_cols(tm, a.tiles_n, BN);
      if (t < c) break;
      t -= c;
    }
    tn = t;
  }
}
struct TUnit {
  int m0, n0, kb0, nkb, nseg;
};
__device__ __forceinline__ TUnit decode_unit(const TKernelArgs& a, int BN, long u) {
  TUnit r;
  const int tile = (int)(u % a.ntiles), part = (int)(u / a.ntiles);
  int tm, tn;
  decode_tile(a, BN, tile, tm, tn);
  r.m0 = tm * TBM;
  r.n0 = tn * BN;
  const int q = a.kblocks / a.parts, rem = a.kblocks % a.parts;
  r.kb0 = part * q + (part < rem ? part : rem);
  r.nkb = q + (part < rem ? 1 : 0);
  r.nseg = (r.nkb + SEG_KBLOCKS - 1) / SEG_KBLOCKS;      // 0 for an empty unit: every role skips it
  return r;
}

// ---------------------------------------------------------------- kernel ----
template <class CFG, int AMODE, int BMODE>
__global__ void __launch_bounds__(T_THREADS, 1)
tgemm_kernel(const __grid_constant__ CUtensorMap mapAh, const __grid_constant__ CUtensorMap mapAl,
             const __grid_constant__ CUtensorMap mapBh, const __grid_constant__ CUtensorMap mapBl,
             const TKernelArgs a) {
  constexpr int BN = CFG::BN, STAGES = CFG::STAGES, NOPS = CFG::NOPS;
  constexpr int A_BYTES = CFG::A_BYTES, B_BYTES = CFG::B_BYTES, STAGE_BYTES = CFG::STAGE_BYTES;
  extern __shared__ uint8_t tg_smem_raw[];
  const uint32_t smem_base = (smem_u32(tg_smem_raw) + 1023u) & ~1023u;      // swizzle-128B atoms need 1024-byte alignment
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  // barrier slots (8 bytes each): full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], then the TMEM base address
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(tg_smem_raw + (tmem_slot - smem_u32(tg_smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapAh);
    tma_prefetch_desc(&mapBh);
    if (NOPS == 2) {
      tma_prefetch_desc(&mapAl);
      tma_prefetch_desc(&mapBl);
    }
    for (int s = 0; s < STAGES; ++s) {
      mbar_init_(full_bar(s), 1);
      mbar_init_(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init_(tfull_bar(s), 1);
      mbar_init_(tempty_bar(s), 4);        // one arrival per epilogue warp
    }
    fence_barrier_init_();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot),
                 "n"(CFG::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ================================================== TMA producer ====
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (long u = blockIdx.x; u < a.units; u += gridDim.x) {
        const TUnit U = decode_unit(a, BN, u);
        for (int kb = 0; kb < U.nkb; ++kb) {
          mbar_wait_(empty_bar(stage), phase ^ 1u);
          mbar_arrive_expect_tx_(full_bar(stage), (uint32_t)STAGE_BYTES);
          const uint32_t sA = smem_base + stage * STAGE_BYTES;
          const uint32_t sB = sA + NOPS * A_BYTES;
          const int k0 = (U.kb0 + kb) * TBK;
#pragma unroll
          for (int o = 0; o < NOPS; ++o) {
            const CUtensorMap* mA = o == 0 ? &mapAh : &mapAl;
            const CUtensorMap* mB = o == 0 ? &mapBh : &mapBl;
            if (AMODE == T_KC) {
              tma_load_2d(sA + o * A_BYTES, mA, full_bar(stage), k0, U.m0);            // box {32 k, 128 rows}
            } else {
#pragma unroll
              for (int j = 0; j < TBM / 32; ++j)                                        // box {32 rows, 32 k}
                tma_load_2d(sA + o * A_BYTES + j * (TBK * 128), mA, full_bar(stage), U.m0 + 32 * j, k0);
            }
            if (BMODE == T_KC) {
              tma_load_2d(sB + o * B_BYTES, mB, full_bar(stage), k0, U.n0);            // box {32 k, BN rows}
            } else {
#pragma unroll
              for (int j = 0; j < BN / 32; ++j)
                tma_load_2d(sB + o * B_BYTES + j * (TBK * 128), mB, full_bar(stage), U.n0 + 32 * j, k0);
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ==================================================== MMA issuer ====
    if (elect_one()) {
      // instruction descriptor: D = F32, A = B = TF32, majors, N >> 3, M >> 4
      constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(AMODE == T_KS) << 15) |
                                 ((uint32_t)(BMODE == T_KS) << 16) | ((uint32_t)(BN >> 3) << 17) |
                                 ((uint32_t)(TBM >> 4) << 24);
      // K-major (KC): rows of 128 B, 8-row swizzle atoms 1024 B apart (SBO); one UMMA_K = 32 B along the row.
      // MN-major (KS): 32-element (128 B) row chunks, [32 k][128 B] per chunk = 4096 B apart (LBO); the 32-byte-base
      //                swizzle atom is 4 k-rows = 512 B (SBO), one UMMA_K = 8 k-rows = 1024 B.
      constexpr uint32_t A_LBO = AMODE == T_KC ? 16u : (uint32_t)(TBK * 128), A_SBO = AMODE == T_KC ? 1024u : 512u;
      constexpr uint32_t B_LBO = BMODE == T_KC ? 16u : (uint32_t)(TBK * 128), B_SBO = BMODE == T_KC ? 1024u : 512u;
      constexpr uint32_t A_LT = AMODE == T_KC ? 2u : 1u, B_LT = BMODE == T_KC ? 2u : 1u;
      constexpr uint32_t A_KSTEP = AMODE == T_KC ? (UMMA_K * 4) : (UMMA_K * 128);
      constexpr uint32_t B_KSTEP = BMODE == T_KC ? (UMMA_K * 4) : (UMMA_K * 128);
      const uint64_t da0 = umma_desc(0u, A_LBO, A_SBO, A_LT), db0 = umma_desc(0u, B_LBO, B_SBO, B_LT);
      const uint32_t a_hi = (uint32_t)(da0 >> 32), a_lo0 = (uint32_t)da0;
      const uint32_t b_hi = (uint32_t)(db0 >> 32), b_lo0 = (uint32_t)db0;
      int stage = 0;
      uint32_t phase = 0;
      uint32_t it = 0;                       // accumulator-stage use counter
      for (long u = blockIdx.x; u < a.units; u += gridDim.x) {
        const TUnit U = decode_unit(a, BN, u);
        for (int sg = 0; sg < U.nseg; ++sg, ++it) {
          const uint32_t as = it & 1u, aphase = (it >> 1) & 1u;
          mbar_wait_(tempty_bar(as), aphase ^ 1u);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + as * BN;
          const int kb_begin = sg * SEG_KBLOCKS;
          const int kb_end = (kb_begin + SEG_KBLOCKS < U.nkb) ? kb_begin + SEG_KBLOCKS : U.nkb;
          for (int kb = kb_begin; kb < kb_end; ++kb) {
            mbar_wait_(full_bar(stage), phase);
            tc_fence_after();
            const uint32_t sA = smem_base + stage * STAGE_BYTES;
            const uint32_t sB = sA + NOPS * A_BYTES;
            // descriptor lo halves of this stage (the hi halves are loop invariant): one add per operand per MMA
            const uint32_t a_lo = a_lo0 + (sA >> 4), b_lo = b_lo0 + (sB >> 4);
#pragma unroll
            for (int kk = 0; kk < TBK / UMMA_K; ++kk) {
              const uint32_t ak = a_lo + kk * (A_KSTEP >> 4), bk = b_lo + kk * (B_KSTEP >> 4);
              const uint32_t acc0 = (kb > kb_begin || kk > 0) ? 1u : 0u;
              if (NOPS == 1) {
                umma_tf32_lohi(tmem_d, ak, a_hi, bk, b_hi, idesc, acc0);
              } else {
                umma_tf32_lohi(tmem_d, ak + (A_BYTES >> 4), a_hi, bk, b_hi, idesc, acc0);     // small terms first
                umma_tf32_lohi(tmem_d, ak, a_hi, bk + (B_BYTES >> 4), b_hi, idesc, 1u);
                umma_tf32_lohi(tmem_d, ak, a_hi, bk, b_hi, idesc, 1u);
              }
            }
            umma_commit(empty_bar(stage));                   // smem slot free once these MMAs have read it
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
          umma_commit(tfull_bar(as));                        // accumulator segment complete
        }
      }
    }
  } else {
    // ====================================================== epilogue ====
    const int quarter = warp & 3;            // TMEM lanes 32 * (warp % 4) .. + 31 are the ones this warp may read
    const int row_local = quarter * 32 + lane;
    uint32_t it = 0;
    for (long u = blockIdx.x; u < a.units; u += gridDim.x) {
      const TUnit U = decode_unit(a, BN, u);
      const int grow = U.m0 + row_local;
      for (int sg = 0; sg < U.nseg; ++sg, ++it) {
        const uint32_t as = it & 1u, aphase = (it >> 1) & 1u;
        mbar_wait_(tfull_bar(as), aphase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * BN;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + c, v);
          tmem_wait_ld();
          if (a.ws != nullptr) {
            // raw FP64 partial tile; the same thread owns the same addresses in every segment
            double* wp = a.ws + (size_t)u * (size_t)(TBM * BN) + (size_t)row_local * BN + c;
            const bool add = (sg > 0) || (a.ws_add_first != 0);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              double o0 = 0.0, o1 = 0.0, o2 = 0.0, o3 = 0.0;
              if (add) ld_global_v4(wp + j, o0, o1, o2, o3);
              st_global_v4(wp + j, o0 + (double)__uint_as_float(v[j]), o1 + (double)__uint_as_float(v[j + 1]),
                           o2 + (double)__uint_as_float(v[j + 2]), o3 + (double)__uint_as_float(v[j + 3]));
            }
          } else if (grow < a.M) {
            const int gcol = U.n0 + c;
            const double rs = a.alpha * (a.rowscale ? a.rowscale[grow] : 1.0);
            double* cp = a.C + (long)grow * a.ldc + gcol;
            if (a.c_vec && gcol + 32 <= a.N) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                double s0 = rs, s1 = rs, s2 = rs, s3 = rs;
                if (a.colscale) {
                  s0 *= a.colscale[gcol + j];
                  s1 *= a.colscale[gcol + j + 1];
                  s2 *= a.colscale[gcol + j + 2];
                  s3 *= a.colscale[gcol + j + 3];
                }
                st_global_v4(cp + j, s0 * (double)__uint_as_float(v[j]), s1 * (double)__uint_as_float(v[j + 1]),
                             s2 * (double)__uint_as_float(v[j + 2]), s3 * (double)__uint_as_float(v[j + 3]));
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                if (gcol + j < a.N) {
                  const double cs = a.colscale ? a.colscale[gcol + j] : 1.0;
                  cp[j] = rs * cs * (double)__uint_as_float(v[j]);
                }
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_(tempty_bar(as));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(CFG::TMEM_COLS)
                 : "memory");
  }
}

// Sum the FP64 partial tiles of all parts in a fixed order and apply the scaling;
// lower: only r >= c is produced and mirrored (exactly symmetric result).
template <int BN>
__global__ void __launch_bounds__(256) tgemm_reduce_kernel(const TKernelArgs a) {
  const long per_tile = (long)TBM * BN;
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= per_tile * a.ntiles) return;
  const int tile = (int)(idx / per_tile), e = (int)(idx % per_tile);
  int tm, tn;
  decode_tile(a, BN, tile, tm, tn);
  const int r = tm * TBM + e / BN, c = tn * BN + e % BN;
  if (r >= a.M || c >= a.N) return;
  if (a.lower && r < c) return;
  double s = 0.0;
  const double* wp = a.ws + (size_t)tile * per_tile + e;
  for (int part = 0; part < a.parts; ++part) s += wp[(size_t)part * a.ntiles * per_tile];
  double v = s * a.alpha;
  if (a.rowscale) v *= a.rowscale[r];
  if (a.colscale) v *= a.colscale[c];
  a.C[(long)r * a.ldc + c] = v;
  if (a.lower && r != c) a.C[(long)c * a.ldc + r] = v;
}

// FP64 -> TF32 hi (+ lo), four columns per thread.
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__global__ void __launch_bounds__(256) tf32_convert_kernel(const double* __restrict__ X, long ldx, long rows, int cols,
                                                           const double* __restrict__ rowscale, int sqrt_scale,
                                                           float* __restrict__ hi, float* __restrict__ lo, long ldo,
                                                           int x_vec) {
  const int groups = (int)(ldo / 4);
  const long total = rows * groups;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const long r = idx / groups;
    const int c = (int)(idx % groups) * 4;
    double x[4] = {0.0, 0.0, 0.0, 0.0};
    const double* xp = X + r * ldx + c;
    if (x_vec && c + 4 <= cols) {
      const double2 p0 = ld_stream2(xp), p1 = ld_stream2(xp + 2);
      x[0] = p0.x; x[1] = p0.y; x[2] = p1.x; x[3] = p1.y;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (c + j < cols) x[j] = xp[j];
    }
    if (rowscale) {
      double sc = rowscale[r];
      if (sqrt_scale) sc = (sc == sc) ? sqrt(fmax(sc, 0.0)) : sc;     // a NaN weight stays NaN (fmax would drop it)
#pragma unroll
      for (int j = 0; j < 4; ++j) x[j] *= sc;
    }
    float h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      h[j] = to_tf32((float)x[j]);
      l[j] = to_tf32((float)(x[j] - (double)h[j]));
    }
    *reinterpret_cast<float4*>(hi + r * ldo + c) = make_float4(h[0], h[1], h[2], h[3]);
    if (lo) *reinterpret_cast<float4*>(lo + r * ldo + c) = make_float4(l[0], l[1], l[2], l[3]);
  }
}

// ------------------------------------------------------------ host side ----
// 2-D FP32 tensor map.  KC: dims {K, rows}, box {32, box_rows}, 128-byte swizzle of 16-byte chunks;
// KS: dims {rows, K}, box {32, 32}, 128-byte swizzle of 32-byte chunks (what MN-major TF32 operands need).
int make_map(CUtensorMap* map, const float* base, int mode, long rows, long K, long ld, int box_rows) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) {
    set_error("tgemm: cuTensorMapEncodeTiled is not available from this driver");
    return VT_ERR_CUDA;
  }
  cuuint64_t gdim[2], gstride[1];
  cuuint32_t box[2], estr[2] = {1, 1};
  if (mode == T_KC) {
    gdim[0] = (cuuint64_t)K; gdim[1] = (cuuint64_t)rows;
    box[0] = TBK; box[1] = (cuuint32_t)box_rows;
  } else {
    gdim[0] = (cuuint64_t)rows; gdim[1] = (cuuint64_t)K;
    box[0] = 32; box[1] = TBK;
  }
  gstride[0] = (cuuint64_t)ld * 4;
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE,
                         mode == T_KC ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("tgemm: cuTensorMapEncodeTiled failed with code %d (rows=%ld K=%ld ld=%ld mode=%d)", (int)r, rows, K, ld,
              mode);
    return VT_ERR_CUDA;
  }
  return VT_OK;
}

int count_tiles(int M, int N, int BN, int lower) {
  const int tm = (M + TBM - 1) / TBM, tn = (N + BN - 1) / BN;
  if (!lower) return tm * tn;
  int n = 0;
  for (int i = 0; i < tm; ++i) n += lower_cols(i, tn, BN);
  return n;
}

int pick_parts(int ntiles, int kblocks) {
  const int G = num_sms();
  if (ntiles >= 2 * G) return 1;
  int pmax = kblocks / 16;                     // at least 16 k-blocks (512 k) per unit
  if (pmax > 4 * G) pmax = 4 * G;
  if (pmax < 2) return 1;
  int best = 1;
  double best_eff = 0.0;
  for (int P = 1; P <= pmax; ++P) {
    const long U = (long)ntiles * P;
    const double eff = (double)U / ((double)G * (double)((U + G - 1) / G));
    if (eff > best_eff + 1e-9) { best_eff = eff; best = P; }
    if (eff >= 0.9) break;                     // few, long units: the FP64 partial tiles should stay in L2
  }
  return best;
}

struct TLaunch {
  TGemmParams p;
  int lower;
  int ws_add_first;     // accumulate into an already initialised workspace
  int finalize;         // run the reduction into C
  int force_ws;         // keep the result in the workspace even for a single part / segment
};

template <class CFG, int AMODE, int BMODE>
int launch_cfg(const TLaunch& L, cudaStream_t stream) {
  const TGemmParams& p = L.p;
  constexpr int BN = CFG::BN;
  TKernelArgs a{};
  a.M = p.M; a.N = p.N;
  a.kblocks = (int)((p.K + TBK - 1) / TBK);
  a.tiles_m = (p.M + TBM - 1) / TBM;
  a.tiles_n = (p.N + BN - 1) / BN;
  a.lower = L.lower;
  a.ntiles = count_tiles(p.M, p.N, BN, L.lower);
  a.parts = p.parts > 0 ? p.parts : pick_parts(a.ntiles, a.kblocks);   // explicit parts are kept (empty units are skipped)
  if (a.parts < 1) a.parts = 1;
  a.units = (long)a.ntiles * a.parts;
  a.C = p.C; a.ldc = p.ldc;
  a.alpha = p.alpha;
  a.colscale = p.colscale; a.rowscale = p.rowscale;
  const int max_unit_kb = (a.kblocks + a.parts - 1) / a.parts;
  const bool use_ws = L.force_ws || a.parts > 1 || max_unit_kb > SEG_KBLOCKS || L.lower;
  a.ws = nullptr;
  if (use_ws) {
    const size_t need = (size_t)a.units * TBM * BN * 8;
    VT_REQUIRE(p.workspace && p.workspace_bytes >= need, "tgemm: workspace too small (%zu bytes needed, %zu given)", need,
               p.workspace_bytes);
    a.ws = p.workspace;
  }
  a.ws_add_first = L.ws_add_first;
  a.c_vec = (p.ldc % 4 == 0) && (reinterpret_cast<uintptr_t>(p.C) % 32 == 0);

  CUtensorMap mAh, mAl, mBh, mBl;
  int st = make_map(&mAh, p.A_hi, AMODE, p.M, p.K, p.lda, TBM);
  if (st != VT_OK) return st;
  st = make_map(&mBh, p.B_hi, BMODE, p.N, p.K, p.ldb, BN);
  if (st != VT_OK) return st;
  mAl = mAh; mBl = mBh;
  if (CFG::NOPS == 2) {
    st = make_map(&mAl, p.A_lo, AMODE, p.M, p.K, p.lda, TBM);
    if (st != VT_OK) return st;
    st = make_map(&mBl, p.B_lo, BMODE, p.N, p.K, p.ldb, BN);
    if (st != VT_OK) return st;
  }
  auto kern = tgemm_kernel<CFG, AMODE, BMODE>;
  VT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CFG::SMEM_BYTES));
  const long slots = num_sms();
  const int grid = (int)(a.units < slots ? a.units : slots);
  if (a.kblocks > 0 && a.units > 0) {
    kern<<<grid, T_THREADS, CFG::SMEM_BYTES, stream>>>(mAh, mAl, mBh, mBl, a);
    VT_LAUNCH_CHECK();
  }
  if (use_ws && L.finalize) {
    const long total = (long)a.ntiles * TBM * BN;
    tgemm_reduce_kernel<BN><<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(a);
    VT_LAUNCH_CHECK();
  }
  return VT_OK;
}

using CfgT1 = TCfg<256, 1>;
using CfgT3 = TCfg<128, 3>;

int tgemm_dispatch(const TLaunch& L, cudaStream_t stream) {
  const TGemmParams& p = L.p;
  VT_REQUIRE(p.M >= 0 && p.N >= 0 && p.K >= 0, "tgemm: negative dimension");
  if (p.M == 0 || p.N == 0) return VT_OK;
  VT_REQUIRE(p.A_hi && p.B_hi && (p.C || !L.finalize), "tgemm: null operand");
  VT_REQUIRE(p.K > 0, "tgemm: K must be positive");
  VT_REQUIRE((p.A_lo == nullptr) == (p.B_lo == nullptr), "tgemm: give both or neither low-order operand");
  VT_REQUIRE(p.lda % 4 == 0 && p.ldb % 4 == 0, "tgemm: operand leading dimensions must be multiples of 4 floats");
  VT_REQUIRE(reinterpret_cast<uintptr_t>(p.A_hi) % 16 == 0 && reinterpret_cast<uintptr_t>(p.B_hi) % 16 == 0,
             "tgemm: operands must be 16-byte aligned");
  VT_REQUIRE(p.amode == p.bmode, "tgemm: mixed operand layouts are not instantiated");
  const bool x3 = p.A_lo != nullptr;
  if (p.amode == T_KC) return x3 ? launch_cfg<CfgT3, T_KC, T_KC>(L, stream) : launch_cfg<CfgT1, T_KC, T_KC>(L, stream);
  return x3 ? launch_cfg<CfgT3, T_KS, T_KS>(L, stream) : launch_cfg<CfgT1, T_KS, T_KS>(L, stream);
}

size_t ws_bytes_for(int M, int N, long K, int split, int lower, int parts) {
  const int BN = split == 3 ? CfgT3::BN : CfgT1::BN;
  const int ntiles = count_tiles(M, N, BN, lower);
  const int kblocks = (int)((K + TBK - 1) / TBK);
  int P = parts > 0 ? parts : pick_parts(ntiles, kblocks);
  if (P > kblocks) P = kblocks;
  if (P < 1) P = 1;
  // one part and one FP32 accumulation segment: the epilogue scales and stores directly, no partial tiles
  if (!lower && P == 1 && kblocks <= SEG_KBLOCKS) return 0;
  return (size_t)ntiles * P * TBM * BN * 8;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Rows of X converted per pass of the chunked drivers.  Measured on B200 (D = 1024,
// tools/tgemm_probe.py time_parts): a 39 MB chunk that stays in L2 costs 9.7 ms per 1M
// observations (the fixed costs of the two launches dominate), 155 MB 6.4 ms, 620 MB
// 6.2 ms - so the chunk is sized for launch amortisation, not for L2 residency.
long chunk_rows(long N, int D, int split, int tile_n, int tiles_m) {
  const long ld = (D + 3) / 4 * 4;
  const size_t budget = (size_t)160 << 20;
  long nb = (long)(budget / ((size_t)ld * 4 * (split == 3 ? 2 : 1))) / tile_n;
  if (nb < 1) nb = 1;
  if (tiles_m > 0) {
    // the chunk's tiles_m * nb output tiles should fill whole waves of the persistent grid
    const int G = num_sms();
    long best = nb;
    double best_eff = 0.0;
    for (long b = nb; b >= 1 && b > nb / 2; --b) {
      const long T = b * tiles_m;
      const double eff = (double)T / ((double)G * (double)((T + G - 1) / G));
      if (eff > best_eff + 1e-9) { best_eff = eff; best = b; }
    }
    nb = best;
  }
  long rows = nb * tile_n;
  if (rows > N) rows = N;
  return rows;
}

}  // namespace

namespace tc05 {
EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
}  // namespace tc05

size_t tgemm_workspace_bytes(int M, int N, long K, int split) { return ws_bytes_for(M, N, K, split, 0, 0); }

int tgemm_launch(const TGemmParams& p, cudaStream_t stream) {
  TLaunch L{};
  L.p = p;
  L.lower = 0;
  L.ws_add_first = 0;
  L.finalize = 1;
  L.force_ws = 0;
  return tgemm_dispatch(L, stream);
}

int tf32_convert(const double* X, long ldx, long rows, int cols, const double* rowscale, int sqrt_scale, float* hi,
                 float* lo, long ldo, cudaStream_t stream) {
  VT_REQUIRE(X && hi, "tf32_convert: null pointer");
  VT_REQUIRE(rows >= 0 && cols >= 1 && ldx >= cols && ldo >= cols && ldo % 4 == 0, "tf32_convert: bad shape");
  VT_REQUIRE(reinterpret_cast<uintptr_t>(hi) % 16 == 0 && (!lo || reinterpret_cast<uintptr_t>(lo) % 16 == 0),
             "tf32_convert: outputs must be 16-byte aligned");
  if (rows == 0) return VT_OK;
  const int x_vec = (ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(X) % 16 == 0);
  const long total = rows * (ldo / 4);
  long blocks = (total + 255) / 256;
  const long cap = (long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  tf32_convert_kernel<<<(unsigned)blocks, 256, 0, stream>>>(X, ldx, rows, cols, rowscale, sqrt_scale, hi, lo, ldo, x_vec);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

// ---- S = -Hinv diag(resid) X^T --------------------------------------------
// Workspace: Hinv hi [lo], one chunk of X hi [lo], and - once D > 4096 (more than one FP32 accumulation segment
// along k = D) - the FP64 partial tiles of one chunk's GEMM.
size_t ij_apply_tf32_workspace_bytes(long N, int D, int split) {
  const long ld = (D + 3) / 4 * 4;
  const int nops = split == 3 ? 2 : 1;
  const long ch = chunk_rows(N, D, split, split == 3 ? CfgT3::BN : CfgT1::BN, (D + TBM - 1) / TBM);
  return align_up((size_t)D * ld * 4, 256) * nops + align_up((size_t)ch * ld * 4, 256) * nops +
         ws_bytes_for(D, (int)ch, D, split, 0, 1);
}

int ij_apply_tf32(const double* Hinv, long ldh, const double* X, long ldx, long N, int D, const double* resid,
                  double* S, long lds, int split, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Hinv && X && resid && S && workspace, "ij_apply_tf32: null pointer");
  VT_REQUIRE(split == 1 || split == 3, "ij_apply_tf32: split must be 1 (tf32) or 3 (tf32x3)");
  VT_REQUIRE(D >= 1 && N >= 0 && ldh >= D && ldx >= D && lds >= N, "ij_apply_tf32: bad shape");
  VT_REQUIRE(workspace_bytes >= ij_apply_tf32_workspace_bytes(N, D, split), "ij_apply_tf32: workspace too small");
  if (N == 0) return VT_OK;
  const long ld = (D + 3) / 4 * 4;
  const int nops = split == 3 ? 2 : 1;
  const long ch = chunk_rows(N, D, split, split == 3 ? CfgT3::BN : CfgT1::BN, (D + TBM - 1) / TBM);
  char* w = static_cast<char*>(workspace);
  const size_t hbytes = align_up((size_t)D * ld * 4, 256), xbytes = align_up((size_t)ch * ld * 4, 256);
  float* Hh = reinterpret_cast<float*>(w);
  float* Hl = nops == 2 ? reinterpret_cast<float*>(w + hbytes) : nullptr;
  float* Xh = reinterpret_cast<float*>(w + hbytes * nops);
  float* Xl = nops == 2 ? reinterpret_cast<float*>(w + hbytes * nops + xbytes) : nullptr;
  double* ws = reinterpret_cast<double*>(w + (hbytes + xbytes) * nops);
  const size_t ws_bytes = ws_bytes_for(D, (int)ch, D, split, 0, 1);
  int st = tf32_convert(Hinv, ldh, D, D, nullptr, 0, Hh, Hl, ld, stream);
  if (st != VT_OK) return st;
  for (long r0 = 0; r0 < N; r0 += ch) {
    const long rows = (N - r0 < ch) ? N - r0 : ch;
    st = tf32_convert(X + r0 * ldx, ldx, rows, D, nullptr, 0, Xh, Xl, ld, stream);
    if (st != VT_OK) return st;
    TGemmParams p{};
    p.M = D; p.N = (int)rows; p.K = D;
    p.A_hi = Hh; p.A_lo = Hl; p.lda = ld; p.amode = T_KC;
    p.B_hi = Xh; p.B_lo = Xl; p.ldb = ld; p.bmode = T_KC;
    p.C = S + r0; p.ldc = lds;
    p.alpha = -1.0;
    p.colscale = resid + r0;
    p.rowscale = nullptr;
    p.parts = 1;
    p.workspace = ws_bytes ? ws : nullptr;
    p.workspace_bytes = ws_bytes;
    st = tgemm_launch(p, stream);
    if (st != VT_OK) return st;
  }
  return VT_OK;
}

// ---- H = X^T diag(s) X -----------------------------------------------------
namespace {
int syrk_parts(long ch, int D, int split) {
  const int BN = split == 3 ? CfgT3::BN : CfgT1::BN;
  return pick_parts(count_tiles(D, D, BN, 1), (int)((ch + TBK - 1) / TBK));
}
}  // namespace

size_t syrk_tf32_workspace_bytes(long N, int D, int split) {
  const long ld = (D + 3) / 4 * 4;
  const int nops = split == 3 ? 2 : 1;
  const long ch = chunk_rows(N, D, split, TBK, 0);
  return align_up((size_t)ch * ld * 4, 256) * nops + ws_bytes_for(D, D, ch, split, 1, syrk_parts(ch, D, split));
}

int syrk_tf32(const double* X, long ldx, long N, int D, const double* s, double* H, long ldh, int split,
              void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(X && H && workspace, "syrk_tf32: null pointer");
  VT_REQUIRE(split == 1 || split == 3, "syrk_tf32: split must be 1 (tf32) or 3 (tf32x3)");
  VT_REQUIRE(D >= 1 && N >= 1 && ldx >= D && ldh >= D, "syrk_tf32: bad shape");
  VT_REQUIRE(workspace_bytes >= syrk_tf32_workspace_bytes(N, D, split), "syrk_tf32: workspace too small");
  const long ld = (D + 3) / 4 * 4;
  const int nops = split == 3 ? 2 : 1;
  const long ch = chunk_rows(N, D, split, TBK, 0);
  const int parts = syrk_parts(ch, D, split);
  char* w = static_cast<char*>(workspace);
  const size_t xbytes = align_up((size_t)ch * ld * 4, 256);
  float* Xh = reinterpret_cast<float*>(w);
  float* Xl = nops == 2 ? reinterpret_cast<float*>(w + xbytes) : nullptr;
  double* ws = reinterpret_cast<double*>(w + xbytes * nops);
  const size_t ws_bytes = workspace_bytes - xbytes * nops;
  VT_CUDA(cudaMemsetAsync(ws, 0, ws_bytes_for(D, D, ch, split, 1, parts), stream));   // every chunk accumulates
  for (long r0 = 0; r0 < N; r0 += ch) {
    const long rows = (N - r0 < ch) ? N - r0 : ch;
    int st = tf32_convert(X + r0 * ldx, ldx, rows, D, s ? s + r0 : nullptr, 1, Xh, Xl, ld, stream);
    if (st != VT_OK) return st;
    TLaunch L{};
    TGemmParams& p = L.p;
    p.M = D; p.N = D; p.K = rows;
    p.A_hi = Xh; p.A_lo = Xl; p.lda = ld; p.amode = T_KS;
    p.B_hi = Xh; p.B_lo = Xl; p.ldb = ld; p.bmode = T_KS;
    p.C = H; p.ldc = ldh;
    p.alpha = 1.0;
    p.parts = parts;                               // the same unit layout for every chunk
    p.workspace = ws; p.workspace_bytes = ws_bytes;
    L.lower = 1;
    L.force_ws = 1;
    L.ws_add_first = 1;
    L.finalize = (r0 + rows >= N);
    st = tgemm_dispatch(L, stream);
    if (st != VT_OK) return st;
  }
  return VT_OK;
}

}  // namespace vt
