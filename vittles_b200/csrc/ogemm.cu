// FP64-grade GEMM on the INT8 tensor cores by error-free slicing - see ogemm.cuh.
#include "ogemm.cuh"
#include "grouploo.cuh"
#include "tc05.cuh"
#include <cstdlib>

namespace vt {

using namespace tc05;

namespace {

constexpr int OBM = 128;               // tile rows (TMEM lanes)
constexpr int OBN = 64;                // tile columns: S accumulators x 64 columns <= 512 TMEM columns
constexpr int OBK = 128;               // int8 elements (bytes) per k-block = one 128-byte swizzle row
constexpr int O_UMMA_K = 32;           // k per tcgen05.mma.kind::i8
constexpr int O_THREADS = 576;         // warps 0-7: slice the rows of the NEXT chunk while this one is multiplied,
                                       // warps 8-15: epilogue, warp 16: TMA producer, warp 17: MMA issuer + TMEM owner
constexpr int O_EPI_WARPS = 8, O_CONV_WARPS = 8;
constexpr int W_EPI0 = O_CONV_WARPS, W_TMA = O_CONV_WARPS + O_EPI_WARPS, W_MMA = W_TMA + 1;   // W_EPI0 % 4 == 0 (TMEM quarters)
constexpr int A_TILE_BYTES = OBM * OBK;        // 16 KB: one slice of the A tile for one k-block
constexpr int B_TILE_BYTES = OBN * OBK;        //  8 KB: one slice of the B tile for one k-block
constexpr int A_RING = 6;                      // A slices stream through a ring of this depth
constexpr int B_BUFS = 2;                      // all S slices of the B tile, double buffered over k-blocks

template <int S>
struct OCfg {
  static constexpr int B_BUF_BYTES = S * B_TILE_BYTES;
  static constexpr int SMEM_BYTES = B_BUFS * B_BUF_BYTES + A_RING * A_TILE_BYTES + 1024 + 256;
};

struct SliceJob {
  const double* X; long ldx; long rows; int cols;
  int8_t* out; long ldo; long slice_stride;
  double* scale_out; const double* fold;
  // transposed job (colmax != nullptr): out[s][feature][observation] of sq_n x_ni, one scale per feature
  const double* sq; const unsigned long long* colmax;
};

struct OKernelArgs {
  int M, N, kblocks, tiles_m, tiles_n;
  long ntiles;             // output tiles (all, or those touching the lower triangle)
  int parts;               // split-K: unit u = part * ntiles + tile; part p writes C + p * part_stride
  long units;
  int lower;
  int accumulate;          // C += result instead of C = result
  long part_stride;
  double* C; long ldc;
  double alpha;
  const double* rowscale;
  const double* colscale;
  int c_vec;
  SliceJob next;                // rows to slice during this launch (X == nullptr: none; cols <= 1024)
  unsigned long long* timing;   // development aid (VT_OGEMM_TIMING=1): clocks the MMA thread waits, summed over CTAs
  int tri;                      // A lower triangular (OBM == OBK): row block tm needs the k-blocks 0 .. tm only
                                // (honoured by the EPI_QUAD instances)
};

// Epilogue of ogemm_kernel: EPI_STORE writes C; EPI_QUAD writes, for every column n, the partial sums of squares
// of the 32 rows of each warp, P[4 tm + quarter][n] (C = P, ldc = its pitch): no tile of C is stored.
constexpr int EPI_STORE = 0, EPI_QUAD = 1;

// lower: row block tm keeps the column blocks 0 .. (tm*OBM + OBM-1) / OBN
__host__ __device__ inline int o_lower_cols(int tm, int tiles_n) {
  const int c = (tm * OBM + OBM - 1) / OBN + 1;
  return c < tiles_n ? c : tiles_n;
}
struct OUnit {
  int m0, n0, kb0, nkb, part;
};
template <int EPI>
__device__ __forceinline__ OUnit o_decode(const OKernelArgs& a, long u) {
  OUnit r;
  if constexpr (EPI == EPI_QUAD) {
    if (a.tri) {
      // Row block tm costs tm + 1 k-blocks.  Units stay in the order "row blocks fastest" (the CTAs running together
      // share the B slices in L2) with the heaviest row block first, and every other wave of gridDim.x units is
      // dealt to the CTAs in reverse: the CTA that drew a heavy tile in one wave draws a light one in the next.
      // (When 2 gridDim.x is a multiple of tiles_m, the two row blocks a CTA draws in a pair of waves add up to
      // tiles_m - 1, and the static round-robin is balanced exactly.)
#ifndef VT_QF_NAIVE_ORDER
      const long G = gridDim.x, wave = u / G, p = u % G;
      const long len = (a.units - wave * G < G) ? a.units - wave * G : G;
      const long tile = wave * G + ((wave & 1) ? len - 1 - p : p);
      const int tm = a.tiles_m - 1 - (int)(tile % a.tiles_m);
#else   // measurement aid (tools/loo_probe.py): the order of the rectangular product, lightest row block first
      const long tile = u;
      const int tm = (int)(tile % a.tiles_m);
#endif
      r.part = 0;
      r.m0 = tm * OBM;
      r.n0 = (int)(tile / a.tiles_m) * OBN;
      r.kb0 = 0;
      r.nkb = (tm + 1 < a.kblocks) ? tm + 1 : a.kblocks;
      return r;
    }
  }
  const long tile = u % a.ntiles;
  r.part = (int)(u / a.ntiles);
  int tm, tn;
  if (!a.lower) {
    tm = (int)(tile % a.tiles_m);       // row blocks fastest: CTAs that run together share the B slices in L2
    tn = (int)(tile / a.tiles_m);
  } else {
    long t = tile;
    for (tm = 0; tm < a.tiles_m - 1; ++tm) {
      const int c = o_lower_cols(tm, a.tiles_n);
      if (t < c) break;
      t -= c;
    }
    tn = (int)t;
  }
  r.m0 = tm * OBM;
  r.n0 = tn * OBN;
  const int q = a.kblocks / a.parts, rem = a.kblocks % a.parts;
  r.kb0 = r.part * q + (r.part < rem ? r.part : rem);
  r.nkb = q + (r.part < rem ? 1 : 0);
  return r;
}

// One CTA per SM walks output tiles (row blocks fastest, so that the CTAs running
// together share the B slices in L2).  Per k-block the S slices of the B tile are
// loaded once (one 3-D TMA box) and the slices of the A tile stream through a
// ring; slice s of A meets slices t = 0 .. S-1-s of B, and product (s, t) goes to
// accumulator s + t.  Every INT8 tile loaded is used by (S+1)/2 products on
// average, which keeps the L2 -> shared-memory traffic at ~47 B/clk/SM at the
// tensor peak.  The products of one A slice are issued as ONE stacked
// instruction (see the MMA issuer below); measured (ncu, S = 7, r02): tensor
// pipe 80 % active, sm__memory_throughput 77 % - 389 KB of shared-memory operand
// reads plus 168 KB of TMA writes per k-block against 3.5 k clocks of MMA issue -
// and the epilogue exposed for 11 % of the tile time (all 448 of 512 TMEM columns
// hold accumulators).  DESIGN.md 3.1 has the numbers.
// Balanced base-256 digits.  q = rint(x 2^(8S-2) / sigma) (|q| <= 2^(8S-2) <= 2^54) is written as
// q = sum_p d_p 256^p with every d_p in [-128, 127]: with the bias B = sum_p 128 256^p the ordinary bytes e_p of
// u = q + B are d_p + 128, i.e. the digits are the bytes of u ^ B.  An int8 digit then carries a full 8 bits
// (sign-magnitude digits carry 7), so 7 slices hold 54 bits and S (S + 1) / 2 = 28 digit products do the work
// of the 36 that 8 sign-magnitude slices need.
// The row maximum, its exponent and q are formed with integer instructions only, from the bit patterns: the
// converter warps of the GEMM kernel slice next to a saturated tensor pipe, where FP64 instructions of other warps
// wait ~60 clocks each for their pipe (ncu: stall_math_pipe_throttle on every DMUL / DFMA / DADD of the converters)
// while the integer pipe is idle, and the stand-alone slicers run the same code so that there is one rounding rule.
// x = +-M 2^(eb - 1075) with the 53-bit significand M, so t = x 2^(8S-2-e) = 2M >> n with n = k2 - eb,
// k2 = e + 1078 - 8S, rounded to nearest even by adding half an ulp minus one plus the bit that would become the
// last (n >= 0 because |x| < 2^e, except in a row whose maximum is subnormal, where the shift goes left).
// u = q + B is kept as two words, lo = positions 0..3 and hi = positions 4..S-1; slice `sl` (0 = most significant
// of `nslices`) of four values is packed with PRMT into one word (byte j = value j).
// (oracle/slicing.py is the CPU model; tests/test_gpu_ozaki.py compares digit for digit.)
struct Fixed4 {
  uint32_t lo[4], hi[4];       // biased digits: positions 0..3 in the bytes of lo, the rest in the bytes of hi
};
// |x| as an unsigned integer orders like the double; Inf and NaN sit above every finite value
__device__ __forceinline__ unsigned long long abs_bits(double x) {
  return (unsigned long long)__double_as_longlong(x) & 0x7fffffffffffffffULL;
}
// frexp exponent of a finite non-negative double given by its bit pattern (0 for zero), in integer instructions
__device__ __forceinline__ int frexp_exponent_bits(unsigned long long mb) {
  const int eb = (int)(mb >> 52);
  if (eb) return eb - 1022;
  return mb ? -1010 - __clzll((long long)mb) : 0;      // subnormal: highest set bit p = 63 - clz  ->  p - 1073
}
__host__ __device__ constexpr unsigned long long digit_bias64(int nslices) { return 0x8080808080808080ULL >> (8 * (8 - nslices)); }
__device__ __forceinline__ void fixed4_set_bits(Fixed4& f, int j, unsigned long long bits, int k2, unsigned long long bias64) {
  const int eb = (int)((bits >> 52) & 0x7ffULL);
  unsigned long long m = bits & 0x000fffffffffffffULL;
  m = (eb ? (m | 0x0010000000000000ULL) : m) << 1;             // subnormal: exponent 1, no hidden bit
  const int n0 = k2 - (eb ? eb : 1);
  const int n = n0 < 0 ? 0 : (n0 > 63 ? 63 : n0);              // right shift; left shift only under a subnormal maximum
  const int nl = n0 < 0 ? (n0 < -63 ? 63 : -n0) : 0;           // (rows with Inf / NaN, whose scale is NaN, get garbage)
  const unsigned long long last = (m >> n) & 1ULL;
  const unsigned long long add = n ? ((1ULL << (n - 1)) - 1ULL + last) : 0ULL;
  const unsigned long long q = ((m + add) >> n) << nl;
  const unsigned long long u = ((long long)bits < 0 ? 0ULL - q : q) + bias64;
  f.lo[j] = (uint32_t)u;
  f.hi[j] = (uint32_t)(u >> 32);
}
template <int S>
__device__ __forceinline__ uint32_t fixed4_digits(const Fixed4& f, int sl) {
  const int pos = S - 1 - sl;                      // digit position from the least significant one
  const uint32_t sel = (uint32_t)(pos < 4 ? pos : pos - 4);
  const uint32_t pick = sel | ((4u + sel) << 4);   // PRMT: byte `sel` of the first source, byte `sel` of the second
  uint32_t p01, p23;
  if (pos < 4) {
    p01 = __byte_perm(f.lo[0], f.lo[1], pick);
    p23 = __byte_perm(f.lo[2], f.lo[3], pick);
  } else {
    p01 = __byte_perm(f.hi[0], f.hi[1], pick);
    p23 = __byte_perm(f.hi[2], f.hi[3], pick);
  }
  return __byte_perm(p01, p23, 0x5410) ^ 0x80808080u;      // biased byte e -> digit e - 128
}

// One warp per row: row maximum -> power-of-two scale -> S balanced base-256 digits,
// so that 2^-6 sum_s d_s 2^{-8s} reproduces x / sigma to 8 S - 2 bits (round to nearest).
// Rows of at most 128 * RC elements are held in registers between the two passes (RC = 0: re-read).
template <int S, int RC>
__device__ __forceinline__ void slice_one_row(const SliceJob& jb, long r, int lane, bool vec) {
  const double* xr = jb.X + r * jb.ldx;
  const int cols = jb.cols;
  unsigned long long mb = 0ULL;                      // bit pattern of the row maximum of |x|
  double xv[RC > 0 ? RC : 1][4];
  if constexpr (RC > 0) {
#pragma unroll
    for (int ch = 0; ch < RC; ++ch) {
      const int c0 = ch * 128 + lane * 4;
      if (vec && c0 + 4 <= cols) {
        const double2 a0 = *reinterpret_cast<const double2*>(xr + c0), a1 = *reinterpret_cast<const double2*>(xr + c0 + 2);
        xv[ch][0] = a0.x; xv[ch][1] = a0.y; xv[ch][2] = a1.x; xv[ch][3] = a1.y;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) xv[ch][j] = (c0 + j < cols) ? xr[c0 + j] : 0.0;
      }
    }
#pragma unroll
    for (int ch = 0; ch < RC; ++ch)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned long long b = abs_bits(xv[ch][j]);
        mb = b > mb ? b : mb;
      }
  } else {
    for (int c = lane; c < cols; c += 32) {
      const unsigned long long b = abs_bits(xr[c]);
      mb = b > mb ? b : mb;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, mb, o);
    mb = other > mb ? other : mb;
  }
  const bool finite = mb < 0x7ff0000000000000ULL;
  int e = 0;
  if (finite) e = frexp_exponent_bits(mb);
  // a row with an Inf or NaN gets a NaN scale: every result that touches it is NaN, as in FP64 arithmetic
  if (lane == 0)
    jb.scale_out[r] = finite ? ldexp(1.0, e) * (jb.fold ? jb.fold[r] : 1.0) : __longlong_as_double(0x7ff8000000000000LL);
  // four consecutive elements per lane: one 4-byte store per slice, 128 contiguous bytes per warp
  int8_t* orow = jb.out + r * jb.ldo;
  if constexpr (RC > 0) {
#pragma unroll
    for (int ch = 0; ch < RC; ++ch) {
      const int c0 = ch * 128 + lane * 4;
      if (c0 < jb.ldo) {
        Fixed4 f;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          fixed4_set_bits(f, j, (unsigned long long)__double_as_longlong(xv[ch][j]), e + 1078 - 8 * S, digit_bias64(S));
#pragma unroll
        for (int s = 0; s < S; ++s)
          *reinterpret_cast<uint32_t*>(orow + (long)s * jb.slice_stride + c0) = fixed4_digits<S>(f, s);
      }
    }
  } else {
    for (int c0 = lane * 4; c0 < jb.ldo; c0 += 128) {
      Fixed4 f;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        fixed4_set_bits(f, j, (c0 + j < cols) ? (unsigned long long)__double_as_longlong(xr[c0 + j]) : 0ULL,
                        e + 1078 - 8 * S, digit_bias64(S));
#pragma unroll
      for (int s = 0; s < S; ++s)
        *reinterpret_cast<uint32_t*>(orow + (long)s * jb.slice_stride + c0) = fixed4_digits<S>(f, s);
    }
  }
}

template <int S, int RC>
__global__ void __launch_bounds__(256) ozaki_slice_kernel(const SliceJob jb) {
  const int lane = threadIdx.x & 31;
  const long warp0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long nwarps = ((long)gridDim.x * blockDim.x) >> 5;
  const bool vec = (jb.ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(jb.X) % 16 == 0);
  for (long r = warp0; r < jb.rows; r += nwarps) slice_one_row<S, RC>(jb, r, lane, vec);
}
// rows of up to 1024 elements stay in registers, narrow rows in an instance with fewer of them
template <int S>
void (*row_slicer(int cols))(SliceJob) {
  return cols <= 128 ? ozaki_slice_kernel<S, 1> : cols <= 256 ? ozaki_slice_kernel<S, 2>
       : cols <= 512 ? ozaki_slice_kernel<S, 4> : cols <= 1024 ? ozaki_slice_kernel<S, 8> : ozaki_slice_kernel<S, 0>;
}

// Tile of 32 observations x 32 features per warp, lane = feature: 32 coalesced 256-byte reads (all in flight at
// once), the 32 values of a feature stay in the lane's registers, and the digits of 16 consecutive observations of
// one slice leave as one 16-byte store (two per 32-byte sector, back to back) - the transposition costs no shared
// memory, so the converter warps of the GEMM kernel can run it next to the operand ring.  Observations past `rows`
// are written as zeros up to the next multiple of 16 (the GEMM's tensor map ends at `rows` anyway).
constexpr int ST_OBS = 32, ST_FEAT = 32, ST_GROUP = 8;      // a CTA step: ST_GROUP consecutive tiles along the observations
template <int S>
__device__ __forceinline__ void slice_t_tile(const SliceJob& jb, long n0, int i0, int lane, bool first) {
  const int i = i0 + lane;
  const bool live = i < jb.cols;
  int e = 0;
  if (live) {
    const unsigned long long mb = jb.colmax[i];
    const double m = __longlong_as_double((long long)mb);
    const bool finite = mb < 0x7ff0000000000000ULL;
    if (finite) e = frexp_exponent_bits(mb);
    if (first) jb.scale_out[i] = finite ? ldexp(1.0, e) : m;   // NaN scale: row and column i of H become NaN
  }
  double xv[ST_OBS];
  if ((n0 + ST_OBS <= jb.rows) && (i0 + ST_FEAT <= jb.cols)) {
    const double* xp = jb.X + n0 * jb.ldx + i;
#pragma unroll
    for (int q = 0; q < ST_OBS; ++q) xv[q] = xp[q * jb.ldx];
    if (jb.sq) {                  // the one FP64 instruction per element (unweighted: none at all)
#pragma unroll
      for (int q = 0; q < ST_OBS; ++q) xv[q] *= jb.sq[n0 + q];
    }
  } else {
#pragma unroll
    for (int q = 0; q < ST_OBS; ++q) {
      const long n = n0 + q;
      xv[q] = (n < jb.rows && live) ? jb.X[n * jb.ldx + i] : 0.0;
      if (jb.sq && n < jb.rows) xv[q] *= jb.sq[n];                      // |x sq| < 2^e (same products as colmax)
    }
  }
#pragma unroll
  for (int h = 0; h < ST_OBS / 16; ++h) {
    Fixed4 f[4];
#pragma unroll
    for (int g4 = 0; g4 < 4; ++g4)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        fixed4_set_bits(f[g4], j, (unsigned long long)__double_as_longlong(xv[16 * h + 4 * g4 + j]), e + 1078 - 8 * S,
                        digit_bias64(S));
    if (live && n0 + 16 * h < jb.rows) {
      int8_t* o = jb.out + (long)i * jb.ldo + n0 + 16 * h;
#pragma unroll
      for (int sl = 0; sl < S; ++sl) {
        uint4 w;
        w.x = fixed4_digits<S>(f[0], sl); w.y = fixed4_digits<S>(f[1], sl);
        w.z = fixed4_digits<S>(f[2], sl); w.w = fixed4_digits<S>(f[3], sl);
        *reinterpret_cast<uint4*>(o + (long)sl * jb.slice_stride) = w;
      }
    }
  }
}

// CTA steps (feature blocks fastest: a wave reads whole rows of X), `nw` warps of which this one is `w`
template <int S>
__device__ __forceinline__ void slice_t_job(const SliceJob& jb, long cta, long nctas, int w, int nw, int lane) {
  const long span = (long)ST_OBS * nw;
  const long steps_x = (jb.rows + span - 1) / span;
  const int tiles_y = (jb.cols + ST_FEAT - 1) / ST_FEAT;
  for (long t = cta; t < steps_x * tiles_y; t += nctas) {
    const long n0 = (t / tiles_y) * span + (long)w * ST_OBS;
    if (n0 < jb.rows) slice_t_tile<S>(jb, n0, (int)(t % tiles_y) * ST_FEAT, lane, t < tiles_y && w == 0);
  }
}

// Exact INT64 -> FP64 for |u| < 2^51 without a conversion instruction.
__device__ __forceinline__ double exact_double(long long u) {
  return __longlong_as_double(u + 0x4338000000000000LL) - 6755399441055744.0;
}
__device__ __forceinline__ double pair_double(int hi, int lo) { return exact_double((long long)hi * 256 + (long long)lo); }

template <int S, int EPI>
__global__ void __launch_bounds__(O_THREADS, 1)
ogemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const OKernelArgs a) {
  constexpr int B_BUF_BYTES = OCfg<S>::B_BUF_BYTES;
  extern __shared__ uint8_t og_smem_raw[];
  const uint32_t smem_base = (smem_u32(og_smem_raw) + 1023u) & ~1023u;
  const uint32_t sB0 = smem_base;                                   // B_BUFS x [S][64][128 B]
  const uint32_t sA0 = smem_base + B_BUFS * B_BUF_BYTES;            // A_RING x [128][128 B]
  const uint32_t bar_base = sA0 + A_RING * A_TILE_BYTES;
  auto bfull = [&](int i) { return bar_base + 8u * i; };
  auto bempty = [&](int i) { return bar_base + 8u * (B_BUFS + i); };
  auto afull = [&](int i) { return bar_base + 8u * (2 * B_BUFS + i); };
  auto aempty = [&](int i) { return bar_base + 8u * (2 * B_BUFS + A_RING + i); };
  const uint32_t tfull = bar_base + 8u * (2 * B_BUFS + 2 * A_RING);
  const uint32_t tempty = tfull + 8u;
  const uint32_t tmem_slot = tempty + 8u;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(og_smem_raw + (tmem_slot - smem_u32(og_smem_raw)));

  // Warp roles by DESCENDING issue priority (the arbiter favours the highest warp id): W_MMA, W_TMA, the epilogue
  // warps, and at the bottom the converter warps, which only fill idle issue slots.
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == W_TMA && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapB);
    for (int i = 0; i < B_BUFS; ++i) { mbar_init_(bfull(i), 1); mbar_init_(bempty(i), 1); }
    for (int i = 0; i < A_RING; ++i) { mbar_init_(afull(i), 1); mbar_init_(aempty(i), 1); }
    mbar_init_(tfull, 1);
    mbar_init_(tempty, O_EPI_WARPS);
    fence_barrier_init_();
  }
  if (warp == W_MMA) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == W_TMA) {
    // ================================================== TMA producer ====
    if (elect_one()) {
      int bs = 0, as = 0;
      uint32_t bph = 0, aph = 0;
      for (long u = blockIdx.x; u < a.units; u += gridDim.x) {
        const OUnit U = o_decode<EPI>(a, u);
        const int m0 = U.m0, n0 = U.n0;
        for (int kb = U.kb0; kb < U.kb0 + U.nkb; ++kb) {
          mbar_wait_(bempty(bs), bph ^ 1u);
          mbar_arrive_expect_tx_(bfull(bs), (uint32_t)B_BUF_BYTES);
          tma_load_3d(sB0 + bs * B_BUF_BYTES, &mapB, bfull(bs), kb * OBK, n0, 0);        // box {128 B, 64 rows, S slices}
          if (++bs == B_BUFS) { bs = 0; bph ^= 1u; }
#pragma unroll 1
          for (int s = 0; s < S; ++s) {
            mbar_wait_(aempty(as), aph ^ 1u);
            mbar_arrive_expect_tx_(afull(as), (uint32_t)A_TILE_BYTES);
            tma_load_3d(sA0 + as * A_TILE_BYTES, &mapA, afull(as), kb * OBK, m0, s);     // box {128 B, 128 rows, 1 slice}
            if (++as == A_RING) { as = 0; aph ^= 1u; }
          }
        }
      }
    }
  } else if (warp == W_MMA) {
    // ==================================================== MMA issuer ====
    if (elect_one()) {
      // instruction descriptor: D = S32, A = B = signed INT8, both K-major, N >> 3, M >> 4
      constexpr uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OBM >> 4) << 24);
      // K-major 128-byte-swizzled operand: descriptor hi half = SBO 1024 B | version 1 | SWIZZLE_128B (constant),
      // lo half = (address >> 4) | LBO 16 B << 16; one UMMA_K = 32 B = +2, one B slice = 8 KB = +512.
      const uint64_t d0 = umma_desc(0u, 16u, 1024u, 2u);
      const uint32_t desc_hi = (uint32_t)(d0 >> 32), desc_lo0 = (uint32_t)d0;
      int bs = 0, as = 0;
      uint32_t bph = 0, aph = 0, tph = 0;
      long long w_t = 0, w_b = 0, w_a = 0;
      const long long t_begin = clock64();
      for (long u = blockIdx.x; u < a.units; u += gridDim.x) {
        const OUnit U = o_decode<EPI>(a, u);
        if (U.nkb == 0) continue;              // every role skips an empty unit
        long long c0 = clock64();
        mbar_wait_(tempty, tph ^ 1u);          // the epilogue has drained the accumulators of the previous tile
        w_t += clock64() - c0;
        tc_fence_after();
        for (int kb = 0; kb < U.nkb; ++kb) {
          c0 = clock64();
          mbar_wait_(bfull(bs), bph);
          w_b += clock64() - c0;
          const uint32_t b_lo0 = desc_lo0 + ((sB0 + bs * B_BUF_BYTES) >> 4);
          const uint32_t first = kb == 0 ? 0u : 1u;
#pragma unroll
          for (int s = 0; s < S; ++s) {
            c0 = clock64();
            mbar_wait_(afull(as), aph);
            w_a += clock64() - c0;
            tc_fence_after();
            const uint32_t a_lo0 = desc_lo0 + ((sA0 + as * A_TILE_BYTES) >> 4);
            // Slice s of A meets slices 0 .. S-1-s of B, whose tiles are CONTIGUOUS in the B box (64 rows of
            // 128 bytes each), and product (s, t) belongs to accumulator s + t = columns 64 (s + t): one
            // tcgen05.mma with N = 64 (S - s) (cut at 256) does them all and reads the A tile once instead of
            // S - s times - 10 instructions and 96 KB of shared-memory operand reads per k-step for S = 7
            // instead of 28 instructions and 168 KB (the N = 64 form is bound by those reads).
            // (measured, bare issue loop: an instruction of N columns costs max(N / 2, 34 + 0.36 N) clocks - 128 for
            // N = 256, 101 for 192, 80 for 128, 57 for 64 - so 448 columns go as 256 + 192, 384 as 192 + 192, ...)
            const int NTOT = OBN * (S - s);
            const int NPART = (NTOT + 255) / 256;
            const int NFIRST = ((NTOT / NPART) + 63) / 64 * 64;           // balanced parts, multiples of 64
#pragma unroll
            for (int pn = 0; pn < NPART; ++pn) {
              const int c0 = pn * NFIRST;
              const int n = (pn == NPART - 1) ? NTOT - c0 : NFIRST;
              const uint32_t idesc = idesc0 | ((uint32_t)(n >> 3) << 17);
              const uint32_t tmem_d = tmem_base + (uint32_t)(s * OBN + c0);
              const uint32_t b_lo = b_lo0 + (uint32_t)((c0 / OBN) * (B_TILE_BYTES >> 4));
#pragma unroll
              for (int kk = 0; kk < OBK / O_UMMA_K; ++kk)
                umma_i8_lohi(tmem_d, a_lo0 + 2u * kk, desc_hi, b_lo + 2u * kk, desc_hi, idesc,
                             (s == 0 && kk == 0) ? first : 1u);
            }
            umma_commit(aempty(as));
            if (++as == A_RING) { as = 0; aph ^= 1u; }
          }
          umma_commit(bempty(bs));
          if (++bs == B_BUFS) { bs = 0; bph ^= 1u; }
        }
        umma_commit(tfull);
        tph ^= 1u;
      }
      if (a.timing) {
        atomicAdd(a.timing + 0, (unsigned long long)(clock64() - t_begin));
        atomicAdd(a.timing + 1, (unsigned long long)w_t);
        atomicAdd(a.timing + 2, (unsigned long long)w_b);
        atomicAdd(a.timing + 3, (unsigned long long)w_a);
        atomicAdd(a.timing + 4, 1ULL);
      }
    }
  } else if (warp >= W_EPI0) {
    // ====================================================== epilogue ====
    // Eight warps: warp w reads TMEM lanes 32 (w % 4) .. + 31 (the quarter a warp may address) and the column half
    // (w - 2) / 4 of every accumulator.  sum_l P_l 2^-8l is evaluated by Horner's rule in FP64 from the least
    // significant accumulator: every P_l is an exact double and each FMA rounds at 2^-53 of a partial sum that is
    // 2^-8l of the leading terms - far below the 2^-54 sigma tau truncation of the digits themselves.
    const int ew = warp - W_EPI0;
    const int quarter = warp & 3, chalf = ew >> 2;
    const int row_local = quarter * 32 + lane;
    uint32_t tph = 0;
    for (long u = blockIdx.x; u < a.units; u += gridDim.x) {
      const OUnit U = o_decode<EPI>(a, u);
      if (U.nkb == 0) continue;
      const int m0 = U.m0, n0 = U.n0;
      const int grow = m0 + row_local;
      double* Cpart = a.C + (long)U.part * a.part_stride;
      // a . b = sigma tau 2^-12 sum_l 2^-8l P_l, and the Horner sum below carries a factor 256
      const double rs = (grow < a.M) ? a.alpha * (a.rowscale ? a.rowscale[grow] : 1.0) * (1.0 / 1048576.0) : 0.0;
      // lane j keeps the scale of column j of this warp's 32 columns (fetched before the accumulators are
      // awaited: a global load behind the TMEM wait would sit on the critical path of every strip)
      const int ccol = n0 + chalf * (OBN / 2) + lane;
      const double cs_lane = (a.colscale && ccol < a.N) ? a.colscale[ccol] : 1.0;
      mbar_wait_(tfull, tph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(chalf * (OBN / 2));
#pragma unroll 1
      for (int c = 0; c < OBN / 2; c += 8) {
        uint32_t v[S][8];
#pragma unroll
        for (int g = 0; g < S; ++g) tmem_ld8(taddr + (uint32_t)(g * OBN + c), v[g]);
        tmem_wait_ld();
        if (c + 8 == OBN / 2) {
          // the last loads have landed: the accumulators go back to the MMA warp now, and the arithmetic and the
          // stores of this final chunk overlap the next tile's first MMAs
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_(tempty);
        }
        double out[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          // Horner from the least significant accumulator over PAIRS of accumulators: P_l 256 + P_{l+1} is formed
          // in INT64 and converted exactly by adding it to the bit pattern of 1.5 2^52 (an I2F.F64 issues at a
          // quarter of the DADD / DFMA rate and one per accumulator made the conversions the epilogue's bound)
          double t;
          int g;
          if constexpr (S % 2 == 1) {
            t = exact_double((long long)(int)v[S - 1][j]);
            g = S - 3;
            t = fma(t, 1.0 / 256.0, pair_double((int)v[g][j], (int)v[g + 1][j]));
          } else {
            g = S - 2;
            t = pair_double((int)v[g][j], (int)v[g + 1][j]);
          }
#pragma unroll
          for (g -= 2; g >= 0; g -= 2) t = fma(t, 1.0 / 65536.0, pair_double((int)v[g][j], (int)v[g + 1][j]));
          out[j] = t * (rs * __shfl_sync(0xffffffffu, cs_lane, c + j));      // t = 256 sum_l P_l 2^-8l
        }
        if constexpr (EPI == EPI_QUAD) {
          // sum over the warp's 32 rows (lanes) of the squares of its 8 columns: a transpose-reduce in a fixed tree
          // (each step halves the columns a lane keeps and sums them with the partner's; a + b == b + a, so the
          // result does not depend on which lane forms it), then the last two steps over the lanes that share a
          // column.  Rows past M have rs = 0 and add zeros.
          double q[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) q[j] = out[j] * out[j];
#pragma unroll
          for (int w = 4; w >= 1; w >>= 1) {             // lane bit 4, 3, 2 -> keep the upper or lower w columns
            const bool up = (lane & (w << 2)) != 0;
#pragma unroll
            for (int j = 0; j < w; ++j) {
              const double send = up ? q[j] : q[j + w];
              const double keep = up ? q[j + w] : q[j];
              q[j] = keep + __shfl_xor_sync(0xffffffffu, send, w << 2);
            }
          }
          double v = q[0];                               // column (lane >> 2) of the 8, summed over 8 lanes so far
          v += __shfl_xor_sync(0xffffffffu, v, 2);
          v += __shfl_xor_sync(0xffffffffu, v, 1);
          const int gcol = n0 + chalf * (OBN / 2) + c + (lane >> 2);
          if ((lane & 3) == 0 && gcol < a.N) Cpart[(long)(m0 / OBM * 4 + quarter) * a.ldc + gcol] = v;
        } else if (grow < a.M) {
          const int gcol = n0 + chalf * (OBN / 2) + c;
          double* cp = Cpart + (long)grow * a.ldc + gcol;
          if (a.c_vec && gcol + 8 <= a.N) {
#pragma unroll
            for (int j = 0; j < 8; j += 4) {
              double o0 = 0.0, o1 = 0.0, o2 = 0.0, o3 = 0.0;
              if (a.accumulate) ld_global_v4(cp + j, o0, o1, o2, o3);
              st_global_v4(cp + j, o0 + out[j], o1 + out[j + 1], o2 + out[j + 2], o3 + out[j + 3]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (gcol + j < a.N) cp[j] = (a.accumulate ? cp[j] : 0.0) + out[j];
          }
        }
      }
      tph ^= 1u;
    }
  } else if (a.next.X != nullptr) {
    // ===================================================== converters ====
    // The digits of the next chunk's rows, written while the tensor pipe works on this chunk: the slicing pass
    // (HBM bound on its own: 8 bytes read, S written per element) disappears behind the GEMM.  Four consecutive
    // rows per CTA and step, one warp per row, the row held in registers between the maximum and the digits.
    const int cw = warp;
    const bool vec = (a.next.ldx % 2 == 0) && (reinterpret_cast<uintptr_t>(a.next.X) % 16 == 0);
    const long long t_begin = clock64();
    if (a.next.colmax) {
      slice_t_job<S>(a.next, blockIdx.x, gridDim.x, cw, O_CONV_WARPS, lane);
    } else {
      for (long r = (long)blockIdx.x * O_CONV_WARPS + cw; r < a.next.rows; r += (long)gridDim.x * O_CONV_WARPS)
        slice_one_row<S, 8>(a.next, r, lane, vec);
    }
    if (a.timing && lane == 0) {
      atomicAdd(a.timing + 5, (unsigned long long)(clock64() - t_begin));
      atomicAdd(a.timing + 6, 1ULL);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc<512>(tmem_base);
}

// ---- Hessian assembly: the contraction runs over the observations, so the digits are written
// TRANSPOSED (out[s][feature][observation], observations contiguous = K-major for the same GEMM
// kernel) and the power-of-two scale belongs to the feature (row of X^T).

// colmax[i] = max_n sqrt(s_n) |x_ni| over all rows given, as the bit pattern of a non-negative double
// (which orders like an unsigned integer) so that atomicMax can combine the CTAs.
__global__ void __launch_bounds__(256) ozaki_colmax_kernel(const double* __restrict__ X, long ldx, long rows, int cols,
                                                           const double* __restrict__ s, double* __restrict__ sq_out,
                                                           unsigned long long* __restrict__ colmax) {
  constexpr int ROWS_PER_STEP = 32;
  __shared__ double sq[ROWS_PER_STEP];
  const long nsteps = (rows + ROWS_PER_STEP - 1) / ROWS_PER_STEP;
  constexpr int CPT = 8;                                   // columns per thread: up to 2048 features in one sweep
  for (int cbase = 0; cbase < cols; cbase += CPT * 256) {
    double m[CPT];
#pragma unroll
    for (int j = 0; j < CPT; ++j) m[j] = 0.0;
    for (long st = blockIdx.x; st < nsteps; st += gridDim.x) {
      const long r_begin = st * ROWS_PER_STEP;
      const int nr = (int)(rows - r_begin < ROWS_PER_STEP ? rows - r_begin : ROWS_PER_STEP);
      __syncthreads();
      if (threadIdx.x < nr) {
        // sqrt of the weight once per observation (also kept for the slicing kernel)
        double v = 1.0;
        if (s) {
          const double sv = s[r_begin + threadIdx.x];
          v = (sv == sv) ? sqrt(fmax(sv, 0.0)) : sv;         // a NaN weight stays NaN (fmax would drop it)
        }
        sq[threadIdx.x] = v;
        if (cbase == 0 && sq_out) sq_out[r_begin + threadIdx.x] = v;
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        const int c = cbase + threadIdx.x + j * 256;
        if (c < cols) {
          double mm = m[j];
#pragma unroll 8
          for (int r = 0; r < nr; ++r) {
            const double v = fabs(X[(r_begin + r) * ldx + c]) * sq[r];
            // a non-finite product poisons the column: the quiet-NaN pattern is above every finite one in atomicMax
            mm = (v <= 1.7976931348623157e308 && mm == mm) ? fmax(mm, v) : __longlong_as_double(0x7ff8000000000000LL);
          }
          m[j] = mm;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      const int c = cbase + threadIdx.x + j * 256;
      if (c < cols) atomicMax(colmax + c, (unsigned long long)__double_as_longlong(m[j]));
    }
  }
}

template <int S>
__global__ void __launch_bounds__(32 * ST_GROUP) ozaki_slice_t_kernel(const SliceJob jb) {
  slice_t_job<S>(jb, blockIdx.x, gridDim.x, threadIdx.x >> 5, ST_GROUP, threadIdx.x & 31);
}

// H = sum of the split-K partial buffers over the lower triangle, mirrored (exactly symmetric).
__global__ void __launch_bounds__(256) ozaki_syrk_finish_kernel(const double* __restrict__ P, int parts, long part_stride,
                                                                int D, double* __restrict__ H, long ldh) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)D * D) return;
  const int r = (int)(idx / D), c = (int)(idx % D);
  if (r < c) return;
  double v = 0.0;
  for (int p = 0; p < parts; ++p) v += P[(long)p * part_stride + (long)r * D + c];
  H[(long)r * ldh + c] = v;
  if (r != c) H[(long)c * ldh + r] = v;
}

// 3-D uint8 tensor map over the slices: dims {K, rows, S}, box {128, box_rows, box_slices}, 128-byte swizzle.
int make_slice_map(CUtensorMap* map, const int8_t* base, long rows, int K, long ld, long slice_stride, int nslices,
                   int box_rows, int box_slices) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) {
    set_error("ogemm: cuTensorMapEncodeTiled is not available from this driver");
    return VT_ERR_CUDA;
  }
  cuuint64_t gdim[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)nslices};
  cuuint64_t gstride[2] = {(cuuint64_t)ld, (cuuint64_t)slice_stride};
  cuuint32_t box[3] = {(cuuint32_t)OBK, (cuuint32_t)box_rows, (cuuint32_t)box_slices};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(base), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("ogemm: cuTensorMapEncodeTiled failed with code %d (rows=%ld K=%d ld=%ld slice_stride=%ld)", (int)r, rows,
              K, ld, slice_stride);
    return VT_ERR_CUDA;
  }
  return VT_OK;
}

// VT_OGEMM_TIMING=1: a device buffer of 8 counters {total, wait accumulators, wait B, wait A, CTAs} that every
// launch adds to; vt_debug_ogemm_timing() reads and clears it.
unsigned long long* ogemm_timing_buffer() {
  static unsigned long long* buf = [] {
    const char* e = getenv("VT_OGEMM_TIMING");
    unsigned long long* p = nullptr;
    if (e && e[0] == '1' && cudaMalloc(&p, 64) == cudaSuccess) cudaMemset(p, 0, 64);
    return p;
  }();
  return buf;
}

template <int S, int EPI>
int launch_s(const CUtensorMap& mA, const CUtensorMap& mB, const OKernelArgs& a, cudaStream_t stream) {
  auto kern = ogemm_kernel<S, EPI>;
  VT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, OCfg<S>::SMEM_BYTES));
  VT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  const long slots = num_sms();
  // CTAs without a unit still run their share of the slicing job
  const int grid = (int)((a.units < slots && !a.next.X) ? a.units : slots);
  kern<<<grid, O_THREADS, OCfg<S>::SMEM_BYTES, stream>>>(mA, mB, a);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

inline size_t align_up(size_t x, size_t al) { return (x + al - 1) / al * al; }

long ozaki_chunk_rows(long N, int D, int nslices) {
  const long ld = (D + 15) / 16 * 16;
  const size_t budget = (size_t)288 << 20;                 // all slices of one chunk
  long nb = (long)(budget / ((size_t)ld * nslices)) / OBN;
  if (nb < 1) nb = 1;
  // tiles_m * nb output tiles should fill whole waves of the persistent grid
  const int G = num_sms(), tiles_m = (D + OBM - 1) / OBM;
  long best = nb;
  double best_eff = 0.0;
  for (long b = nb; b >= 1 && b > nb / 2; --b) {
    const long T = b * tiles_m;
    const double eff = (double)T / ((double)G * (double)((T + G - 1) / G));
    if (eff > best_eff + 1e-9) { best_eff = eff; best = b; }
  }
  long rows = best * OBN;
  if (rows > N) rows = N;
  return rows;
}

}  // namespace

unsigned long long* ogemm_timing_buffer_public() { return ogemm_timing_buffer(); }

int ozaki_slice(const double* X, long ldx, long rows, int cols, int8_t* out, long ldo, long slice_stride, int nslices,
                double* scale_out, const double* fold, cudaStream_t stream) {
  VT_REQUIRE(X && out && scale_out, "ozaki_slice: null pointer");
  VT_REQUIRE(rows >= 0 && cols >= 1 && ldx >= cols && ldo >= cols && ldo % 16 == 0, "ozaki_slice: bad shape");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES && slice_stride >= rows * ldo && slice_stride % 16 == 0,
             "ozaki_slice: bad slice layout");
  VT_REQUIRE(reinterpret_cast<uintptr_t>(out) % 16 == 0, "ozaki_slice: output must be 16-byte aligned");
  if (rows == 0) return VT_OK;
  const int bt = 256;
  long blocks = (rows + bt / 32 - 1) / (bt / 32);
  const long cap = (long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  const SliceJob jb{X, ldx, rows, cols, out, ldo, slice_stride, scale_out, fold, nullptr, nullptr};
  const auto kern = nslices == 5 ? row_slicer<5>(cols) : nslices == 6 ? row_slicer<6>(cols) : row_slicer<7>(cols);
  kern<<<(unsigned)blocks, bt, 0, stream>>>(jb);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

// Transposed digits out[s][feature][observation] of sq_n x_ni (the Hessian's operand) as a launch of its own.
int ozaki_slice_t(const double* X, long ldx, long rows, int cols, const double* sq, const unsigned long long* colmax,
                  int8_t* out, long ldo, long slice_stride, int nslices, double* scale_out, cudaStream_t stream) {
  VT_REQUIRE(X && colmax && out && scale_out, "ozaki_slice_t: null pointer");      // sq == nullptr: unweighted
  VT_REQUIRE(rows >= 1 && cols >= 1 && ldx >= cols && ldo >= rows && ldo % 16 == 0 && slice_stride >= (long)cols * ldo &&
             slice_stride % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0, "ozaki_slice_t: bad layout");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES, "ozaki_slice_t: 5, 6 or 7 slices");
  const SliceJob jb{X, ldx, rows, cols, out, ldo, slice_stride, scale_out, nullptr, sq, colmax};
  const long steps = ((rows + ST_OBS * ST_GROUP - 1) / (ST_OBS * ST_GROUP)) * ((cols + ST_FEAT - 1) / ST_FEAT);
  const long cap = (long)num_sms() * 6;
  const unsigned grid = (unsigned)(steps < cap ? steps : cap);
  const auto kern = nslices == 5 ? ozaki_slice_t_kernel<5> : nslices == 6 ? ozaki_slice_t_kernel<6> : ozaki_slice_t_kernel<7>;
  kern<<<grid, 32 * ST_GROUP, 0, stream>>>(jb);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

namespace {
struct OLaunchOpts {
  int lower = 0, parts = 1, accumulate = 0;
  int epi = EPI_STORE, tri = 0;
  long part_stride = 0;
  SliceJob next{};              // rows sliced by the converter warps of this launch (X == nullptr: none)
};

int ogemm_launch_opts(int M, int N, int K, const int8_t* A, long lda, long a_slice_stride, const int8_t* B, long ldb,
                      long b_slice_stride, int nslices, double alpha, const double* rowscale, const double* colscale,
                      double* C, long ldc, const OLaunchOpts& o, cudaStream_t stream) {
  VT_REQUIRE(M >= 0 && N >= 0 && K >= 1, "ogemm: bad dimensions");
  if (M == 0 || N == 0) return VT_OK;
  VT_REQUIRE(A && B && C, "ogemm: null operand");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES, "ogemm: 5, 6 or 7 slices are instantiated");
  VT_REQUIRE(o.parts >= 1 && (K + o.parts - 1) / o.parts <= OZAKI_MAX_K + OBK,
             "ogemm: K = %d in %d part(s) exceeds %d per part (INT32 accumulation bound)", K, o.parts, OZAKI_MAX_K);
  VT_REQUIRE(lda % 16 == 0 && ldb % 16 == 0 && a_slice_stride % 16 == 0 && b_slice_stride % 16 == 0,
             "ogemm: pitches must be multiples of 16 bytes");
  VT_REQUIRE(reinterpret_cast<uintptr_t>(A) % 16 == 0 && reinterpret_cast<uintptr_t>(B) % 16 == 0,
             "ogemm: operands must be 16-byte aligned");
  if (o.lower) VT_REQUIRE(M == N, "ogemm: lower-only output must be square");
  VT_REQUIRE(!o.tri || (o.epi == EPI_QUAD && !o.lower && o.parts == 1), "ogemm: triangular K range: quadratic forms only");
  CUtensorMap mA, mB;
  int st = make_slice_map(&mA, A, M, K, lda, a_slice_stride, nslices, OBM, 1);
  if (st != VT_OK) return st;
  st = make_slice_map(&mB, B, N, K, ldb, b_slice_stride, nslices, OBN, nslices);
  if (st != VT_OK) return st;
  OKernelArgs a{};
  a.M = M; a.N = N;
  a.kblocks = (K + OBK - 1) / OBK;
  a.tiles_m = (M + OBM - 1) / OBM;
  a.tiles_n = (N + OBN - 1) / OBN;
  a.lower = o.lower;
  if (o.lower) {
    a.ntiles = 0;
    for (int tm = 0; tm < a.tiles_m; ++tm) a.ntiles += o_lower_cols(tm, a.tiles_n);
  } else {
    a.ntiles = (long)a.tiles_m * a.tiles_n;
  }
  a.parts = o.parts;
  a.units = a.ntiles * a.parts;
  a.accumulate = o.accumulate;
  a.part_stride = o.part_stride;
  a.C = C; a.ldc = ldc;
  a.alpha = alpha;
  a.rowscale = rowscale; a.colscale = colscale;
  a.c_vec = (ldc % 4 == 0) && (reinterpret_cast<uintptr_t>(C) % 32 == 0) && (o.part_stride % 4 == 0);
  a.next = o.next;
  if (a.next.X)
    VT_REQUIRE((a.next.colmax || a.next.cols <= 1024) && a.next.ldo % 16 == 0,
               "ogemm: in-kernel slicing takes rows of at most 1024 elements");
  a.timing = ogemm_timing_buffer();
  a.tri = o.tri;
  if (o.epi == EPI_QUAD) {
    switch (nslices) {
      case 5: return launch_s<5, EPI_QUAD>(mA, mB, a, stream);
      case 6: return launch_s<6, EPI_QUAD>(mA, mB, a, stream);
      default: return launch_s<7, EPI_QUAD>(mA, mB, a, stream);
    }
  }
  switch (nslices) {
    case 5: return launch_s<5, EPI_STORE>(mA, mB, a, stream);
    case 6: return launch_s<6, EPI_STORE>(mA, mB, a, stream);
    default: return launch_s<7, EPI_STORE>(mA, mB, a, stream);
  }
}
}  // namespace

// ---- INT8 tensor peak probe -------------------------------------------------
// One CTA per SM; one elected thread issues tcgen05.mma.kind::i8 (M = 128, K = 32) on resident shared-memory
// operands (pseudo-random bytes: the power drawn depends on the data) with no loads in the loop.  Per iteration
// the four k-steps of one 128-byte k-block against floor(448 / n_tile) accumulators of N = n_tile columns.
namespace {
constexpr int PROBE_COLS = 448;
__global__ void __launch_bounds__(128, 1) i8_peak_kernel(int n_tile, long iters, long long* clocks_out) {
  extern __shared__ uint8_t pk_smem_raw[];
  const uint32_t base = (smem_u32(pk_smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = base, sB = base + A_TILE_BYTES, bars = sB + PROBE_COLS * OBK, slot = bars + 64;
  uint8_t* gen = pk_smem_raw + (base - smem_u32(pk_smem_raw));
  for (int i = threadIdx.x; i < (A_TILE_BYTES + PROBE_COLS * OBK) / 4; i += blockDim.x) {
    uint32_t h = (uint32_t)i * 2654435761u + blockIdx.x * 40503u;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
    reinterpret_cast<uint32_t*>(gen)[i] = h;
  }
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) mbar_init_(bars + 8u * i, 1);
    fence_barrier_init_();
  }
  if (warp == 1) tmem_alloc<512>(slot);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");      // generic-proxy fills -> tensor-core reads
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<uint32_t*>(pk_smem_raw + (slot - smem_u32(pk_smem_raw)));
  if (warp == 1 && elect_one()) {
    constexpr uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OBM >> 4) << 24);
    const uint64_t d0 = umma_desc(0u, 16u, 1024u, 2u);
    const uint32_t desc_hi = (uint32_t)(d0 >> 32), desc_lo0 = (uint32_t)d0;
    const uint32_t a_lo0 = desc_lo0 + (sA >> 4), b_lo0 = desc_lo0 + (sB >> 4);
    const long long t0 = clock64();
    uint32_t ph[4] = {0, 0, 0, 0};
    for (long it = 0; it < iters; ++it) {
      const int r = (int)(it & 3);
      if (it >= 4) { mbar_wait_(bars + 8u * r, ph[r]); ph[r] ^= 1u; }     // at most four iterations in flight
      for (int c0 = 0; c0 + n_tile <= PROBE_COLS; c0 += n_tile) {       // whole instructions of N = n_tile only
        const int n = n_tile;
        const uint32_t idesc = idesc0 | ((uint32_t)(n >> 3) << 17);
#pragma unroll
        for (int kk = 0; kk < OBK / O_UMMA_K; ++kk)
          umma_i8_lohi(tmem_base + (uint32_t)c0, a_lo0 + 2u * kk, desc_hi, b_lo0 + (uint32_t)(c0 * (OBK >> 4)) + 2u * kk,
                       desc_hi, idesc, 1u);
      }
      umma_commit(bars + 8u * r);
    }
    for (long it = (iters > 4 ? iters - 4 : 0); it < iters; ++it) {
      const int r = (int)(it & 3);
      mbar_wait_(bars + 8u * r, ph[r]);
      ph[r] ^= 1u;
    }
    if (blockIdx.x == 0) clocks_out[0] = clock64() - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}
}  // namespace

int i8_peak_probe(double seconds, int n_tile, double* tops, double* clocks_per_mma, cudaStream_t stream) {
  VT_REQUIRE(tops && seconds > 0 && n_tile >= 16 && n_tile <= 256 && n_tile % 16 == 0, "i8_peak_probe: bad arguments");
  long long* clk = nullptr;
  VT_CUDA(cudaMalloc(&clk, 8));
  cudaEvent_t e0, e1;
  VT_CUDA(cudaEventCreate(&e0));
  VT_CUDA(cudaEventCreate(&e1));
  const int smem = A_TILE_BYTES + PROBE_COLS * OBK + 1024 + 256;
  VT_CUDA(cudaFuncSetAttribute(i8_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int grid = num_sms();
  auto run = [&](long iters, float* ms) -> int {
    VT_CUDA(cudaEventRecord(e0, stream));
    i8_peak_kernel<<<grid, 128, smem, stream>>>(n_tile, iters, clk);
    VT_LAUNCH_CHECK();
    VT_CUDA(cudaEventRecord(e1, stream));
    VT_CUDA(cudaEventSynchronize(e1));
    VT_CUDA(cudaEventElapsedTime(ms, e0, e1));
    return VT_OK;
  };
  const long iters0 = 2000;
  float ms = 0.f;
  int st = run(iters0, &ms);
  if (st == VT_OK) st = run(iters0, &ms);
  long iters = iters0;
  if (st == VT_OK) {
    const double want = seconds * 1e3 / (ms > 1e-3f ? ms : 1e-3f) * (double)iters0;
    iters = want > 4e9 ? 4000000000L : (long)want;
    if (iters < iters0) iters = iters0;
    st = run(iters, &ms);
  }
  if (st == VT_OK) {
    const int per_iter = PROBE_COLS / n_tile;                  // instructions per k-step
    *tops = 2.0 * OBM * (double)(per_iter * n_tile) * OBK * (double)grid * (double)iters / (ms * 1e-3) / 1e12;
    if (clocks_per_mma) {
      long long c = 0;
      VT_CUDA(cudaMemcpy(&c, clk, 8, cudaMemcpyDeviceToHost));
      *clocks_per_mma = (double)c / ((double)iters * per_iter * (OBK / O_UMMA_K));
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(clk);
  return st;
}

}  // namespace vt
extern "C" int vt_debug_ogemm_timing(unsigned long long* out8) {
  unsigned long long* b = vt::ogemm_timing_buffer_public();
  if (!b) return 1;
  if (cudaMemcpy(out8, b, 64, cudaMemcpyDeviceToHost) != cudaSuccess) return 2;
  cudaMemset(b, 0, 64);
  return 0;
}
namespace vt {

int ogemm_launch(int M, int N, int K, const int8_t* A, long lda, long a_slice_stride, const int8_t* B, long ldb,
                 long b_slice_stride, int nslices, double alpha, const double* rowscale, const double* colscale, double* C,
                 long ldc, cudaStream_t stream) {
  VT_REQUIRE(K <= OZAKI_MAX_K, "ogemm: K = %d exceeds %d (INT32 accumulation bound)", K, OZAKI_MAX_K);
  return ogemm_launch_opts(M, N, K, A, lda, a_slice_stride, B, ldb, b_slice_stride, nslices, alpha, rowscale, colscale, C,
                           ldc, OLaunchOpts{}, stream);
}

namespace {
// Rows of X (N x D) against a D x D matrix A on the INT8 engine, chunk by chunk: A is sliced once, chunk c of X
// (ozaki_chunk_rows rows from row c (ch - overlap), scale tau_n * fold[n]; fold == nullptr: tau_n) into one of two
// digit buffers, and product(r0, rows, Bs, tau, o) runs the GEMM of the chunk with the slicing job `o.next` of the
// chunk after it.  The last chunk is the first that reaches row N.
// Chunk c + 1 is sliced by the converter warps of the GEMM of chunk c (rows of up to 1024 elements; longer rows:
// a separate slicing launch per chunk).
struct RowChunks {
  long ld, ch;
  size_t a_bytes, sigma_bytes, b_bytes, tau_bytes;
  RowChunks(long N, int D, int nslices)
      : ld((D + 15) / 16 * 16), ch(ozaki_chunk_rows(N, D, nslices)), a_bytes(align_up((size_t)nslices * D * ld, 256)),
        sigma_bytes(align_up((size_t)D * 8, 256)), b_bytes(align_up((size_t)nslices * ch * ld, 256)),
        tau_bytes(align_up((size_t)ch * 8, 256)) {}
  size_t bytes() const { return a_bytes + sigma_bytes + 2 * (b_bytes + tau_bytes); }
};

template <class Product>
int ozaki_row_chunks(const double* A, long lda, const double* X, long ldx, long N, int D, const double* fold,
                     int nslices, long overlap, void* workspace, cudaStream_t stream, Product&& product) {
  const RowChunks rc(N, D, nslices);
  const long ld = rc.ld, ch = rc.ch, stride = ch - overlap;
  VT_REQUIRE(ch == N || stride > 0, "ozaki_row_chunks: chunks of %ld rows cannot overlap by %ld", ch, overlap);
  char* w = static_cast<char*>(workspace);
  int8_t* As = reinterpret_cast<int8_t*>(w);
  w += rc.a_bytes;
  double* sigma = reinterpret_cast<double*>(w);
  w += rc.sigma_bytes;
  int8_t* Bs[2];
  double* tau[2];
  for (int b = 0; b < 2; ++b) {
    Bs[b] = reinterpret_cast<int8_t*>(w);
    w += rc.b_bytes;
    tau[b] = reinterpret_cast<double*>(w);
    w += rc.tau_bytes;
  }
  int st = ozaki_slice(A, lda, D, D, As, ld, (long)D * ld, nslices, sigma, nullptr, stream);
  if (st != VT_OK) return st;
  const bool fuse = D <= 1024;
  long c = 0;
  for (long r0 = 0;; r0 += stride, ++c) {
    const int b = (int)(c & 1);
    const long rows = (N - r0 < ch) ? N - r0 : ch;
    const bool last = r0 + ch >= N;
    if (!fuse || c == 0) {
      st = ozaki_slice(X + r0 * ldx, ldx, rows, D, Bs[b], ld, ch * ld, nslices, tau[b], fold ? fold + r0 : nullptr, stream);
      if (st != VT_OK) return st;
    }
    OLaunchOpts o;
    const long n0 = r0 + stride;
    if (fuse && !last) {
      const long nrows = (N - n0 < ch) ? N - n0 : ch;
      o.next = SliceJob{X + n0 * ldx, ldx, nrows, D, Bs[b ^ 1], ld, ch * ld, tau[b ^ 1], fold ? fold + n0 : nullptr,
                        nullptr, nullptr};
    }
    st = product(r0, rows, As, sigma, Bs[b], tau[b], ld, ch, o);
    if (st != VT_OK) return st;
    if (last) break;
  }
  return VT_OK;
}

// out[n] = sum of the 4 tiles_m partial sums of squares of column n, in a fixed order (no atomics: two calls give
// the same bits).
__global__ void __launch_bounds__(256) quad_forms_finish_kernel(const double* __restrict__ P, int nparts, long ldp,
                                                                long rows, double* __restrict__ out) {
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= rows) return;
  double v = 0.0;
  for (int p = 0; p < nparts; ++p) v += P[(long)p * ldp + n];
  out[n] = v;
}
}  // namespace

size_t ij_apply_ozaki_workspace_bytes(long N, int D, int nslices) { return RowChunks(N, D, nslices).bytes(); }

int ij_apply_ozaki(const double* Hinv, long ldh, const double* X, long ldx, long N, int D, const double* resid,
                   double* S, long lds, int nslices, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Hinv && X && resid && S && workspace, "ij_apply_ozaki: null pointer");
  VT_REQUIRE(D >= 1 && D <= OZAKI_MAX_K && N >= 0 && ldh >= D && ldx >= D && lds >= N, "ij_apply_ozaki: bad shape");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES, "ij_apply_ozaki: 5, 6 or 7 slices");
  VT_REQUIRE(workspace_bytes >= ij_apply_ozaki_workspace_bytes(N, D, nslices), "ij_apply_ozaki: workspace too small");
  if (N == 0) return VT_OK;
  // tau_n resid_n: the residual is folded into the column scale
  return ozaki_row_chunks(Hinv, ldh, X, ldx, N, D, resid, nslices, 0, workspace, stream,
                          [&](long r0, long rows, const int8_t* As, const double* sigma, const int8_t* Bs,
                              const double* tau, long ld, long ch, const OLaunchOpts& o) {
                            return ogemm_launch_opts(D, (int)rows, D, As, ld, (long)D * ld, Bs, ld, ch * ld, nslices,
                                                     -1.0, sigma, tau, S + r0, lds, o, stream);
                          });
}

// ---- out[n] = |Linv x_n|^2 ---------------------------------------------------
size_t quad_forms_ozaki_workspace_bytes(long N, int D, int nslices) {
  const RowChunks rc(N, D, nslices);
  return rc.bytes() + align_up((size_t)4 * ((D + OBM - 1) / OBM) * rc.ch * 8, 256);
}

int quad_forms_ozaki(const double* Linv, long ldl, const double* X, long ldx, long N, int D, double* out, int nslices,
                     void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Linv && X && out && workspace, "quad_forms_ozaki: null pointer");
  VT_REQUIRE(D >= 1 && D <= OZAKI_MAX_K && N >= 0 && ldl >= D && ldx >= D, "quad_forms_ozaki: bad shape");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES, "quad_forms_ozaki: 5, 6 or 7 slices");
  VT_REQUIRE(workspace_bytes >= quad_forms_ozaki_workspace_bytes(N, D, nslices), "quad_forms_ozaki: workspace too small");
  if (N == 0) return VT_OK;
  const RowChunks rc(N, D, nslices);
  double* P = reinterpret_cast<double*>(static_cast<char*>(workspace) + rc.bytes());    // (4 tiles_m) x ch partials
  const int nparts = 4 * ((D + OBM - 1) / OBM);
  return ozaki_row_chunks(Linv, ldl, X, ldx, N, D, nullptr, nslices, 0, workspace, stream,
                          [&](long r0, long rows, const int8_t* As, const double* sigma, const int8_t* Bs,
                              const double* tau, long ld, long ch, OLaunchOpts o) {
                            o.epi = EPI_QUAD;
                            o.tri = 1;          // Linv is lower triangular (the caller's contract)
                            int st = ogemm_launch_opts(D, (int)rows, D, As, ld, (long)D * ld, Bs, ld, ch * ld, nslices,
                                                       1.0, sigma, tau, P, ch, o, stream);
                            if (st != VT_OK) return st;
                            quad_forms_finish_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, stream>>>(P, nparts, ch,
                                                                                                          rows, out + r0);
                            VT_LAUNCH_CHECK();
                            return VT_OK;
                          });
}

// ---- leave-one-group-out -------------------------------------------------------
size_t group_loo_ozaki_workspace_bytes(long N, int D, int nslices) {
  const RowChunks rc(N, D, nslices);
  return rc.bytes() + align_up((size_t)D * rc.ch * 8, 256);
}

int group_loo_ozaki(const double* Linv, long ldl, const double* X, long ldx, long N, int D, const int64_t* starts,
                    long G, const double* s, const double* u, const double* z, int method, double* zpred, double* h,
                    int nslices, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  VT_REQUIRE(Linv && X && starts && s && u && z && zpred && h && workspace, "group_loo_ozaki: null pointer");
  VT_REQUIRE(D >= 1 && D <= OZAKI_MAX_K && N >= 0 && G >= 0 && G <= N && ldl >= D && ldx >= D,
             "group_loo_ozaki: bad shape");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES, "group_loo_ozaki: 5, 6 or 7 slices");
  VT_REQUIRE(method == GROUP_LOO_IJ || method == GROUP_LOO_NS, "group_loo_ozaki: method 0 (IJ) or 1 (Newton step)");
  VT_REQUIRE(workspace_bytes >= group_loo_ozaki_workspace_bytes(N, D, nslices), "group_loo_ozaki: workspace too small");
  if (N == 0) return VT_OK;
  const RowChunks rc(N, D, nslices);
  double* U = reinterpret_cast<double*>(static_cast<char*>(workspace) + rc.bytes());    // D x ch: U = Linv X_c^T
  return ozaki_row_chunks(Linv, ldl, X, ldx, N, D, nullptr, nslices, GROUP_LOO_OVERLAP, workspace, stream,
                          [&](long r0, long rows, const int8_t* As, const double* sigma, const int8_t* Bs,
                              const double* tau, long ld, long ch, const OLaunchOpts& o) {
                            int st = ogemm_launch_opts(D, (int)rows, D, As, ld, (long)D * ld, Bs, ld, ch * ld, nslices,
                                                       1.0, sigma, tau, U, ch, o, stream);
                            if (st != VT_OK) return st;
                            const long stride = ch - GROUP_LOO_OVERLAP;
                            const long hi = (r0 + ch >= N) ? N : r0 + stride;
                            return group_loo_chunk(GroupLooChunk{U, 1, ch, r0, rows, D, starts, G, r0, hi, s, u, z,
                                                                 method, zpred, h}, stream);
                          });
}

// ---- H = X^T diag(s) X -----------------------------------------------------
namespace {
struct SyrkPlan {
  int parts;
  long chunk, ld;
  size_t slices_bytes, cmax_bytes, scale_bytes, sq_bytes, part_bytes;
};
SyrkPlan syrk_plan(long N, int D, int nslices) {
  SyrkPlan p;
  const int tiles_m = (D + OBM - 1) / OBM, tiles_n = (D + OBN - 1) / OBN;
  long ntiles = 0;
  for (int tm = 0; tm < tiles_m; ++tm) ntiles += o_lower_cols(tm, tiles_n);
  int parts = (int)(num_sms() / ntiles);
  if (parts < 1) parts = 1;
  if (parts > 16) parts = 16;
  p.parts = parts;
  long chunk = (long)parts * OZAKI_MAX_K;                       // every part accumulates at most 16384 observations in INT32
  const size_t budget = (size_t)320 << 20;                      // all slices of one chunk
  const long by_mem = (long)(budget / ((size_t)nslices * D)) / (parts * OBK) * (parts * OBK);
  if (by_mem >= (long)parts * OBK && by_mem < chunk) chunk = by_mem;
  if (chunk > N) chunk = N;
  p.chunk = chunk;
  p.ld = (chunk + 15) / 16 * 16;
  p.slices_bytes = align_up((size_t)nslices * D * p.ld, 256);
  p.cmax_bytes = align_up((size_t)D * 8, 256);
  p.scale_bytes = align_up((size_t)D * 8, 256);
  p.sq_bytes = align_up((size_t)N * 8, 256);
  p.part_bytes = align_up((size_t)parts * D * D * 8, 256);
  return p;
}
}  // namespace

size_t syrk_ozaki_workspace_bytes(long N, int D, int nslices) {
  const SyrkPlan p = syrk_plan(N, D, nslices);
  return 2 * p.slices_bytes + p.cmax_bytes + p.scale_bytes + p.sq_bytes + p.part_bytes;
}

int syrk_ozaki(const double* X, long ldx, long N, int D, const double* s, double* H, long ldh, int nslices,
               const double* sq_in, const unsigned long long* colmax_in, void* workspace, size_t workspace_bytes,
               cudaStream_t stream) {
  VT_REQUIRE(X && H && workspace, "syrk_ozaki: null pointer");
  VT_REQUIRE(D >= 1 && N >= 1 && ldx >= D && ldh >= D, "syrk_ozaki: bad shape");
  VT_REQUIRE(nslices >= OZAKI_MIN_SLICES && nslices <= OZAKI_MAX_SLICES, "syrk_ozaki: 5, 6 or 7 slices");
  VT_REQUIRE(workspace_bytes >= syrk_ozaki_workspace_bytes(N, D, nslices), "syrk_ozaki: workspace too small");
  const SyrkPlan p = syrk_plan(N, D, nslices);
  char* w = static_cast<char*>(workspace);
  int8_t* Xs[2];
  for (int b = 0; b < 2; ++b) {
    Xs[b] = reinterpret_cast<int8_t*>(w);
    w += p.slices_bytes;
  }
  unsigned long long* cmax = reinterpret_cast<unsigned long long*>(w);
  w += p.cmax_bytes;
  double* sigma = reinterpret_cast<double*>(w);
  w += p.scale_bytes;
  double* sq = reinterpret_cast<double*>(w);
  w += p.sq_bytes;
  double* P = reinterpret_cast<double*>(w);
  const long slice_stride = (long)D * p.ld;
  // sqrt of the weights and the per-feature maxima of sqrt(s_n) |x_ni| (the power-of-two scale of each row of X^T
  // is common to all chunks: the error bound is relative to sigma_i sigma_j anyway): taken from the caller when the
  // statistics pass has already produced them (vt_glm_stats_colmax), else one sweep over all of X
  VT_REQUIRE((sq_in == nullptr) == (colmax_in == nullptr), "syrk_ozaki: sq and colmax come together");
  const double* sq_use = sq;
  const unsigned long long* cmax_use = cmax;
  if (colmax_in) {
    sq_use = sq_in;
    cmax_use = colmax_in;
  } else {
    VT_CUDA(cudaMemsetAsync(cmax, 0, (size_t)D * 8, stream));
    long nsteps = (N + 31) / 32;
    const long cap = (long)num_sms() * 8;
    if (!s) sq_use = nullptr;            // unweighted: the slicers skip the multiplication
    ozaki_colmax_kernel<<<(unsigned)(nsteps < cap ? nsteps : cap), 256, 0, stream>>>(X, ldx, N, D, s, s ? sq : nullptr, cmax);
    VT_LAUNCH_CHECK();
  }
  VT_CUDA(cudaMemsetAsync(P, 0, (size_t)p.parts * D * D * 8, stream));      // every chunk (and part) accumulates
  // Chunk c + 1 is sliced by the converter warps of the GEMM of chunk c; only chunk 0 takes a slicing launch.
  auto job = [&](long r0, int b) {
    const long rows = (N - r0 < p.chunk) ? N - r0 : p.chunk;
    return SliceJob{X + r0 * ldx, ldx, rows, D, Xs[b], p.ld, slice_stride, sigma, nullptr, sq_use ? sq_use + r0 : nullptr, cmax_use};
  };
  int st = VT_OK;
  long c = 0;
  for (long r0 = 0; r0 < N; r0 += p.chunk, ++c) {
    const int b = (int)(c & 1);
    const long rows = (N - r0 < p.chunk) ? N - r0 : p.chunk;
    if (c == 0) {
      const SliceJob jb = job(r0, b);
      st = ozaki_slice_t(jb.X, ldx, jb.rows, D, jb.sq, cmax_use, Xs[b], p.ld, slice_stride, nslices, sigma, stream);
      if (st != VT_OK) return st;
    }
    OLaunchOpts o;
    o.lower = 1;
    o.parts = p.parts;
    o.accumulate = 1;
    o.part_stride = (long)D * D;
    if (r0 + p.chunk < N) o.next = job(r0 + p.chunk, b ^ 1);
    st = ogemm_launch_opts(D, D, (int)rows, Xs[b], p.ld, slice_stride, Xs[b], p.ld, slice_stride, nslices, 1.0, sigma, sigma,
                           P, D, o, stream);
    if (st != VT_OK) return st;
  }
  const long total = (long)D * D;
  ozaki_syrk_finish_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(P, p.parts, (long)D * D, D, H, ldh);
  VT_LAUNCH_CHECK();
  return VT_OK;
}

}  // namespace vt
