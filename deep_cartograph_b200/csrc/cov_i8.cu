// Exact covariance engine (DCG_COV_TC_I8X3): integer tensor cores, TMA-staged operands.
//
//     S0[i,j] = sum_t z_t[i] z_t[j]        St[i,j] = sum_t z_t[i] z_{t+lag}[j]       (reference
//     cv_calculator.py:2244-2261: mlcolvar create_timelagged_dataset + TICA.compute's sums)
//
// The float32 engines (cov_tc.cu) accumulate in FP32 inside the tensor core; at C2 (1M frames x
// 1000 features) their accumulation error (1.6e-6 of the sums) moves the TICA eigenvectors by
// 2.7e-5 -- the eigenvector error is ~1000x the RANDOM part of the relative error of the sums --
// which misses the 1e-5 tolerance.  This engine makes the accumulation EXACT instead:
//
//   1. quantise (one HBM-bound pass, i8_quantize_kernel): every value becomes a 23-bit fixed-point
//      integer  q = rint((x - c_j) * 2^e_j),  c_j = mean_j (so x - c_j is the reference's own float32
//      subtraction, cv_calculator.py:834), 2^e_j the largest power of two that keeps |q| < 2^22 given
//      the column's min / max.  Two integer series are written, each as three balanced base-256
//      digits (int8 planes d0, d1, d2: value = d2 2^16 + d1 2^8 + d0, digits in [-128, 127]) in
//      FEATURE-major, frame-contiguous layout (the K-major operand layout of the contraction):
//          Z: q_t                    U: q_t + q_{t+lag}   (the lagged pair sum, |u| < 2^23)
//   2. contract (cov_i8_kernel): tcgen05.mma.cta_group::2.kind::i8 (int8 x int8 -> int32, exact;
//      twice the FP16 rate) on eight of the nine digit products,
//          A = d2 d2                 (weight 2^32)
//          B = d2 d1 + d1 d2         (weight 2^24)
//          C = d2 d0 + d1 d1 + d0 d2 (weight 2^16)
//          D = d1 d0 + d0 d1         (weight 2^8)         [only d0 d0 is left out: < 2^-30 of the scale.
//             Leaving D out as well costs 4e-9 rms of the sums at M = 1e6 -- and 1.3e-5 in the TICA
//             eigenvectors at C2, measured]
//      into four int32 TMEM accumulators per 256 x N tile (N <= 128: 4 N <= 512 TMEM columns), for up
//      to 32768 frames per work item with no intermediate rounding at all.  Both Grams are symmetric:
//      only tiles that touch the upper triangle are computed,
//          S0 = Z^T Z,      G = U^T U = S0 + S0' + St + St^T      (S0' = S0 shifted by `lag` frames)
//      and the symmetric part of St -- the only part the reference uses: mlcolvar symmetrises C_tau --
//      follows EXACTLY (same integers) as  (St + St^T)/2 = (G - 2 S0 + H - T)/2  with the 2 lag boundary
//      rows H = sum_{t<lag} z z^T, T = sum_{t>=M} z z^T (i8_finish_kernel).  This needs 2 x 20 instead of
//      20 + 28 tiles at F = 1000, and no operand is ever read at a frame offset: TMA boxes must start
//      16-byte aligned in global memory, which an arbitrary lag on 1-byte elements is not (measured:
//      cudaErrorIllegalInstruction, tools_dev/tma_probe.cu).
//      Operands are staged by TMA (cp.async.bulk.tensor, SWIZZLE_128B boxes of 128 frames) straight from
//      the digit planes (128-byte rows: with 64-byte rows the TMA unit, ~2.3 clocks per box row, was the
//      bound): no thread touches an operand.  Warp roles: 0 = TMA producer, 1 = MMA issuer
//      (leader CTA), 2-5 = epilogue (int32 -> FP64: A 2^32 + B 2^24 + C 2^16 is exact in a double,
//      scaled by 2^-e_i 2^-e_j / (range_i range_j), red.global.add.f64).
//
// Error model: the fixed-point rounding of the inputs, |z - z'| <= 2^-23 max|x - c| / range -- the
// float32 resolution of the data -- is unbiased and independent between frames, so its effect on the
// sums is ~ sqrt(2/M) 2^-23: 1e-10 relative at M = 1e6, against a worst case of 1e-6.  The omitted
// d0 d0 product is a bias: every diagonal entry is low by sum d0^2 ~ 5461 M integer units.
// tests/test_cov_i8_exact.py holds the outputs to an exact integer model of this arithmetic.
//
// Frames are processed in windows (the planes of a window live in the caller's workspace).
// Roofline: tensor pipe (kind::i8); HBM for the quantise pass (4 + 6 bytes per element).
#include <cuda.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "dcg_common.cuh"
#include "tc_common.cuh"

namespace dcg {

using namespace tc;

namespace {

constexpr int kTileM = 256;            // tile rows (features I): UMMA M of the CTA pair
constexpr int kHalfM = 128;            // rows staged per CTA
constexpr int kMaxN = 128;             // tile columns (features J): 4 accumulators x N <= 512 TMEM columns
constexpr int kStageFrames = 128;      // frames per pipeline stage = one SWIZZLE_128B box row (a full 128-byte line)
constexpr int kPlaneA = kHalfM * kStageFrames;                 // 8 KB: one digit plane of the A half
constexpr int kMaxItemFrames = 32768;  // int32 headroom: 3 * 128 * 128 * 32768 < 2^31
constexpr int kKSteps = kStageFrames / 32;    // kind::i8 MMAs have K = 32
constexpr int kThreads = 192;          // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int kQMax = 4161536;         // 2^22 - 2^15: |q_t + q_{t+lag}| <= 2^23 - 2^16, top digit in [-127, 127]

__host__ __device__ constexpr int plane_b_bytes(int N) { return (N / 2) * kStageFrames; }
__host__ __device__ constexpr int stage_bytes(int N) { return 3 * kPlaneA + 3 * plane_b_bytes(N); }
inline int num_stages(int N) { return std::min(8, (int)((227 * 1024 - 2048) / stage_bytes(N))); }

struct Tile8 {
  int ia0, ia1;        // first feature of the 128 rows staged by CTA 0 / CTA 1 of the pair (-1: none)
  int j0;              // first feature of the N columns
  int hi;              // one past the last valid feature (block / matrix edge), rows and columns
  int kind;            // 0 = S0 = Z^T Z, 1 = G = U^T U; only the upper triangle (j >= i) is written
  int tr0, tr1;        // the half computes a block BELOW the diagonal and writes its transpose
};

// Work tiles of one symmetric Gram per diagonal region (the whole matrix, or each hTICA block).
// N == 128: the region is a grid of 128 x 128 blocks of which the upper triangle incl. the diagonal is
// needed; a tile pairs two blocks that share their COLUMN block (the B operand of the pair MMA) -- a
// block (r, c) may also be computed as (c, r) and written transposed, so the odd block left over in
// every even column c = 4m (its diagonal block) is paired with the one of column 4m + 2, block (4m, 4m+2),
// computed as (4m+2, 4m): nb (nb + 1) / 2 blocks in ceil(that / 2) tiles (18 instead of 20 at nb = 8, 5
// instead of 6 at nb = 4).  Other N (narrow matrices): 256-row x N tiles that touch the upper triangle.
__host__ __device__ inline int enum_tiles8(int f, int block, int N, bool want_s0, bool want_st, Tile8* out) {
  int n = 0;
  const int w = block > 0 ? block : f;
  for (int b0 = 0; b0 < f; b0 += w) {
    const int b1 = b0 + w < f ? b0 + w : f;
    for (int kind = 0; kind < 2; ++kind) {
      if (!(kind == 0 ? want_s0 : want_st)) continue;
      if (N != kHalfM) {
        for (int i0 = b0; i0 < b1; i0 += kTileM)
          for (int j0 = b0; j0 < b1; j0 += N) {
            if (j0 + N <= i0) continue;
            if (out) out[n] = Tile8{i0, i0 + kHalfM < b1 ? i0 + kHalfM : -1, j0, b1, kind, 0, 0};
            ++n;
          }
        continue;
      }
      const int nb = (b1 - b0 + kHalfM - 1) / kHalfM;
      for (int c = 0; c < nb; ++c) {
        const int skip = (c & 1) ? -1 : ((c & 3) == 0 ? c : c - 2);      // the block left over in an even column
        int first = -1;
        for (int r = 0; r <= c; ++r) {
          if (r == skip) continue;
          if (first < 0) { first = r; continue; }
          if (out) out[n] = Tile8{b0 + first * kHalfM, b0 + r * kHalfM, b0 + c * kHalfM, b1, kind, 0, 0};
          ++n;
          first = -1;
        }
        if ((c & 3) == 0) {            // diagonal block (c, c) + block (c + 2, c), written transposed as (c, c + 2)
          if (out) out[n] = Tile8{b0 + c * kHalfM, c + 2 < nb ? b0 + (c + 2) * kHalfM : -1, b0 + c * kHalfM, b1, kind, 0, 1};
          ++n;
        }
      }
    }
  }
  return n;
}

__global__ void plan8_kernel(Tile8* tiles, int f, int block, int N, bool want_s0, bool want_st) {
  if (threadIdx.x == 0 && blockIdx.x == 0) enum_tiles8(f, block, N, want_s0, want_st, tiles);
}

// ---- per-feature quantisation parameters -----------------------------------------------------------
// shift[j] = c_j, mul[j] = 2^e_j (float), scale[j] = 2^-e_j / range_j (double)
__global__ void i8_prep_kernel(int f, const float* __restrict__ mean, const float* __restrict__ range,
                               const float* __restrict__ xmin, const float* __restrict__ xmax,
                               float* __restrict__ shift, float* __restrict__ mul, double* __restrict__ scale) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= f) return;
  const float c = mean ? mean[j] : 0.f;
  const float r = range ? range[j] : 1.f;
  float amax = fmaxf(fabsf(xmax[j] - c), fabsf(xmin[j] - c));
  if (!(amax > 0.f) || !isfinite(amax)) amax = 1.f;
  // largest power of two with amax * 2^e <= kQMax (one ulp of slack for the float32 subtraction)
  int e = ilogbf((float)kQMax / (amax * 1.0000002f));
  e = e > 100 ? 100 : (e < -100 ? -100 : e);
  if (c != 0.f && isfinite(c)) e = min(e, 120 - ilogbf(c));       // c 2^e stays finite (the fused kernel's single FMA)
  shift[j] = c;
  mul[j] = ldexpf(1.f, e);
  scale[j] = ldexp(1.0, -e) / (double)r;
}

// ---- quantise: X (frames x features, float32) -> int8 digit planes of Z and U, feature-major ---------
constexpr int kQF = 64;     // features per tile
constexpr int kQT = 128;    // frames per tile (one 128-byte line per feature and plane)
constexpr int kQRow = 33;   // words per shared-memory row (128 bytes + 4 padding)

__device__ __forceinline__ int quantize1(float x, float c, float m, int& clamped) {
  const float y = (x - c) * m;                         // the reference's float32 subtraction, then an exact scaling
  clamped += fabsf(y) > (float)kQMax + 0.5f;
  return max(-kQMax, min(kQMax, __float2int_rn(y)));
}

// byte K of a, b, c, d -> one word (a in the lowest byte)
template <int K>
__device__ __forceinline__ uint32_t pack_byte(int a, int b, int c, int d) {
  const uint32_t lo = __byte_perm((uint32_t)a, (uint32_t)b, ((4 + K) << 4) | K);
  const uint32_t hi = __byte_perm((uint32_t)c, (uint32_t)d, ((4 + K) << 4) | K);
  return __byte_perm(lo, hi, 0x5410);
}
// Balanced base-256 digits of an integer q (|q| < 2^23):
//   d0 = byte 0 of q,  d1 = byte 0 of (q + 128) >> 8 = byte 1 of q + 128,
//   d2 = byte 0 of (((q + 128) >> 8) + 128) >> 8 = byte 2 of q + 128 + 32768      (floors nest)
// (digits4_biased below works on q + 0x8080, where all three are plain bytes up to a flipped top bit)

// q + kDigitBias by the float "magic number" rounding (RN-even like __float2int_rn, on the full-rate FP pipe):
// |y| <= kQMax < 2^22, so y + 1.5 2^23 has unit spacing and its mantissa bits are the integer.
constexpr int kDigitBias = 0x8080;
// y = (x - c) 2^e as ONE fused multiply-add, x 2^e - c 2^e: both products are exact (i8_prep_kernel keeps c 2^e
// finite), so the single rounding is the rounding of the reference's float32 subtraction, scaled.
// The symmetric clamp is one instruction (min of the magnitudes, sign of y).
__device__ __forceinline__ float clamp_sym(float y) {
  float r;
  asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(r) : "f"(y), "f"((float)kQMax));
  return r;
}
__device__ __forceinline__ float max3_abs(float a, float y0, float y1) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(fabsf(y0)), "f"(fabsf(y1)));
  return r;
}
__device__ __forceinline__ int quantize_biased(float y) {
  return __float_as_int(clamp_sym(y) + 12582912.f) - (0x4B400000 - kDigitBias);
}
// balanced digits of four biased integers q' = q + 0x8080 (digits4 above adds 128 / 32896 per digit):
//   d0 = byte 0 of q = byte 0 of q' with its top bit flipped, d1 = byte 1 of q + 128 = byte 1 of q' with its top
//   bit flipped, d2 = byte 2 of q + 32896 = byte 2 of q'
__device__ __forceinline__ void digits4_biased(int a, int b, int c, int d, uint32_t& w0, uint32_t& w1, uint32_t& w2) {
  w0 = pack_byte<0>(a, b, c, d) ^ 0x80808080u;
  w1 = pack_byte<1>(a, b, c, d) ^ 0x80808080u;
  w2 = pack_byte<2>(a, b, c, d);
}

// planes: [set (Z, U)][digit 0..2][feature][frame], frame stride 1, feature stride wpad, digit stride
// f * wpad, set stride 3 * f * wpad.  `pairs` frames of the window starting at row `row0` of X.
template <bool WITH_U>
__global__ void __launch_bounds__(256, 3)
i8_quantize_kernel(const float* __restrict__ X, int64_t row0, int64_t pairs, int lag, int f, int64_t ld,
                   const float* __restrict__ shift, const float* __restrict__ mul,
                   int8_t* __restrict__ planes, int64_t wpad, int tiles_per_block,
                   long long* __restrict__ qsum_t, long long* __restrict__ qsum_lag, int* __restrict__ info, int vec4) {
  extern __shared__ __align__(16) unsigned char qsmem[];
  uint32_t (*tile)[kQF][kQRow] = reinterpret_cast<uint32_t (*)[kQF][kQRow]>(qsmem);   // [3 or 6 planes][feature][word]
  __shared__ unsigned long long ssum[2][kQF];
  const int tid = threadIdx.x;
  // 4 features x 4 frames per thread and pass.  A warp covers 8 feature quads x 4 frame quads so that its
  // transposed shared-memory stores (word index 33 * feature + frame quad) hit 32 different banks; its
  // global loads are 128-byte row segments.
  const int fe4 = ((tid >> 5) & 1) * 8 + (tid & 7), frq = (tid >> 6) * 4 + ((tid >> 3) & 3);
  const int f0 = blockIdx.x * kQF;
  const int fc = f0 + 4 * fe4;
  float c[4], m[4];
  bool ok[4];
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    ok[v] = fc + v < f;
    c[v] = ok[v] ? shift[fc + v] : 0.f;
    m[v] = ok[v] ? mul[fc + v] : 0.f;
  }
  if (tid < 2 * kQF) ssum[tid / kQF][tid % kQF] = 0ull;
  long long acc_t[4] = {0, 0, 0, 0}, acc_l[4] = {0, 0, 0, 0};
  int clamped = 0;
  const size_t plane_stride = (size_t)f * (size_t)wpad;
  const size_t lag_off = (size_t)lag * (size_t)ld;
  const int64_t tile0 = (int64_t)blockIdx.y * tiles_per_block;
  for (int tt = 0; tt < tiles_per_block; ++tt) {
    const int64_t t0 = (tile0 + tt) * kQT;               // first frame of the tile (window-local)
    if (t0 >= pairs) break;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      float x[4][4], xl[4][4];                           // [frame r][feature v]
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int64_t t = t0 + 64 * h + 4 * frq + r;
        const float* px = X + (size_t)(row0 + t) * (size_t)ld + fc;
        const bool live = t < pairs;
        if (live && vec4 && ok[3]) {
          const float4 a = ldg_stream4(px);
          x[r][0] = a.x; x[r][1] = a.y; x[r][2] = a.z; x[r][3] = a.w;
          if (WITH_U) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(px + lag_off));
            xl[r][0] = b.x; xl[r][1] = b.y; xl[r][2] = b.z; xl[r][3] = b.w;
          }
        } else {
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            x[r][v] = (live && ok[v]) ? ldg_stream1(px + v) : c[v];
            if (WITH_U) xl[r][v] = (live && ok[v]) ? __ldg(px + lag_off + v) : c[v];
          }
        }
      }
      const int w = 16 * h + frq;
      float amax = 0.f;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        // biased integers q + 0x8080 (quantize_biased), one FMA + clamp + magic-number rounding per value
        int q[4], u[4];
        int ps = 0, pl = 0;                              // |q| < 2^22: four of them fit an int
        const float ncm = -c[v] * m[v];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const float y = fmaf(x[r][v], m[v], ncm);
          q[r] = quantize_biased(y);
          ps += q[r];
          if (WITH_U) {
            const float yl = fmaf(xl[r][v], m[v], ncm);
            amax = max3_abs(amax, y, yl);
            const int ql = quantize_biased(yl);
            pl += ql;
            u[r] = q[r] + ql - kDigitBias;
          } else {
            amax = fmaxf(amax, fabsf(y));
          }
        }
        acc_t[v] += ps - 4 * kDigitBias;
        if (WITH_U) acc_l[v] += pl - 4 * kDigitBias;
        const int fe = 4 * fe4 + v;
        uint32_t w0, w1, w2;
        digits4_biased(q[0], q[1], q[2], q[3], w0, w1, w2);
        tile[0][fe][w] = w0; tile[1][fe][w] = w1; tile[2][fe][w] = w2;
        if (WITH_U) {
          digits4_biased(u[0], u[1], u[2], u[3], w0, w1, w2);
          tile[3][fe][w] = w0; tile[4][fe][w] = w1; tile[5][fe][w] = w2;
        }
      }
      clamped += amax > (float)kQMax + 0.5f;             // groups of 4 x 4 values that held a clamped one
    }
    __syncthreads();
    // (3 or 6) planes x 64 features x 128 bytes -> global, 16 bytes per thread and step, 128-byte lines
#pragma unroll
    for (int it = 0; it < (WITH_U ? 12 : 6); ++it) {
      const int chunk = it * 256 + tid;
      const int p = chunk >> 9, row = (chunk >> 3) & 63, cw = chunk & 7;
      if (f0 + row < f) {
        const uint32_t* src = &tile[p][row][4 * cw];
        const uint4 v4 = make_uint4(src[0], src[1], src[2], src[3]);
        int8_t* dst = planes + (size_t)p * plane_stride + (size_t)(f0 + row) * (size_t)wpad + (size_t)t0 + 16 * cw;
        *reinterpret_cast<uint4*>(dst) = v4;
      }
    }
    __syncthreads();
  }
  if (qsum_t) {
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      atomicAdd(&ssum[0][4 * fe4 + v], (unsigned long long)acc_t[v]);
      if (WITH_U) atomicAdd(&ssum[1][4 * fe4 + v], (unsigned long long)acc_l[v]);
    }
    __syncthreads();
    if (tid < kQF && f0 + tid < f) {
      atomicAdd((unsigned long long*)qsum_t + f0 + tid, ssum[0][tid]);
      if (WITH_U) atomicAdd((unsigned long long*)qsum_lag + f0 + tid, ssum[1][tid]);
    }
  }
  if (clamped && info) atomicAdd(info, clamped);
}

// Finish: column sums from the exact integer totals, and the symmetric part of St from the two Grams.
//   a = sum_{t<M} z_t, b = sum_{t>=lag} z_t = sum_{t<M} z_{t+lag}
//   (St + St^T)/2 = (G - 2 S0 + H - T)/2,  H = sum_{t<lag} z z^T,  T = sum_{t>=M} z z^T  (rows re-quantised
//   here with the same arithmetic, exact integers); written to BOTH triangles of St.  S0 keeps its upper
//   triangle (dcg.h).  Entries outside the diagonal blocks (block mode) are left as they are.
__global__ void i8_finish_sums_kernel(int f, const double* __restrict__ scale, const long long* __restrict__ qsum_t,
                                      const long long* __restrict__ qsum_lag, int lag,
                                      double* __restrict__ sum_t, double* __restrict__ sum_lag) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= f) return;
  if (sum_t) sum_t[j] = (double)qsum_t[j] * scale[j];
  if (sum_lag) sum_lag[j] = (double)(lag > 0 ? qsum_lag[j] : qsum_t[j]) * scale[j];
}

__global__ void __launch_bounds__(256)
i8_finish_st_kernel(const float* __restrict__ X, int64_t n_rows, int f, int64_t ld, int lag, int block,
                    const float* __restrict__ shift, const float* __restrict__ mul, const double* __restrict__ scale,
                    const double* __restrict__ S0, double* __restrict__ St) {
  const int j = blockIdx.x * 16 + (threadIdx.x & 15), i = blockIdx.y * 16 + (threadIdx.x >> 4);
  if (i >= f || j >= f || j < i) return;
  if (block > 0 && i / block != j / block) return;
  const int64_t M = n_rows - lag;
  const float ci = shift[i], mi = mul[i], cj = shift[j], mj = mul[j];
  long long d = 0;                                        // H - T in integer units
  int dummy = 0;
  for (int t = 0; t < lag; ++t) {
    const float* rh = X + (size_t)t * ld;
    const float* rt = X + (size_t)(M + t) * ld;
    d += (long long)quantize1(rh[i], ci, mi, dummy) * quantize1(rh[j], cj, mj, dummy);
    d -= (long long)quantize1(rt[i], ci, mi, dummy) * quantize1(rt[j], cj, mj, dummy);
  }
  const size_t ij = (size_t)i * f + j, ji = (size_t)j * f + i;
  const double v = 0.5 * (St[ij] - 2.0 * S0[ij] + (double)d * scale[i] * scale[j]);
  St[ij] = v;
  St[ji] = v;
}

// ---- contraction ------------------------------------------------------------------------------------
struct Params8 {
  const Tile8* tiles;
  int n_tiles;
  int64_t n_items;       // n_tiles * n_ranges, range-major
  int64_t granule;       // frames per work item (multiple of kStageFrames)
  int64_t pairs;         // lagged pairs in this window
  int N;                 // tile width (multiple of 32, <= kMaxN)
  int n_stages;
  int f;
  double* S0;
  double* St;
  const double* scale;   // per feature: 2^-e / range
  int dbg;               // diagnostics (DCG_I8_DBG): 1 = no TMA, 2 = no MMA, 4 = no TMEM loads
};

__device__ __forceinline__ uint32_t cluster_ctarank8() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync8() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote8(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(rank) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster8(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 4-D tiled TMA load (frame, feature, digit, set) into this CTA's shared memory; completion (bytes) is
// signalled on the barrier at `bar_addr` -- a shared::cluster address, the LEADER CTA's barrier for both
// CTAs of the pair.  The box must start 16-byte aligned in global memory: frame coordinates are
// multiples of 64 here.
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar_addr,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tmem_alloc2_8(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
               ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2_8(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void mma2_i8_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma2_commit_both8(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
// kind::i8 instruction descriptor: signed 8-bit operands, both K-major, int32 accumulate, dense
__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// K-major SWIZZLE_128B operand: rows of 128 bytes, 8-row swizzle atoms of 1024 bytes (= SBO)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t start) {
  uint64_t d = 0;
  d |= (uint64_t)((start >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                 // LBO (unused for swizzled K-major operands)
  d |= (uint64_t)(1024 >> 4) << 32;       // SBO
  d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
  return d;
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
cov_i8_kernel(const __grid_constant__ CUtensorMap map_a,      // planes [set][digit][feature][frame], box 64 x 128
              const __grid_constant__ CUtensorMap map_b,      // same tensor, box 64 x N/2
              const Params8 p) {
  extern __shared__ unsigned char smem_raw8[];
  const uint32_t smem_base = (smem_u32(smem_raw8) + 1023u) & ~1023u;
  __shared__ uint64_t full_bar[8], empty_bar[8], acc_full, acc_empty;
  __shared__ uint32_t tmem_base_s;
  __shared__ double epi_smem[4 * 32 * 9];          // per epilogue warp: 32 rows x 8 columns (+1 padding)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank8();
  const int N = p.N, NS = p.n_stages;
  const uint32_t pb = (uint32_t)plane_b_bytes(N), sb = (uint32_t)stage_bytes(N);

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&acc_full, 1);
    mbar_init(&acc_empty, 2 * 4);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc2_8(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync8();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  uint32_t gs = 0, gi = 0;       // stages / items consumed so far (all roles agree)
  const int64_t cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  for (int64_t item = cluster_id; item < p.n_items; item += n_clusters, ++gi) {
    const int64_t range = item / p.n_tiles;
    const Tile8 td = p.tiles[item - range * p.n_tiles];
    const int64_t f0 = range * p.granule;
    const int64_t f1 = f0 + p.granule < p.pairs ? f0 + p.granule : p.pairs;
    const uint32_t nS = (uint32_t)((f1 - f0 + kStageFrames - 1) / kStageFrames);

    if (warp == 0) {
      // ===================== TMA producer (one lane per CTA) ===========================================
      if (lane == 0) {
        const int set = td.kind;                                   // 0: Z planes (S0), 1: U planes (G)
        // a CTA without a row block stages rows beyond the tensor extent: zero-filled by the TMA unit
        const int ia_t = rank ? td.ia1 : td.ia0;
        const int ia = ia_t < 0 ? p.f : ia_t, jb = td.j0 + (int)rank * (N / 2);
        for (uint32_t s = 0; s < nS; ++s) {
          const uint32_t g = gs + s, slot = g % NS;
          mbar_wait(&empty_bar[slot], ((g / NS) & 1) ^ 1);
          if (p.dbg & 1) { if (rank == 0) mbar_arrive(&full_bar[slot]); continue; }
          // both CTAs' copies complete on the leader's barrier (peer bit of the address cleared)
          const uint32_t bar = smem_u32(&full_bar[slot]) & 0xFEFFFFFFu;
          if (rank == 0) mbar_expect_tx(&full_bar[slot], 2 * sb);
          const uint32_t dst = smem_base + slot * sb;
          // items start at multiples of the stage length; frames at and beyond the window's pair count
          // are zero-filled by the TMA unit (tensor extent), so a last partial stage needs no masking
          const int t = (int)(f0 + (int64_t)s * kStageFrames);
#pragma unroll
          for (int pl = 0; pl < 3; ++pl) tma_load_4d(dst + pl * kPlaneA, &map_a, bar, t, ia, pl, set);
#pragma unroll
          for (int pl = 0; pl < 3; ++pl) tma_load_4d(dst + 3 * kPlaneA + pl * pb, &map_b, bar, t, jb, pl, set);
        }
      }
    } else if (warp == 1) {
      // ===================== MMA issuer (leader CTA) ===================================================
      if (rank == 0) {
        const uint32_t idesc = make_idesc_i8(kTileM, N);
        const uint32_t accA = tmem, accB = tmem + N, accC = tmem + 2 * N, accD = tmem + 3 * N;
        mbar_wait_cluster8(&acc_empty, (gi & 1) ^ 1);
        tc_fence_after();
        for (uint32_t s = 0; s < nS; ++s) {
          const uint32_t g = gs + s, slot = g % NS;
          mbar_wait_cluster8(&full_bar[slot], (g / NS) & 1);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t st = smem_base + slot * sb;
            // planes are stored d0, d1, d2 (plane index = digit index)
            const uint64_t a0 = make_smem_desc_sw128(st), a1 = make_smem_desc_sw128(st + kPlaneA),
                           a2 = make_smem_desc_sw128(st + 2 * kPlaneA);
            const uint32_t sbb = st + 3 * kPlaneA;
            const uint64_t b0 = make_smem_desc_sw128(sbb), b1 = make_smem_desc_sw128(sbb + pb),
                           b2 = make_smem_desc_sw128(sbb + 2 * pb);
#pragma unroll
            for (int h = 0; h < kKSteps && !(p.dbg & 2); ++h) {
              const uint64_t o = (uint64_t)(h * 32 >> 4);            // 32 frames = 32 bytes along K
              const uint32_t first = (s == 0 && h == 0) ? 0u : 1u;
              mma2_i8_ss(accA, a2 + o, b2 + o, idesc, first);
              mma2_i8_ss(accB, a2 + o, b1 + o, idesc, first);
              mma2_i8_ss(accB, a1 + o, b2 + o, idesc, 1u);
              mma2_i8_ss(accC, a2 + o, b0 + o, idesc, first);
              mma2_i8_ss(accC, a1 + o, b1 + o, idesc, 1u);
              mma2_i8_ss(accC, a0 + o, b2 + o, idesc, 1u);
              mma2_i8_ss(accD, a1 + o, b0 + o, idesc, first);
              mma2_i8_ss(accD, a0 + o, b1 + o, idesc, 1u);
            }
            mma2_commit_both8(&empty_bar[slot]);
            if (s + 1 == nS) mma2_commit_both8(&acc_full);
          }
          __syncwarp();
        }
      }
    } else {
      // ===================== epilogue: int32 accumulators -> FP64 result ================================
      const int q = warp & 3;                                  // TMEM lane quarter of this warp
      const uint32_t lane_base = (uint32_t)(q * 32) << 16;
      mbar_wait(&acc_full, gi & 1);
      tc_fence_after();
      // Row `32 q + lane` of this CTA's half of the tile sits in this lane.  The FP64 adds go out 8 columns
      // of 4 rows per instruction (64 contiguous bytes per row) through a small shared-memory transpose:
      // one row per lane would touch 32 different lines per instruction (measured: 20 us per work item).
      const int ia_t = rank ? td.ia1 : td.ia0;
      const bool transposed = (rank ? td.tr1 : td.tr0) != 0;
      const int row0 = ia_t + 32 * q;
      const int gi_row = row0 + lane;
      const bool row_ok = ia_t >= 0 && gi_row < td.hi;
      const double si = row_ok ? p.scale[gi_row] : 0.0;
      double* sE = epi_smem + (warp - 2) * (32 * 9);
      double* outm = td.kind == 0 ? p.S0 : p.St;
      for (int c0 = 0; c0 < N && !(p.dbg & 4) && ia_t >= 0; c0 += 16) {
        uint32_t va[16], vb[16], vc[16], vd[16];
        tmem_ld_x16(tmem + lane_base + c0, va);
        tmem_ld_x16(tmem + N + lane_base + c0, vb);
        tmem_ld_x16(tmem + 2 * N + lane_base + c0, vc);
        tmem_ld_x16(tmem + 3 * N + lane_base + c0, vd);
        tmem_ld_wait();
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int cb = td.j0 + c0 + 8 * half;                   // first column of this group of 8
          if (cb >= td.hi) continue;                               // beyond the edge (warp-uniform)
          if (!transposed && cb + 7 < row0) continue;              // wholly below the diagonal (warp-uniform)
          double v8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int jj = 8 * half + j, gj = cb + j;
            // sum of the digit products down to weight 2^8 (only d0 d0 is left out): an integer below
            // 2^63 whose double is exact to 2^-53 relative
            const double v = (double)(int)va[jj] * 4294967296.0 + (double)(int)vb[jj] * 16777216.0 +
                             (double)(int)vc[jj] * 65536.0 + (double)(int)vd[jj] * 256.0;
            v8[j] = gj < td.hi ? v * si * p.scale[gj] : 0.0;
          }
          if (transposed) {
            // block below the diagonal: entry (gi, gj) goes to (gj, gi); for a fixed column the 32 lanes
            // write 32 consecutive doubles -- coalesced straight from the registers
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (row_ok && cb + j < td.hi) atomicAdd(outm + (size_t)(cb + j) * p.f + gi_row, v8[j]);
            continue;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) sE[lane * 9 + j] = v8[j];
          __syncwarp();
          const int col = lane & 7, gj = cb + col;
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) {
            const int row = 4 * rr + (lane >> 3), gi = row0 + row;
            if (gi < td.hi && gj < td.hi && gj >= gi) atomicAdd(outm + (size_t)gi * p.f + gj, sE[row * 9 + col]);
          }
          __syncwarp();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote8(&acc_empty, 0);
    }
    gs += nS;
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync8();
  if (warp == 1) tmem_dealloc2_8(tmem, 512);
}

// ---- fused quantise + contraction (the default whenever the 128-wide tile plan applies) -------------------
// One persistent kernel; the digit planes never leave L2.  The frames are cut into windows of Wf frames;
// the planes of R consecutive windows live in a ring in global memory that is small enough to stay in L2.
// Every CTA carries, next to the TMA / MMA / epilogue warps of the kernel above, kQuantWarps warps that
// quantise the windows one ring slot ahead of the consumers:
//     quantiser warp:  wait until every cluster has consumed window w - R   (counter done[w % kCtr])
//                      quantise its share of window w into slot w % R        (32 features x 32 frames per item)
//     signalling warp: (one per CTA; the quantisers talk to it through shared memory and never wait for a
//                      device-scope fence themselves)  when the CTA's quantisers are through window w:
//                      fence, release: ready[w % kCtr] += 1
//     TMA producer:    wait until every CTA has released window w (counter ready[w % kCtr]), then
//                      stage its cluster's share of the window exactly as above
//     MMA issuer:      when the last stage of window w has landed: done[w % kCtr] += 1
// The counters are monotonic (target x (w / kCtr + 1)); kCtr >= R makes the modulo safe: a quantiser can only
// reach window w + kCtr after every cluster has consumed window w + kCtr - R >= w.
// Work is TILE-STATIONARY: cluster c owns unit c = (tile, frame split) for the whole launch and accumulates
// it in TMEM across windows; the int32 accumulators are flushed to the FP64 result every 32768 frames.
// n_tiles > clusters: several launches ("rounds"), each quantising only the features its tiles touch.
// All CTAs of the grid must be co-resident (they wait on each other): the host launches no more clusters than
// cudaOccupancyMaxActiveClusters reports.
// Warp roles of the fused kernel, by warpgroup (setmaxnreg works on aligned groups of 4 warps):
//   warps 0-3   TMA producer, MMA issuer, signalling warp, (idle)        32 registers per thread
//   warps 4-7   epilogue (TMEM lane quarter = warp & 3)                   80
//   warps 8-19  quantisers                                               120
// The kernel is launched at 96 registers per thread (640 threads: 61440 registers, the pool setmaxnreg moves
// registers within -- asking for more than the pool holds blocks forever): 128 x (32 + 80) + 384 x 120 = 60416.
constexpr int kQuantWarps = 12;
constexpr int kFirstQuantWarp = 8;
constexpr int kFThreads = 32 * (kFirstQuantWarp + kQuantWarps);
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
constexpr int kCtr = 16;               // counters per direction (>= ring depth)
constexpr int kMaxRing = 8;

struct ParamsF {
  const Tile8* tiles;    // the tiles of this round
  int n_units;           // tiles x S (<= clusters)
  int S;                 // frame splits per tile
  int64_t pairs;         // lagged pairs (M)
  int Wf, R, n_win;      // frames per window, ring depth, windows
  int share_stages;      // stages of 128 frames per unit and window = Wf / S / 128
  int f;
  double* S0;
  double* St;
  const double* scale;
  // quantiser
  const float* X;
  int64_t ld;
  int lag;               // 0: no lagged rows (PCA)
  const float* shift;
  const float* mul;
  int8_t* planes;        // [set][digit][feature][R * Wf]
  int64_t wring;         // bytes per feature row of the ring (allocation stride, >= R * Wf)
  int flo, fhi;          // features this round needs
  int fg0, n_fg;         // first group of 32 features (absolute index) and number of groups
  int lanes;             // quantiser warps per feature group
  int own_lo, own_hi;    // features whose column sums this round accumulates
  int store_z, store_u;
  long long* qsum_t;
  long long* qsum_lag;
  int* info;
  int vec4;
  int ready_target;      // CTAs with at least one active quantiser warp
  int* ready;            // [kCtr]
  int* done;             // [kCtr]
  int dbg;               // diagnostics (DCG_I8_DBG): 1 = quantisers skip their items, 2 = no TMA / MMA, 4 = no fences
};

// spin on a counter with relaxed loads (an acquire load invalidates L1 on every poll); one fence after the wait
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void wait_counter_gpu(const int* p, int target, unsigned ns) {
  while (ld_relaxed_gpu(p) < target) __nanosleep(ns);
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
}
__device__ __forceinline__ void red_release_gpu(int* p) {
  asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(p) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// stages of 128 frames that unit split `split` contracts in window w
__device__ __forceinline__ int win_stages(const ParamsF& p, int w, int split) {
  const int64_t valid = p.pairs - (int64_t)w * p.Wf;                       // > 0; may exceed Wf
  const int64_t rem = (valid < p.Wf ? valid : (int64_t)p.Wf) - (int64_t)split * p.share_stages * kStageFrames;
  if (rem <= 0) return 0;
  const int64_t st = (rem + kStageFrames - 1) / kStageFrames;
  return (int)(st < p.share_stages ? st : p.share_stages);
}

template <bool WITH_LAG>
__device__ __forceinline__ void quantize_window_item(const ParamsF& p, int w, int ch, int feat, int lane,
                                                     const float (&c)[4], const float (&m)[4], const bool (&in_f)[4],
                                                     const bool (&st_ok)[4], long long (&acc_t)[4],
                                                     long long (&acc_l)[4], int& clamped) {
  const int g = lane >> 3;                                      // group of 8 frames
  const int64_t t0 = (int64_t)w * p.Wf + ch * 32 + 8 * g;       // first pair of this thread
  float x[8][4], xl[8][4];
  const size_t lag_off = (size_t)p.lag * (size_t)p.ld;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t t = t0 + i;
    const bool live = t < p.pairs;
    const float* px = p.X + (size_t)t * (size_t)p.ld + feat;
    if (p.dbg & 32) {
#pragma unroll
      for (int v = 0; v < 4; ++v) { x[i][v] = c[v] + (float)i; xl[i][v] = c[v] - (float)i; }
    } else if (live && p.vec4 && in_f[3]) {
      const float4 a = (p.dbg & 64) ? ldg_stream4(px) : __ldg(reinterpret_cast<const float4*>(px));   // L1-allocating: the lagged rows of the same warp merge in L1
      x[i][0] = a.x; x[i][1] = a.y; x[i][2] = a.z; x[i][3] = a.w;
      if (WITH_LAG) {
        const float4 b = (p.dbg & 64) ? ldg_stream4(px + lag_off) : __ldg(reinterpret_cast<const float4*>(px + ((p.dbg & 16) ? 0 : lag_off)));
        xl[i][0] = b.x; xl[i][1] = b.y; xl[i][2] = b.z; xl[i][3] = b.w;
      }
    } else {
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        x[i][v] = (live && in_f[v]) ? ldg_stream1(px + v) : c[v];
        if (WITH_LAG) xl[i][v] = (live && in_f[v]) ? ldg_stream1(px + lag_off + v) : c[v];
      }
    }
  }
  const size_t plane_stride = (size_t)p.f * (size_t)p.wring;
  const size_t col = (size_t)(w % p.R) * (size_t)p.Wf + (size_t)ch * 32 + 8 * g;
  float amax = 0.f;
  const float ncm[4] = {-c[0] * m[0], -c[1] * m[1], -c[2] * m[2], -c[3] * m[3]};
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    // biased integers q + 0x8080 (quantize_biased): the digit bytes are bytes 0, 1 (top bit flipped) and 2
    int q[8], u[8];
    int ps = 0, pl = 0;                                          // |q| < 2^22: eight of them fit an int
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float y = fmaf(x[i][v], m[v], ncm[v]);
      q[i] = quantize_biased(y);
      ps += q[i];
      if (WITH_LAG) {
        const float yl = fmaf(xl[i][v], m[v], ncm[v]);
        amax = max3_abs(amax, y, yl);
        const int ql = quantize_biased(yl);
        pl += ql;
        u[i] = q[i] + ql - kDigitBias;
      } else {
        amax = fmaxf(amax, fabsf(y));
      }
    }
    acc_t[v] += ps - 8 * kDigitBias;
    if (WITH_LAG) acc_l[v] += pl - 8 * kDigitBias;
    if (!st_ok[v] || (p.dbg & 8)) continue;
    int8_t* dst = p.planes + (size_t)(feat + v) * (size_t)p.wring + col;
    if (p.store_z) {
      uint32_t a0, a1, a2, b0, b1, b2;
      digits4_biased(q[0], q[1], q[2], q[3], a0, a1, a2);
      digits4_biased(q[4], q[5], q[6], q[7], b0, b1, b2);
      *reinterpret_cast<uint2*>(dst) = make_uint2(a0, b0);
      *reinterpret_cast<uint2*>(dst + plane_stride) = make_uint2(a1, b1);
      *reinterpret_cast<uint2*>(dst + 2 * plane_stride) = make_uint2(a2, b2);
    }
    if (WITH_LAG && p.store_u) {
      uint32_t a0, a1, a2, b0, b1, b2;
      digits4_biased(u[0], u[1], u[2], u[3], a0, a1, a2);
      digits4_biased(u[4], u[5], u[6], u[7], b0, b1, b2);
      *reinterpret_cast<uint2*>(dst + 3 * plane_stride) = make_uint2(a0, b0);
      *reinterpret_cast<uint2*>(dst + 4 * plane_stride) = make_uint2(a1, b1);
      *reinterpret_cast<uint2*>(dst + 5 * plane_stride) = make_uint2(a2, b2);
    }
  }
  clamped += amax > (float)kQMax + 0.5f;                        // groups of 8 x 4 values that held a clamped one
}

template <bool WITH_LAG>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFThreads, 1)
cov_i8_fused_kernel(const __grid_constant__ CUtensorMap map_a,      // ring [set][digit][feature][frame], box 128 x 128
                    const __grid_constant__ CUtensorMap map_b,      // same tensor, box 128 x 64
                    const ParamsF p) {
  extern __shared__ unsigned char smem_raw8f[];
  const uint32_t smem_base = (smem_u32(smem_raw8f) + 1023u) & ~1023u;
  __shared__ uint64_t full_bar[8], empty_bar[8], acc_full, acc_empty;
  __shared__ uint32_t tmem_base_s;
  __shared__ double epi_smem[4 * 32 * 9];
  __shared__ int q_cnt[kCtr];          // quantiser warps of this CTA that are through window w (slot w % kCtr, monotonic)
  __shared__ int q_can_write;          // last window whose ring slot may be written

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank8();
  constexpr int N = kMaxN;
  constexpr uint32_t pb = (uint32_t)plane_b_bytes(N), sb = (uint32_t)stage_bytes(N);
  constexpr int NS = 3;

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&acc_full, 1);
    mbar_init(&acc_empty, 2 * 4);
    fence_barrier_init();
    for (int i = 0; i < kCtr; ++i) q_cnt[i] = 0;
    q_can_write = p.R - 1;
  }
  if (warp == 1) tmem_alloc2_8(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync8();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  const int unit = (int)(blockIdx.x >> 1);
  const bool has_unit = unit < p.n_units;
  const int split = has_unit ? unit % p.S : 0;
  Tile8 td = p.tiles[has_unit ? unit / p.S : 0];
  const int max_acc = kMaxItemFrames / kStageFrames;             // stages per int32 accumulation

  const int n_qw = p.n_fg * p.lanes;                               // active quantiser warps of the grid
  const int qw0 = (int)blockIdx.x * kQuantWarps;
  const int n_act = n_qw - qw0 < 0 ? 0 : (n_qw - qw0 > kQuantWarps ? kQuantWarps : n_qw - qw0);   // ... of this CTA

  if (warp < 4) {
  setmaxnreg_dec<32>();
  if (warp == 0) {
    // ===================== TMA producer (one lane per CTA) =============================================
    if (lane == 0 && has_unit) {
      const int set = td.kind;
      const int ia_t = rank ? td.ia1 : td.ia0;
      const int ia = ia_t < 0 ? p.f : ia_t, jb = td.j0 + (int)rank * (N / 2);
      const int n_q = p.ready_target;                             // CTAs that release a window
      uint32_t g = 0;
      for (int w = 0; w < p.n_win; ++w) {
        const int nS = win_stages(p, w, split);
        if (nS == 0) continue;
        const int target = n_q * (w / kCtr + 1);
        wait_counter_gpu(p.ready + (w % kCtr), target, 100);
        fence_proxy_async_all();                                  // generic-proxy writes of the quantisers -> TMA reads
        const int base = (w % p.R) * p.Wf + split * p.share_stages * kStageFrames;
        for (int s = 0; s < nS && !(p.dbg & 2); ++s, ++g) {
          const uint32_t slot = g % NS;
          mbar_wait(&empty_bar[slot], ((g / NS) & 1) ^ 1);
          const uint32_t bar = smem_u32(&full_bar[slot]) & 0xFEFFFFFFu;
          if (rank == 0) mbar_expect_tx(&full_bar[slot], 2 * sb);
          const uint32_t dst = smem_base + slot * sb;
          const int t = base + s * kStageFrames;
#pragma unroll
          for (int pl = 0; pl < 3; ++pl) tma_load_4d(dst + pl * kPlaneA, &map_a, bar, t, ia, pl, set);
#pragma unroll
          for (int pl = 0; pl < 3; ++pl) tma_load_4d(dst + 3 * kPlaneA + pl * pb, &map_b, bar, t, jb, pl, set);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================================================
    if (rank == 0 && has_unit) {
      constexpr uint32_t idesc = make_idesc_i8(kTileM, N);
      const uint32_t accA = tmem, accB = tmem + N, accC = tmem + 2 * N, accD = tmem + 3 * N;
      uint32_t g = 0, flushes = 0;
      int acc = 0;
      for (int w = 0; w < p.n_win; ++w) {
        const int nS = win_stages(p, w, split);
        if (acc == 0 && nS > 0) {
          mbar_wait_cluster8(&acc_empty, (flushes & 1) ^ 1);
          tc_fence_after();
        }
        for (int s = 0; s < nS && !(p.dbg & 2); ++s, ++g) {
          const uint32_t slot = g % NS;
          mbar_wait_cluster8(&full_bar[slot], (g / NS) & 1);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t st = smem_base + slot * sb;
            const uint64_t a0 = make_smem_desc_sw128(st), a1 = make_smem_desc_sw128(st + kPlaneA),
                           a2 = make_smem_desc_sw128(st + 2 * kPlaneA);
            const uint32_t sbb = st + 3 * kPlaneA;
            const uint64_t b0 = make_smem_desc_sw128(sbb), b1 = make_smem_desc_sw128(sbb + pb),
                           b2 = make_smem_desc_sw128(sbb + 2 * pb);
#pragma unroll
            for (int h = 0; h < kKSteps; ++h) {
              const uint64_t o = (uint64_t)(h * 32 >> 4);
              const uint32_t first = (acc == 0 && s == 0 && h == 0) ? 0u : 1u;
              mma2_i8_ss(accA, a2 + o, b2 + o, idesc, first);
              mma2_i8_ss(accB, a2 + o, b1 + o, idesc, first);
              mma2_i8_ss(accB, a1 + o, b2 + o, idesc, 1u);
              mma2_i8_ss(accC, a2 + o, b0 + o, idesc, first);
              mma2_i8_ss(accC, a1 + o, b1 + o, idesc, 1u);
              mma2_i8_ss(accC, a0 + o, b2 + o, idesc, 1u);
              mma2_i8_ss(accD, a1 + o, b0 + o, idesc, first);
              mma2_i8_ss(accD, a0 + o, b1 + o, idesc, 1u);
            }
            mma2_commit_both8(&empty_bar[slot]);
          }
          __syncwarp();
        }
        // every load of this cluster from ring slot w % R has landed: the slot may be overwritten
        if (lane == 0) red_release_gpu(p.done + (w % kCtr));
        acc += nS;
        const bool flush = acc > 0 && (w == p.n_win - 1 || acc + p.share_stages > max_acc);
        if (flush) {
          if (elect_one_sync()) mma2_commit_both8(&acc_full);
          __syncwarp();
          ++flushes;
          acc = 0;
        }
      }
    }
  } else if (warp == 2) {
    // ===================== signalling warp of the quantisers ===========================================
      if (lane == 0 && n_act > 0) {
        int wa = p.R, wb = 0;                                      // next window to permit / to release
        while (wb < p.n_win) {
          bool progress = false;
          if (wa < p.n_win) {
            const int wd = wa - p.R;
            if (ld_relaxed_gpu(p.done + (wd % kCtr)) >= p.n_units * (wd / kCtr + 1)) {
              asm volatile("fence.acq_rel.gpu;" ::: "memory");
              *(volatile int*)&q_can_write = wa;
              ++wa;
              progress = true;
            }
          }
          if (*(volatile int*)&q_cnt[wb % kCtr] >= n_act * (wb / kCtr + 1)) {
            if (!(p.dbg & 4)) __threadfence();                     // cumulative: covers the quantisers' stores
            red_release_gpu(p.ready + (wb % kCtr));
            ++wb;
            progress = true;
          }
          if (!progress) __nanosleep(100);
        }
      }
  }
  } else if (warp < kFirstQuantWarp) {
  setmaxnreg_dec<80>();
  {
    // ===================== epilogue: int32 accumulators -> FP64 result ==================================
    if (has_unit) {
      const int q = warp & 3;
      const uint32_t lane_base = (uint32_t)(q * 32) << 16;
      const int ia_t = rank ? td.ia1 : td.ia0;
      const bool transposed = (rank ? td.tr1 : td.tr0) != 0;
      const int row0 = ia_t + 32 * q;
      const int gi_row = row0 + lane;
      const bool row_ok = ia_t >= 0 && gi_row < td.hi;
      const double si = row_ok ? p.scale[gi_row] : 0.0;
      double* sE = epi_smem + (warp - 4) * (32 * 9);
      double* outm = td.kind == 0 ? p.S0 : p.St;
      uint32_t flushes = 0;
      int acc = 0;
      for (int w = 0; w < p.n_win; ++w) {
        acc += win_stages(p, w, split);
        const bool flush = acc > 0 && (w == p.n_win - 1 || acc + p.share_stages > max_acc);
        if (!flush) continue;
        acc = 0;
        mbar_wait(&acc_full, flushes & 1);
        ++flushes;
        tc_fence_after();
        for (int c0 = 0; c0 < N && ia_t >= 0; c0 += 8) {
          const int cb = td.j0 + c0;                               // first column of this group of 8
          if (cb >= td.hi) break;                                  // beyond the edge (warp-uniform)
          if (!transposed && cb + 7 < row0) continue;              // wholly below the diagonal (warp-uniform)
          uint32_t va[8], vb[8], vc[8], vd[8];
          tmem_ld_x8(tmem + lane_base + c0, va);
          tmem_ld_x8(tmem + N + lane_base + c0, vb);
          tmem_ld_x8(tmem + 2 * N + lane_base + c0, vc);
          tmem_ld_x8(tmem + 3 * N + lane_base + c0, vd);
          tmem_ld_wait();
          double v8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int gj = cb + j;
            const double v = (double)(int)va[j] * 4294967296.0 + (double)(int)vb[j] * 16777216.0 +
                             (double)(int)vc[j] * 65536.0 + (double)(int)vd[j] * 256.0;
            v8[j] = gj < td.hi ? v * si * p.scale[gj] : 0.0;
          }
          if (transposed) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (row_ok && cb + j < td.hi) atomicAdd(outm + (size_t)(cb + j) * p.f + gi_row, v8[j]);
            continue;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) sE[lane * 9 + j] = v8[j];
          __syncwarp();
          const int col = lane & 7, gj = cb + col;
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) {
            const int row = 4 * rr + (lane >> 3), gi = row0 + row;
            if (gi < td.hi && gj < td.hi && gj >= gi) atomicAdd(outm + (size_t)gi * p.f + gj, sE[row * 9 + col]);
          }
          __syncwarp();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote8(&acc_empty, 0);
      }
    }
  }
  } else {
  setmaxnreg_inc<120>();
  {
    // ===================== quantisers ===================================================================
    if (qw0 + (warp - kFirstQuantWarp) < n_qw) {
      const int qw = qw0 + (warp - kFirstQuantWarp);
      const int fgi = qw % p.n_fg, ln = qw / p.n_fg;
      const int feat = (p.fg0 + fgi) * 32 + 4 * (lane & 7);
      float c[4], m[4];
      bool in_f[4], st_ok[4], own[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        in_f[v] = feat + v < p.f;
        st_ok[v] = in_f[v] && feat + v >= p.flo && feat + v < p.fhi;
        own[v] = in_f[v] && feat + v >= p.own_lo && feat + v < p.own_hi;
        c[v] = in_f[v] ? p.shift[feat + v] : 0.f;
        m[v] = in_f[v] ? p.mul[feat + v] : 0.f;
      }
      long long acc_t[4] = {0, 0, 0, 0}, acc_l[4] = {0, 0, 0, 0};
      int clamped = 0;
      const int chunks = p.Wf / 32;
      // chunks rotate over the lanes from window to window (the load evens out across windows); frames at and
      // beyond `pairs` are written as zeros up to the end of the last 128-frame stage that is read
      auto live_chunks_of = [&](int w) {
        const int64_t valid = p.pairs - (int64_t)w * p.Wf;
        return valid >= p.Wf ? chunks : (int)((valid + kStageFrames - 1) / kStageFrames) * (kStageFrames / 32);
      };
      auto first_chunk_of = [&](int w) {
        return (int)(((int64_t)ln - ((int64_t)w * chunks) % p.lanes + p.lanes) % p.lanes);
      };
      // L2 prefetch of the rows of the items kPrefetchAhead ahead (one row of 32 features = 128 bytes per lane):
      // with 8 warps per SM, each loading, computing and storing in turn, DRAM latency is otherwise exposed
      const float* pf_base = p.X + (size_t)(p.fg0 + fgi) * 32;
      const int64_t n_rows = p.pairs + p.lag;
      const bool pf_full = (p.fg0 + fgi) * 32 + 31 < p.f;
      auto prefetch_item = [&](int w, int ch) {
        const int64_t row = (int64_t)w * p.Wf + ch * 32 + lane;
        if (row >= n_rows || (p.fg0 + fgi) * 32 >= p.f) return;
        const float* a = pf_base + (size_t)row * (size_t)p.ld;
        if (p.vec4 && pf_full) {
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], 128;" ::"l"(a) : "memory");
        } else {
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
          if (pf_full) asm volatile("prefetch.global.L2 [%0];" ::"l"(a + 31));
        }
      };
      // item cursor: the next (w, ch) of this warp with ch < live(w); w = n_win at the end
      auto next_item = [&](int& w, int& ch) {
        ch += p.lanes;
        while (w < p.n_win && ch >= live_chunks_of(w)) {
          ++w;
          if (w < p.n_win) ch = first_chunk_of(w);
        }
      };
      constexpr int kPrefetchAhead = 2;
      int pw = 0, pch = first_chunk_of(0) - p.lanes;
      next_item(pw, pch);
      for (int i = 0; i < kPrefetchAhead && pw < p.n_win; ++i) {
        prefetch_item(pw, pch);
        next_item(pw, pch);
      }
      for (int w = 0; w < p.n_win; ++w) {
        const int live = live_chunks_of(w);
        if (w >= p.R) {
          while (*(volatile int*)&q_can_write < w) __nanosleep(64);
          __threadfence_block();
        }
        for (int ch = first_chunk_of(w); ch < live && !(p.dbg & 1); ch += p.lanes) {
          if (pw < p.n_win) {
            prefetch_item(pw, pch);
            next_item(pw, pch);
          }
          quantize_window_item<WITH_LAG>(p, w, ch, feat, lane, c, m, in_f, st_ok, acc_t, acc_l, clamped);
        }
        __syncwarp();
        if (lane == 0) {
          __threadfence_block();
          atomicAdd_block(&q_cnt[w % kCtr], 1);
        }
      }
      if (p.qsum_t) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          long long a = acc_t[v], b = acc_l[v];
          a += __shfl_xor_sync(0xffffffffu, a, 8);  a += __shfl_xor_sync(0xffffffffu, a, 16);
          b += __shfl_xor_sync(0xffffffffu, b, 8);  b += __shfl_xor_sync(0xffffffffu, b, 16);
          if (lane < 8 && own[v]) {
            atomicAdd((unsigned long long*)p.qsum_t + feat + v, (unsigned long long)a);
            if (WITH_LAG) atomicAdd((unsigned long long*)p.qsum_lag + feat + v, (unsigned long long)b);
          }
        }
      }
      if (clamped && p.info) atomicAdd(p.info, clamped);
    }
  }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync8();
  if (warp == 1) tmem_dealloc2_8(tmem, 512);
}

// ---- host side ----------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;          // resolved once; the driver entry point is process-wide
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

// planes[2 sets][3 digits][f][wpad] int8; dims (frames, features, digits, sets); box (64 frames, rows, 1, 1)
int make_plane_map(CUtensorMap* map, const int8_t* planes, int64_t frames, int f, int64_t wpad, int n_sets, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return DCG_E_ARCH;
  const cuuint64_t dims[4] = {(cuuint64_t)frames, (cuuint64_t)f, 3, (cuuint64_t)n_sets};
  const cuuint64_t strides[3] = {(cuuint64_t)wpad, (cuuint64_t)wpad * (cuuint64_t)f, (cuuint64_t)wpad * (cuuint64_t)f * 3};
  const cuuint32_t box[4] = {(cuuint32_t)kStageFrames, (cuuint32_t)box_rows, 1, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void*)planes, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : DCG_E_SHAPE;
}

int64_t env_i64(const char* name, int64_t dflt) {
  const char* s = getenv(name);
  return s ? atoll(s) : dflt;
}

// Tile width N (multiple of 32, <= 160).  Wider tiles read less shared memory per MMA (A 4 KB + B N/2 x 32
// bytes per 256 x N x 32 instruction), narrower ones waste less on the diagonal and on the last column
// tile; DCG_I8_N overrides.
int tile_width(int f, int block) {
  const int w = block > 0 ? std::min(block, f) : f;
  const int forced = (int)env_i64("DCG_I8_N", 0);
  if (forced >= 32 && forced <= kMaxN && forced % 32 == 0) return forced;
  int best = 32;
  double best_cost = 1e300;
  for (int N = 32; N <= kMaxN; N += 32) {
    // upper-triangle tiles of one diagonal block x (MMA cycles ~ N) / (shared-memory efficiency)
    int tiles = 0;
    for (int i0 = 0; i0 < w; i0 += kTileM)
      for (int j0 = 0; j0 < w; j0 += N) tiles += j0 + N > i0;
    const double smem_rate = (4096.0 + 32.0 * (N / 2)) / (0.5 * N) + 48.0;     // bytes per clock at full MMA rate
    const double cost = tiles * (double)N * std::max(1.0, smem_rate / 128.0);
    if (cost < best_cost) { best_cost = cost; best = N; }
  }
  return best;
}

// DCG_I8_DEBUG=1: synchronise after every launch and name the failing one on stderr (diagnostics only)
#define DCG_I8_STEP(name)                                                                    \
  do {                                                                                       \
    DCG_LAUNCH_CHECK();                                                                      \
    if (getenv("DCG_I8_DEBUG")) {                                                            \
      cudaError_t _e = cudaStreamSynchronize(st);                                            \
      fprintf(stderr, "[dcg i8] %s: %s\n", name, cudaGetErrorString(_e));                    \
      if (_e != cudaSuccess) return -(int)_e;                                                \
    }                                                                                        \
  } while (0)

// frames per window: the digit planes of a window (3 or 6 bytes per value) stay under ~6 GB
int64_t window_frames(int64_t n_rows, int f, int lag) {
  const int64_t cap = env_i64("DCG_I8_WINDOW_BYTES", (int64_t)6 << 30);
  const int sets = lag > 0 ? 2 : 1;
  int64_t w = std::max<int64_t>(cap / (3 * sets * (int64_t)f), 4096) / 128 * 128;
  return std::min<int64_t>(w, std::max<int64_t>(n_rows - lag, 1));
}

// ---- optional device timing of the two kernels (bench.py's roofline: CUDA events on the launching stream) --
struct Timing8 {
  bool on = false;
  int n = 0;                                 // contraction launches recorded since the last read
  cudaEvent_t q0[64], q1[64], c1[64];        // quantise start / quantise end = contraction start / contraction end
  bool created = false;
};
Timing8 g_timing;                            // diagnostics only: one stream, one thread

struct Layout8 {
  size_t tiles, shift, mul, scale, qsum, counters, planes, total;
  int64_t wf, wpad;
  int n_tiles_max, n_sets;
  bool fused;            // the fused quantise + contraction kernel (ring of digit planes in L2)
  int ring;              // ring depth R
  int64_t ring_budget;   // bytes of digit planes that may be live at once
  int64_t wring;         // bytes per feature row of the ring
};

constexpr int kMaxRounds = 64;
constexpr int kAssumedClusters = 64;   // the fused plan needs at least this many co-resident clusters

// The fused kernel applies to the 128-wide tile plan, and pays off where the contraction is the longer of the two
// phases: its 8 quantiser warps per SM need 4.3 ps per value (the stand-alone quantise kernel, at full occupancy,
// 2.35 ps) against 11 ns per frame and tile-per-cluster for the tensor pipe (measured at C2).  Block-diagonal
// level-1 sums of hTICA (C3: 100 tiles for 4950 features) are quantise-bound and stay on the two-kernel path.
// DCG_I8_FUSED: 0 = never, 1 = by this rule (default), 2 = whenever the plan allows it.
bool fused_applies(int f, int lag, int block) {
  const int64_t mode = env_i64("DCG_I8_FUSED", 1);
  if (mode == 0) return false;
  if (tile_width(f, block) != kHalfM) return false;
  if (ceil_div(f, 32) + 1 > 2 * kAssumedClusters * kQuantWarps) return false;
  const int n_tiles = enum_tiles8(f, block, kHalfM, true, lag > 0, nullptr);
  if (n_tiles > kMaxRounds * kAssumedClusters) return false;
  if (mode >= 2) return true;
  return (double)n_tiles * 35.0 >= (double)f * (lag > 0 ? 1.0 : 0.55);
}

Layout8 layout8(int64_t n_rows, int f, int lag, int block) {
  Layout8 L;
  const int N = tile_width(f, block);
  L.n_tiles_max = enum_tiles8(f, block, N, true, true, nullptr);
  L.n_sets = lag > 0 ? 2 : 1;
  L.fused = fused_applies(f, lag, block);
  L.ring = (int)std::min<int64_t>(std::max<int64_t>(env_i64("DCG_I8_RING", 4), 2), kMaxRing);
  L.ring_budget = std::max<int64_t>(env_i64("DCG_I8_RING_BYTES", (int64_t)36 << 20), 1 << 20);
  L.wring = 0;
  if (L.fused) {
    L.wf = 0;
    // widest window the plan can ask for: one stage per frame split, or the budget on a narrow matrix
    const int one_kind = std::max(1, enum_tiles8(f, block, N, true, false, nullptr));
    const int s_max = std::max(1, (kNumSMs / 2) / std::min(one_kind, kNumSMs / 2));
    const int64_t by_budget = L.ring_budget / (3 * L.n_sets * (int64_t)std::min(f, 1024));
    L.wring = (int64_t)align_up((size_t)std::max<int64_t>((int64_t)L.ring * kStageFrames * s_max, by_budget), 128);
    L.wpad = L.wring;
  } else {
    L.wf = window_frames(n_rows, f, lag);
    L.wpad = (int64_t)align_up((size_t)L.wf, 128);
  }
  size_t o = 256;
  L.tiles = o; o += align_up((size_t)L.n_tiles_max * sizeof(Tile8), 256);
  L.shift = o; o += align_up((size_t)f * 4, 256);
  L.mul = o; o += align_up((size_t)f * 4, 256);
  L.scale = o; o += align_up((size_t)f * 8, 256);
  L.qsum = o; o += align_up((size_t)f * 16, 256);
  L.counters = o; o += align_up((size_t)kMaxRounds * 2 * kCtr * sizeof(int), 256);
  L.planes = align_up(o, 1024); o = L.planes + (size_t)3 * L.n_sets * (size_t)f * (size_t)L.wpad;
  L.total = o + 1024;
  return L;
}

// clusters of the fused kernel that can be resident at once (they wait on each other), per device
int fused_clusters(size_t smem) {
  static int cached[64];
  static bool have[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  if (!have[dev]) {
    int best = kNumSMs / 2;
    for (int v = 0; v < 2; ++v) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(kNumSMs, 1, 1);
      cfg.blockDim = dim3(kFThreads, 1, 1);
      cfg.dynamicSmemBytes = smem;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      int n = 0;
      const void* fn = v ? (const void*)cov_i8_fused_kernel<true> : (const void*)cov_i8_fused_kernel<false>;
      if (cudaOccupancyMaxActiveClusters(&n, fn, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
      best = std::min(best, n);
    }
    cached[dev] = best;
    have[dev] = true;
  }
  return cached[dev];
}

}  // namespace

}  // namespace dcg

using namespace dcg;

extern "C" int dcg_cov_i8_set_timing(int on) {
  if (on && !g_timing.created) {
    for (int i = 0; i < 64; ++i) {
      DCG_CUDA_TRY(cudaEventCreate(&g_timing.q0[i]));
      DCG_CUDA_TRY(cudaEventCreate(&g_timing.q1[i]));
      DCG_CUDA_TRY(cudaEventCreate(&g_timing.c1[i]));
    }
    g_timing.created = true;
  }
  g_timing.on = on != 0;
  g_timing.n = 0;
  return 0;
}

extern "C" int dcg_cov_i8_get_timing(float* quantize_ms, float* contract_ms, int* launches) {
  float q = 0.f, c = 0.f;
  for (int i = 0; i < g_timing.n; ++i) {
    float a = 0.f, b = 0.f;
    DCG_CUDA_TRY(cudaEventSynchronize(g_timing.c1[i]));
    DCG_CUDA_TRY(cudaEventElapsedTime(&a, g_timing.q0[i], g_timing.q1[i]));
    DCG_CUDA_TRY(cudaEventElapsedTime(&b, g_timing.q1[i], g_timing.c1[i]));
    q += a; c += b;
  }
  if (quantize_ms) *quantize_ms = q;
  if (contract_ms) *contract_ms = c;
  if (launches) *launches = g_timing.n;
  g_timing.n = 0;
  return 0;
}

extern "C" size_t dcg_cov_i8_workspace_bytes(int64_t n_rows, int f, int lag, int block) {
  if (n_rows <= 0 || f <= 0 || lag < 0 || lag >= n_rows || block < 0) return 0;
  return layout8(n_rows, f, lag, block).total;
}

extern "C" int dcg_cov_lag_i8_f32(const float* X, int64_t n_rows, int f, int64_t ld, int lag,
                                  const float* mean, const float* range, const float* xmin, const float* xmax,
                                  int block, double* S0, double* St, double* colsum_t, double* colsum_lag,
                                  int* info, void* ws, size_t ws_bytes, void* stream) {
  if (!X || (!S0 && !St) || !xmin || !xmax) return DCG_E_NULL;
  if ((mean == nullptr) != (range == nullptr)) return DCG_E_NULL;
  if (n_rows <= 0 || f <= 0 || ld < f || lag < 0 || lag >= n_rows || block < 0) return DCG_E_SHAPE;
  if (lag == 0) St = nullptr;
  if (St && !S0) return DCG_E_NULL;                  // the symmetric part of St is derived from S0 and G
  const Layout8 L = layout8(n_rows, f, lag, block);
  if (!ws || ws_bytes < L.total) return DCG_E_WORKSPACE;
  int dev = 0, major = 0;
  DCG_CUDA_TRY(cudaGetDevice(&dev));
  DCG_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return DCG_E_ARCH;
  cudaStream_t st = (cudaStream_t)stream;

  char* base = (char*)ws;
  Tile8* d_tiles = (Tile8*)(base + L.tiles);
  float* d_shift = (float*)(base + L.shift);
  float* d_mul = (float*)(base + L.mul);
  double* d_scale = (double*)(base + L.scale);
  long long* d_qsum = (long long*)(base + L.qsum);
  int8_t* d_planes = (int8_t*)(base + L.planes);

  const int64_t M = n_rows - lag;
  const int N = tile_width(f, block);
  const bool with_u = St != nullptr;                 // lag > 0 and the lagged sums are wanted
  const int n_tiles = enum_tiles8(f, block, N, S0 != nullptr, with_u, nullptr);
  if (S0) DCG_CUDA_TRY(cudaMemsetAsync(S0, 0, (size_t)f * f * sizeof(double), st));
  if (St) DCG_CUDA_TRY(cudaMemsetAsync(St, 0, (size_t)f * f * sizeof(double), st));
  if (info) DCG_CUDA_TRY(cudaMemsetAsync(info, 0, sizeof(int), st));
  DCG_CUDA_TRY(cudaMemsetAsync(d_qsum, 0, (size_t)f * 16, st));
  i8_prep_kernel<<<(unsigned)ceil_div(f, 128), 128, 0, st>>>(f, mean, range, xmin, xmax, d_shift, d_mul, d_scale);
  DCG_I8_STEP("prep");
  plan8_kernel<<<1, 32, 0, st>>>(d_tiles, f, block, N, S0 != nullptr, with_u);
  DCG_I8_STEP("plan");

  const bool lag_rows_f = lag > 0;
  if (L.fused) {
    // ---- fused path: per round one persistent launch that quantises and contracts -----------------------
    const size_t fsmem = (size_t)3 * stage_bytes(kMaxN) + 1024;
    DCG_CUDA_TRY(ensure_dynamic_smem((const void*)cov_i8_fused_kernel<true>, fsmem));
    DCG_CUDA_TRY(ensure_dynamic_smem((const void*)cov_i8_fused_kernel<false>, fsmem));
    const int nC = (int)std::min<int64_t>(fused_clusters(fsmem), env_i64("DCG_I8_CLUSTERS", kNumSMs / 2));
    if (nC < 1) return DCG_E_ARCH;
    std::vector<Tile8> tiles((size_t)std::max(n_tiles, 1));
    enum_tiles8(f, block, N, S0 != nullptr, with_u, tiles.data());
    if (ceil_div(n_tiles, nC) > kMaxRounds) return DCG_E_SHAPE;
    int* d_ctr = (int*)(base + L.counters);
    DCG_CUDA_TRY(cudaMemsetAsync(d_ctr, 0, (size_t)kMaxRounds * 2 * kCtr * sizeof(int), st));
    const int vec4f = row_vec_width(X, ld) == 4 ? 1 : 0;
    const bool timedf = g_timing.on && g_timing.n < 64;
    if (timedf) { cudaEventRecord(g_timing.q0[g_timing.n], st); cudaEventRecord(g_timing.q1[g_timing.n], st); }
    int own_from = 0;                                   // column sums: every feature is owned by exactly one round
    const int n_rounds = std::max<int>(1, (int)ceil_div(n_tiles, nC));
    for (int r = 0; r < n_rounds; ++r) {
      const int t0 = r * nC, nt = std::min(nC, n_tiles - t0);
      ParamsF p{};
      int flo = 0, fhi = f, sz = 0, su = 0;
      if (nt > 0) {
        flo = f; fhi = 0;
        for (int i = t0; i < t0 + nt; ++i) {
          const Tile8& t = tiles[(size_t)i];
          const int lo = std::min(t.ia0, t.j0), rows_hi = (t.ia1 >= 0 ? std::max(t.ia0, t.ia1) : t.ia0) + kHalfM;
          flo = std::min(flo, lo);
          fhi = std::max(fhi, std::min(t.hi, std::max(rows_hi, t.j0 + kMaxN)));
          (t.kind == 0 ? sz : su) = 1;
        }
      }
      // the last round also takes the features no tile needs (column sums only: nothing is stored for them)
      const bool last = r == n_rounds - 1;
      const int q_lo = std::min(flo, own_from), q_hi = last ? f : fhi;
      p.tiles = d_tiles + t0;
      p.S = nt > 0 ? std::max(1, nC / nt) : 1;
      p.n_units = std::max(nt, 0) * p.S;
      p.pairs = M;
      p.R = L.ring;
      p.fg0 = q_lo / 32;
      p.n_fg = (int)ceil_div(std::max(q_hi, q_lo + 1), 32) - p.fg0;
      p.lanes = std::max(1, 2 * nC * kQuantWarps / p.n_fg);
      if (p.n_fg > 2 * nC * kQuantWarps) return DCG_E_SHAPE;
      {
        const int64_t unit_frames = (int64_t)kStageFrames * p.S;
        const int64_t by_l2 = L.ring_budget / (3 * (int64_t)L.n_sets * 32 * p.n_fg * p.R);
        int64_t k = std::min<int64_t>(L.wring / p.R, by_l2) / unit_frames;
        k = std::min<int64_t>(k, kMaxItemFrames / kStageFrames);
        k = std::min<int64_t>(k, ceil_div(M, unit_frames));
        k = std::max<int64_t>(k, 1);
        k = std::max<int64_t>(1, env_i64("DCG_I8_WINDOW_STAGES", k));
        p.Wf = (int)(k * unit_frames);
        p.share_stages = (int)k;
        if ((int64_t)p.R * p.Wf > L.wring) return DCG_E_WORKSPACE;
      }
      p.n_win = (int)ceil_div(M, p.Wf);
      p.f = f; p.S0 = S0; p.St = St; p.scale = d_scale;
      p.X = X; p.ld = ld; p.lag = lag; p.shift = d_shift; p.mul = d_mul;
      p.planes = d_planes; p.wring = L.wring;
      p.flo = flo; p.fhi = fhi;
      p.own_lo = own_from; p.own_hi = q_hi;
      own_from = std::max(own_from, q_hi);
      p.store_z = sz; p.store_u = su;
      p.qsum_t = d_qsum; p.qsum_lag = d_qsum + f; p.info = info; p.vec4 = vec4f;
      p.ready = d_ctr + (size_t)r * 2 * kCtr; p.done = p.ready + kCtr;
      p.dbg = (int)env_i64("DCG_I8_DBG", 0);
      p.ready_target = (int)ceil_div((int64_t)p.n_fg * p.lanes, kQuantWarps);
      CUtensorMap ma, mb;
      int rc = make_plane_map(&ma, d_planes, (int64_t)p.R * p.Wf, f, L.wring, L.n_sets, kHalfM);
      if (!rc) rc = make_plane_map(&mb, d_planes, (int64_t)p.R * p.Wf, f, L.wring, L.n_sets, kMaxN / 2);
      if (rc) return rc;
      if (getenv("DCG_I8_DEBUG"))
        fprintf(stderr, "[dcg i8 fused] round %d/%d: tiles %d units %d S %d Wf %d R %d windows %d features [%d,%d) groups %d x lanes %d\n",
                r, n_rounds, nt, p.n_units, p.S, p.Wf, p.R, p.n_win, flo, fhi, p.n_fg, p.lanes);
      // Cooperative launch: the CTAs wait on each other, so the grid must become resident as a whole (two
      // partially resident grids on different streams would otherwise wait for each other's SMs forever).
      {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * nC, 1, 1);
        cfg.blockDim = dim3(kFThreads, 1, 1);
        cfg.dynamicSmemBytes = fsmem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = env_i64("DCG_I8_COOPERATIVE", 1) ? 1 : 0;
        cudaError_t le = lag_rows_f ? cudaLaunchKernelEx(&cfg, cov_i8_fused_kernel<true>, ma, mb, p)
                                    : cudaLaunchKernelEx(&cfg, cov_i8_fused_kernel<false>, ma, mb, p);
        if (le != cudaSuccess && cfg.numAttrs) {           // no cooperative launch of clusters on this driver: plain launch
          if (getenv("DCG_I8_DEBUG")) fprintf(stderr, "[dcg i8 fused] cooperative launch refused (%s): plain launch\n", cudaGetErrorString(le));
          cudaGetLastError();
          cfg.numAttrs = 0;
          le = lag_rows_f ? cudaLaunchKernelEx(&cfg, cov_i8_fused_kernel<true>, ma, mb, p)
                          : cudaLaunchKernelEx(&cfg, cov_i8_fused_kernel<false>, ma, mb, p);
        }
        if (le != cudaSuccess) return -(int)le;
      }
      DCG_I8_STEP("fused");
    }
    if (timedf) cudaEventRecord(g_timing.c1[g_timing.n++], st);
  } else {
  const int ns = num_stages(N);
  const size_t smem = (size_t)ns * stage_bytes(N) + 1024;
  DCG_CUDA_TRY(ensure_dynamic_smem((const void*)cov_i8_kernel, smem));
  DCG_CUDA_TRY(ensure_dynamic_smem((const void*)i8_quantize_kernel<true>, (size_t)6 * kQF * kQRow * 4));
  const int vec4 = row_vec_width(X, ld) == 4 ? 1 : 0;
  const int n_clusters = kNumSMs / 2;
  // the lagged column sum is needed whenever lag > 0, also when only S0 is asked for
  const bool lag_rows = lag > 0;

  for (int64_t w0 = 0; w0 < M; w0 += L.wf) {
    const int64_t pairs = std::min<int64_t>(L.wf, M - w0);
    // ---- quantise the window's pairs [w0, w0 + pairs): Z from row t, U from rows t and t + lag
    const int64_t n_ft = ceil_div(pairs, kQT);
    const int tpb = (int)std::max<int64_t>(1, std::min<int64_t>(32, n_ft / 64));
    dim3 qgrid((unsigned)ceil_div(f, kQF), (unsigned)ceil_div(n_ft, tpb));
    const size_t qsm = (size_t)(lag_rows ? 6 : 3) * kQF * kQRow * 4;
    const bool timed = g_timing.on && g_timing.n < 64;
    if (timed) cudaEventRecord(g_timing.q0[g_timing.n], st);
    if (lag_rows)
      i8_quantize_kernel<true><<<qgrid, 256, qsm, st>>>(X, w0, pairs, lag, f, ld, d_shift, d_mul, d_planes, L.wpad, tpb,
                                                      d_qsum, d_qsum + f, info, vec4);
    else
      i8_quantize_kernel<false><<<qgrid, 256, qsm, st>>>(X, w0, pairs, 0, f, ld, d_shift, d_mul, d_planes, L.wpad, tpb,
                                                       d_qsum, d_qsum + f, info, vec4);
    DCG_I8_STEP("quantize");
    if (timed) cudaEventRecord(g_timing.q1[g_timing.n], st);
    if (n_tiles == 0) continue;
    // ---- contract
    CUtensorMap ma, mb;
    int rc = make_plane_map(&ma, d_planes, pairs, f, L.wpad, L.n_sets, kHalfM);
    if (!rc) rc = make_plane_map(&mb, d_planes, pairs, f, L.wpad, L.n_sets, N / 2);
    if (rc) return rc;
    int64_t g = ceil_div(pairs * n_tiles, (int64_t)n_clusters * 8);
    g = std::min<int64_t>(std::max<int64_t>(ceil_div(g, kStageFrames) * kStageFrames, kStageFrames), kMaxItemFrames);
    g = std::max<int64_t>(kStageFrames, env_i64("DCG_I8_ITEM_FRAMES", g) / kStageFrames * kStageFrames);
    const int64_t n_ranges = ceil_div(pairs, g);
    Params8 p{d_tiles, n_tiles, n_ranges * n_tiles, g, pairs, N, ns, f, S0, St, d_scale,
              (int)env_i64("DCG_I8_DBG", 0)};
    const int nc = (int)std::min<int64_t>(n_clusters, p.n_items);
    cov_i8_kernel<<<2 * nc, kThreads, smem, st>>>(ma, mb, p);
    DCG_I8_STEP("contract");
    if (timed) cudaEventRecord(g_timing.c1[g_timing.n++], st);
  }
  }  // unfused path
  if (colsum_t || colsum_lag) {
    i8_finish_sums_kernel<<<(unsigned)ceil_div(f, 128), 128, 0, st>>>(f, d_scale, d_qsum, d_qsum + f, lag, colsum_t,
                                                                     colsum_lag);
    DCG_I8_STEP("sums");
  }
  if (St) {
    dim3 fg((unsigned)ceil_div(f, 16), (unsigned)ceil_div(f, 16));
    i8_finish_st_kernel<<<fg, 256, 0, st>>>(X, n_rows, f, ld, lag, block, d_shift, d_mul, d_scale, S0, St);
    DCG_I8_STEP("finish");
  }
  return 0;
}
