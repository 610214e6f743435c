// Exact silhouette of L labelings of the same frames in one pass over all frame pairs (scikit-learn's
// silhouette_samples / silhouette_score with the Euclidean metric, reference statistics.py:75), FP64,
// O(n (d + L)) memory: no n x n or chunk x n buffer.
//
// Semantics, per labeling (labels encoded 0..k-1): a_i = (sum of d(i, j) over i's own cluster) / (n_own - 1),
// b_i = min over the other clusters c of (sum of d(i, j) over c) / |c|, s_i = (b_i - a_i) / max(a_i, b_i), and
// NaN -> 0 (singletons, and a = b = 0 when duplicate frames are split across clusters); the score is the mean.
//
// Arithmetic: d(i, j) = sqrt(sum_f (x_f - y_f)^2), features in ascending order, a rounded subtract, multiply and
// add per term (no FMA: the library is built with contraction on, hence the intrinsics), then one __dsqrt_rn:
// the pdist arithmetic of linkage.cu and nearest.cu.  Every distance is computed once and feeds every labeling.
//
// Work split.  A CTA owns kRows consecutive rows i, one per thread, and streams every frame j (coordinates, the
// change mask and the slot codes of its L labels) through shared memory, in frame order.  Thread i keeps one
// FP64 accumulator per (labeling, cluster) slot in shared memory (K = sum_l k_l slots) and, per labeling, one
// running register sum: consecutive frames of a CV trajectory mostly share a cluster, so d(i, j) is added to the
// running sum and the sum is flushed into its slot only when that labeling's label changes.  All threads of a
// warp see the same j, so the flush branch is warp-uniform.  Each labeling tracks its own runs (never keyed on
// the whole label tuple), so a labeling's sums, s_i and score are bitwise the same whether it is scored alone or
// with others.  Each cluster sum of m terms is a sum of non-negative distances, within m u / (1 - m u) of exact.
//
// Finish.  Each thread turns its slots into a_i, b_i and s_i per labeling, writes s_i to the optional per-frame
// output, and the CTA adds its s_i in a fixed order into a per-CTA partial; a second launch adds the partials in
// a fixed order.  No floating-point atomics: the results are bitwise reproducible from run to run.
//
// Labels outside 0..k_l - 1 (or offsets outside 0..K) never index a slot: the prep kernel counts them per
// labeling, their frames contribute to no slot, and that labeling's score (and the s_i of those frames) is NaN.
#include <math_constants.h>
#include <climits>
#include "dcg_common.cuh"

namespace dcg {
namespace {

constexpr int kRows = 64;                // rows i of one CTA, one per thread
constexpr int kMaxTile = 64;             // frames of a staged tile (fewer at large d)
constexpr int kTileDoubles = 2048;       // 16 KB of staged frame coordinates
constexpr int kUnroll = 4;               // independent distances in flight per thread
constexpr int kPrepThreads = 256;
constexpr int kReduceThreads = 256;
constexpr int kMaxSlots = DCG_SILHOUETTE_MAX_SLOTS;
constexpr int kMaxLabelings = DCG_SILHOUETTE_MAX_LABELINGS;
constexpr int kMaxDim = 2048;
constexpr unsigned kNoSlot = 0xFFFFu;

// ---- 1. slot codes and change masks ---------------------------------------------------------------------------
// codes[j * L + l] = offsets[l] + label of frame j in labeling l (kNoSlot when out of range, counted in bad[l]);
// bit l of mask[j] is set when labeling l's label of frame j differs from that of frame j - 1 (mask[0] = 0).
__global__ void __launch_bounds__(kPrepThreads)
sil_prep_kernel(const int* __restrict__ labels, int n, int L, const int* __restrict__ offsets, int K,
                uint16_t* __restrict__ codes, unsigned* __restrict__ mask, int* __restrict__ bad) {
  const int j = blockIdx.x * kPrepThreads + threadIdx.x;
  if (j >= n) return;
  unsigned m = 0;
  for (int l = 0; l < L; ++l) {
    const int o0 = offsets[l], o1 = offsets[l + 1];
    const int* lab = labels + (int64_t)l * n;
    const int v = lab[j];
    const bool ok = o0 >= 0 && o1 <= K && v >= 0 && v < o1 - o0;
    if (!ok) atomicAdd(bad + l, 1);
    codes[(int64_t)j * L + l] = (uint16_t)(ok ? o0 + v : kNoSlot);
    if (j > 0 && lab[j - 1] != v) m |= 1u << l;
  }
  mask[j] = m;
}

// ---- 2. the pass over all pairs ---------------------------------------------------------------------------------
template <int DK>
__device__ __forceinline__ double pair_dist(const double* xr, const double* __restrict__ xrow, const double* y, int d) {
  double s = 0.0;
  if constexpr (DK > 0) {
#pragma unroll
    for (int f = 0; f < DK; ++f) {
      const double t = __dsub_rn(xr[f], y[f]);
      s = __dadd_rn(s, __dmul_rn(t, t));
    }
  } else {
    for (int f = 0; f < d; ++f) {
      const double t = __dsub_rn(__ldg(xrow + f), y[f]);
      s = __dadd_rn(s, __dmul_rn(t, t));
    }
  }
  return __dsqrt_rn(s);
}

// Frame r of the tile: flush the running sums of the labelings whose label changes at r, then add the distance.
template <int LT>
__device__ __forceinline__ void take_frame(double dist, unsigned m, const uint16_t* code_r, int L, int K,
                                           double* acc, double (&run)[LT], int (&slot)[LT]) {
  if (m) {                                // warp-uniform: every thread of the CTA is at the same frame
#pragma unroll
    for (int l = 0; l < LT; ++l) {
      if (l < L && ((m >> l) & 1u)) {
        const int s = slot[l];
        if (s < K) acc[s * kRows] = __dadd_rn(acc[s * kRows], run[l]);
        run[l] = 0.0;
        slot[l] = code_r[l];
      }
    }
  }
#pragma unroll
  for (int l = 0; l < LT; ++l)
    if (l < L) run[l] = __dadd_rn(run[l], dist);
}

// DK > 0: d == DK, the own row held in registers; DK == 0: any d, the own row read through the read-only cache.
// LT >= L: the number of running sums held in registers.  Dynamic shared memory: K x kRows slot accumulators,
// T x d staged coordinates, T masks, T x L slot codes.
template <int DK, int LT>
__global__ void __launch_bounds__(kRows)
sil_pass_kernel(const double* __restrict__ Y, int n, int d, int64_t ld, int L, int K, int T,
                const uint16_t* __restrict__ codes, const unsigned* __restrict__ mask,
                const int* __restrict__ offsets, const int* __restrict__ sizes, double* __restrict__ samples,
                double* __restrict__ partial) {
  extern __shared__ double sm[];
  double* acc_all = sm;
  double* tile = acc_all + (size_t)K * kRows;
  unsigned* tmask = (unsigned*)(tile + (size_t)T * d);
  uint16_t* tcode = (uint16_t*)(tmask + T);
  __shared__ double red[kRows / 32];
  const int tid = threadIdx.x;
  const int i = blockIdx.x * kRows + tid;
  const bool valid = i < n;
  const int iv = valid ? i : n - 1;
  const double* xrow = Y + (int64_t)iv * ld;
  double xr[DK > 0 ? DK : 1];
  if constexpr (DK > 0) {
#pragma unroll
    for (int f = 0; f < DK; ++f) xr[f] = xrow[f];
  }
  double* acc = acc_all + tid;            // slot s of this row at acc[s * kRows]: conflict-free across the warp
  for (int s = 0; s < K; ++s) acc[s * kRows] = 0.0;
  double run[LT];
  int slot[LT];
#pragma unroll
  for (int l = 0; l < LT; ++l) {
    run[l] = 0.0;
    slot[l] = l < L ? (int)codes[l] : (int)kNoSlot;
  }

  for (int j0 = 0; j0 < n; j0 += T) {
    const int cnt = min(T, n - j0);
    __syncthreads();                      // the previous tile is no longer read
    for (int e = tid; e < cnt * d; e += kRows) {
      const int r = e / d;
      tile[e] = Y[(int64_t)(j0 + r) * ld + (e - r * d)];
    }
    for (int r = tid; r < cnt; r += kRows) tmask[r] = mask[j0 + r];
    const uint16_t* src = codes + (int64_t)j0 * L;
    for (int e = tid; e < cnt * L; e += kRows) tcode[e] = src[e];
    __syncthreads();
    int r = 0;
    for (; r + kUnroll <= cnt; r += kUnroll) {
      double dist[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) dist[u] = pair_dist<DK>(xr, xrow, tile + (r + u) * d, d);
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) take_frame<LT>(dist[u], tmask[r + u], tcode + (r + u) * L, L, K, acc, run, slot);
    }
    for (; r < cnt; ++r)
      take_frame<LT>(pair_dist<DK>(xr, xrow, tile + r * d, d), tmask[r], tcode + r * L, L, K, acc, run, slot);
  }
#pragma unroll
  for (int l = 0; l < LT; ++l)
    if (l < L && slot[l] < K) acc[slot[l] * kRows] = __dadd_rn(acc[slot[l] * kRows], run[l]);

  // ---- finish: a_i, b_i, s_i per labeling; per-CTA partial sums of s_i in a fixed order ----
  for (int l = 0; l < L; ++l) {
    const int own = codes[(int64_t)iv * L + l];
    double s;
    if (own >= K) {
      s = CUDART_NAN;
    } else {
      const int c0 = max(offsets[l], 0), c1 = min(offsets[l + 1], K);
      const double a = __ddiv_rn(acc[own * kRows], __dsub_rn((double)sizes[own], 1.0));
      double b = CUDART_INF;
      for (int c = c0; c < c1; ++c) {
        if (c == own) continue;
        const double v = __ddiv_rn(acc[c * kRows], (double)sizes[c]);
        if (v < b) b = v;
      }
      s = __ddiv_rn(__dsub_rn(b, a), a > b ? a : b);
      if (s != s) s = 0.0;                // singletons (a = 0/0) and a = b = 0, as sklearn's nan_to_num
    }
    if (valid && samples) samples[(int64_t)l * n + i] = s;
    const double v = warp_sum(valid ? s : 0.0);
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    if (tid == 0) {
      double t = red[0];
      for (int w = 1; w < kRows / 32; ++w) t = __dadd_rn(t, red[w]);
      partial[(int64_t)blockIdx.x * L + l] = t;
    }
    __syncthreads();
  }
}

// ---- 3. the mean: per-CTA partials added in a fixed order ---------------------------------------------------------
__global__ void __launch_bounds__(kReduceThreads)
sil_reduce_kernel(const double* __restrict__ partial, int blocks, int L, int n, const int* __restrict__ bad,
                  double* __restrict__ scores) {
  __shared__ double red[kReduceThreads / 32];
  const int l = blockIdx.x;
  double v = 0.0;
  for (int b = threadIdx.x; b < blocks; b += kReduceThreads) v = __dadd_rn(v, partial[(int64_t)b * L + l]);
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = red[0];
    for (int w = 1; w < kReduceThreads / 32; ++w) t = __dadd_rn(t, red[w]);
    scores[l] = bad[l] > 0 ? CUDART_NAN : __ddiv_rn(t, (double)n);
  }
}

// ---- workspace layout ------------------------------------------------------------------------------------------
int tile_rows(int d) { return std::max(1, std::min(kMaxTile, kTileDoubles / d)); }

bool sil_shape_ok(int64_t n, int d, int L, int K) {
  return n >= 3 && n <= INT_MAX && d >= 1 && d <= kMaxDim && L >= 1 && L <= kMaxLabelings && K >= 2 * L &&
         K <= kMaxSlots;
}

struct SilLayout {
  size_t bad, mask, codes, partial, total;
  int blocks;
};

SilLayout sil_layout(int64_t n, int L) {
  SilLayout S;
  S.blocks = (int)ceil_div(n, kRows);
  size_t o = 0;
  auto take_bytes = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 256); return at; };
  S.bad = take_bytes((size_t)L * sizeof(int));
  S.mask = take_bytes((size_t)n * sizeof(unsigned));
  S.codes = take_bytes((size_t)n * L * sizeof(uint16_t));
  S.partial = take_bytes((size_t)S.blocks * L * sizeof(double));
  S.total = o;
  return S;
}

size_t pass_smem(int d, int L, int K, int T) {
  return ((size_t)K * kRows + (size_t)T * d) * sizeof(double) + (size_t)T * sizeof(unsigned) +
         (size_t)T * L * sizeof(uint16_t);
}

}  // namespace
}  // namespace dcg

using namespace dcg;

extern "C" size_t dcg_silhouette_workspace_bytes(int64_t n, int L, int K) {
  if (!sil_shape_ok(n, 1, L, K)) return 0;
  return sil_layout(n, L).total;
}

extern "C" int dcg_silhouette_f64(const double* Y, int64_t n, int d, int64_t ld, const int32_t* labels, int L,
                                  const int32_t* offsets, const int32_t* sizes, int K, double* scores,
                                  double* samples, void* ws, size_t ws_bytes, void* stream) {
  if (!sil_shape_ok(n, d, L, K) || ld < d) return DCG_E_SHAPE;
  if (!Y || !labels || !offsets || !sizes || !scores) return DCG_E_NULL;
  const SilLayout S = sil_layout(n, L);
  if (!ws || ws_bytes < S.total) return DCG_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  int* bad = (int*)(w + S.bad);
  unsigned* mask = (unsigned*)(w + S.mask);
  uint16_t* codes = (uint16_t*)(w + S.codes);
  double* partial = (double*)(w + S.partial);
  const int ni = (int)n;

  DCG_CUDA_TRY(cudaMemsetAsync(bad, 0, (size_t)L * sizeof(int), st));
  sil_prep_kernel<<<(unsigned)ceil_div(n, kPrepThreads), kPrepThreads, 0, st>>>(labels, ni, L, offsets, K, codes,
                                                                                mask, bad);
  DCG_LAUNCH_CHECK();
  const int T = tile_rows(d);
  const size_t smem = pass_smem(d, L, K, T);
  auto run = [&](auto kernel) -> int {
    DCG_CUDA_TRY(ensure_dynamic_smem((const void*)kernel, smem));
    kernel<<<(unsigned)S.blocks, kRows, smem, st>>>(Y, ni, d, ld, L, K, T, codes, mask, offsets, sizes, samples,
                                                    partial);
    DCG_LAUNCH_CHECK();
    return 0;
  };
  auto by_labelings = [&](auto dk) -> int {
    constexpr int DK = decltype(dk)::value;
    if (L <= 1) return run(sil_pass_kernel<DK, 1>);
    if (L <= 4) return run(sil_pass_kernel<DK, 4>);
    if (L <= 8) return run(sil_pass_kernel<DK, 8>);
    if (L <= 16) return run(sil_pass_kernel<DK, 16>);
    return run(sil_pass_kernel<DK, 32>);
  };
  int rc;
  switch (d) {
    case 1: rc = by_labelings(std::integral_constant<int, 1>()); break;
    case 2: rc = by_labelings(std::integral_constant<int, 2>()); break;
    case 3: rc = by_labelings(std::integral_constant<int, 3>()); break;
    case 4: rc = by_labelings(std::integral_constant<int, 4>()); break;
    default: rc = by_labelings(std::integral_constant<int, 0>()); break;
  }
  if (rc) return rc;
  sil_reduce_kernel<<<(unsigned)L, kReduceThreads, 0, st>>>(partial, S.blocks, L, ni, bad, scores);
  DCG_LAUNCH_CHECK();
  return 0;
}
