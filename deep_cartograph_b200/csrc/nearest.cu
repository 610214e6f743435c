// Nearest clustered frame of every supplementary frame (reference traj_cluster_workflow.py:207-238,
// assign_closest_cluster = NearestNeighbors(n_neighbors=1).fit(X).kneighbors(Q)), exact in FP64, O((n + m) d)
// memory, no n x m buffer.
//
// Arithmetic: rdist(q, x) = sum_f (q_f - x_f)^2, features in ascending order, a rounded subtract, multiply and
// add per term (no FMA: the library is built with contraction on, hence the intrinsics), then one __dsqrt_rn:
// the KD-tree's arithmetic (and core_dist_kernel's).  Rule: each query takes the lexicographic minimum of
// (rdist, original frame index), so the answer does not depend on frame order, tiling or pruning.
//
// Three steps:
//   1. Spatial order.  A Morton (Z-order) key of the first min(d, 8) coordinates, each quantised over the joint
//      bounding box of frames and queries; frames and queries are sorted by key (cub::DeviceRadixSort, original
//      indices carried) and gathered into compact ordered FP64 copies.
//   2. Tile boxes.  The ordered frames are cut into tiles of T consecutive frames; box[t] = per-dimension
//      [lo, hi] over all d features.  Each CTA takes the box of its own kQB consecutive ordered queries.
//   3. Search.  A CTA seeds the bests of its queries with the tile at its own position in the frame order
//      (binary search of the keys), then visits every other tile unless the box-to-box lower bound is
//      strictly greater than the largest best rdist of its queries.  A visited tile is staged in shared memory;
//      a query skips it when its own point-to-box bound is strictly greater than its own best.
//
// Why pruning is exact with no margin.  The bound is evaluated with the same rounded operations in the same
// order as rdist, on the per-dimension gaps g_f = max(0, fl(lo_t - hi_q), fl(lo_q - hi_t)).  For a frame x in
// the tile and a query q in the block, lo_t <= x_f and q_f <= hi_q, so fl(lo_t - hi_q) <= fl(x_f - q_f) =
// |fl(q_f - x_f)| whenever it is positive (round-to-nearest is monotone and odd), and likewise on the other
// side; hence g_f <= |fl(q_f - x_f)|, fl(g_f g_f) <= fl(t t), and every partial sum of the bound is <= the
// matching partial sum of rdist (a correctly rounded add is monotone in both operands).  The bound is therefore
// <= the computed rdist of every frame of the tile, bit for bit.  A tile is skipped only when the bound is
// strictly greater than a best already held, so no frame that could win, or tie with a lower index, is skipped.
// The block bound only decreases, so a tile that fails the test once fails it for the rest of the search.
//
// Uniform high-dimensional data defeats the pruning; the search then degrades to the brute-force scan plus
// O(n / T) box tests per query block.  counters[0] counts visited tiles and counters[1] the tiles considered
// (query blocks x tiles), so a caller can report the pruned fraction.
#include <cub/device/device_radix_sort.cuh>
#include <math_constants.h>
#include <climits>
#include "dcg_common.cuh"

namespace dcg {
namespace {

constexpr int kQB = 128;                 // queries of one CTA, one per thread
constexpr int kMaxTile = 256;            // frames of a tile (fewer at large d, see tile_rows)
constexpr int kTileDoubles = 6144;       // 48 KB of staged frame coordinates
constexpr int kKeyDims = 8;              // coordinates that enter the Morton key
constexpr int kPrepThreads = 256;
constexpr int kMaxDim = 8192;          // one staged frame + the query box: 24 d bytes of shared memory

__device__ __forceinline__ void take(double& bv, int& bi, double v, int i) {
  if (v < bv || (v == bv && i < bi)) { bv = v; bi = i; }
}

// Order-preserving map of a finite double to a signed 64-bit integer (atomicMin / atomicMax on the box).
__device__ __forceinline__ long long ordered_key(double x) {
  const long long b = __double_as_longlong(x);
  return b >= 0 ? b : b ^ LLONG_MAX;
}
__device__ __forceinline__ double from_ordered_key(long long k) {
  return __longlong_as_double(k >= 0 ? k : k ^ LLONG_MAX);
}

// Box-to-box lower bound of rdist (see the header).  a: [lo, hi] of d doubles each, b likewise.
__device__ __forceinline__ double box_bound(const double* alo, const double* ahi, const double* blo,
                                            const double* bhi, int d) {
  double s = 0.0;
  for (int f = 0; f < d; ++f) {
    double g = __dsub_rn(blo[f], ahi[f]);
    const double h = __dsub_rn(alo[f], bhi[f]);
    if (h > g) g = h;
    if (g < 0.0) g = 0.0;
    s = __dadd_rn(s, __dmul_rn(g, g));
  }
  return s;
}

// ---- 1. joint bounding box of the key coordinates -------------------------------------------------------------
__global__ void box_init_kernel(long long* box) {
  const int f = threadIdx.x;
  if (f < kKeyDims) { box[f] = LLONG_MAX; box[kKeyDims + f] = LLONG_MIN; }
}

__global__ void __launch_bounds__(kPrepThreads)
bbox_kernel(const double* __restrict__ X, int n, int64_t ldx, const double* __restrict__ Q, int m, int64_t ldq,
            int dk, long long* __restrict__ box) {
  double lo[kKeyDims], hi[kKeyDims];
#pragma unroll
  for (int f = 0; f < kKeyDims; ++f) { lo[f] = CUDART_INF; hi[f] = -CUDART_INF; }
  const int64_t total = (int64_t)n + m;
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < total; r += (int64_t)gridDim.x * blockDim.x) {
    const double* p = r < n ? X + r * ldx : Q + (r - n) * ldq;
#pragma unroll
    for (int f = 0; f < kKeyDims; ++f)
      if (f < dk) { const double v = p[f]; lo[f] = fmin(lo[f], v); hi[f] = fmax(hi[f], v); }
  }
#pragma unroll
  for (int f = 0; f < kKeyDims; ++f) {
    if (f >= dk) break;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[f] = fmin(lo[f], __shfl_xor_sync(0xffffffffu, lo[f], o));
      hi[f] = fmax(hi[f], __shfl_xor_sync(0xffffffffu, hi[f], o));
    }
    if ((threadIdx.x & 31) == 0 && lo[f] <= hi[f]) {
      atomicMin(box + f, ordered_key(lo[f]));
      atomicMax(box + kKeyDims + f, ordered_key(hi[f]));
    }
  }
}

// ---- Morton keys ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kPrepThreads)
morton_kernel(const double* __restrict__ Y, int rows, int64_t ld, int dk, int bits, const long long* __restrict__ box,
              unsigned long long* __restrict__ keys, int* __restrict__ idx) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const double levels = (double)(1ull << bits);
  unsigned long long key = 0;
#pragma unroll
  for (int f = 0; f < kKeyDims; ++f) {
    if (f >= dk) break;
    const double lo = from_ordered_key(box[f]), hi = from_ordered_key(box[kKeyDims + f]);
    const double scale = hi > lo ? levels / (hi - lo) : 0.0;     // inf when hi - lo underflows: clamped below
    const double u = (Y[(int64_t)r * ld + f] - lo) * scale;
    const unsigned long long qv = u >= levels - 1.0 ? (1ull << bits) - 1 : (u > 0.0 ? (unsigned long long)u : 0ull);
    for (int b = 0; b < bits; ++b)      // bit b of coordinate f goes to bit b * dk + (dk - 1 - f) of the key
      key |= ((qv >> b) & 1ull) << (b * dk + dk - 1 - f);
  }
  keys[r] = key;
  idx[r] = r;
}

// ---- ordered compact copies and tile boxes --------------------------------------------------------------------
__global__ void __launch_bounds__(kPrepThreads)
gather_kernel(const double* __restrict__ Y, int64_t ld, int d, const int* __restrict__ perm, int64_t total,
              double* __restrict__ out) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / d;
    const int f = (int)(e - r * d);
    out[e] = Y[(int64_t)perm[r] * ld + f];
  }
}

// box[t] = lo[d] then hi[d] over the frames t*T .. t*T + T - 1 of the ordered copy.
__global__ void __launch_bounds__(kPrepThreads)
tile_box_kernel(const double* __restrict__ Xs, int n, int d, int T, int ntiles, double* __restrict__ box) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= (int64_t)ntiles * d) return;
  const int t = (int)(e / d), f = (int)(e - (int64_t)t * d);
  const int r0 = t * T, r1 = min(n, r0 + T);
  double lo = CUDART_INF, hi = -CUDART_INF;
  for (int r = r0; r < r1; ++r) { const double v = Xs[(int64_t)r * d + f]; lo = fmin(lo, v); hi = fmax(hi, v); }
  box[(int64_t)t * 2 * d + f] = lo;
  box[(int64_t)t * 2 * d + d + f] = hi;
}

// ---- 3. search -----------------------------------------------------------------------------------------------
// DK > 0: d == DK, the query held in registers; DK == 0: any d, the query read from the ordered copy.
// Dynamic shared memory: T * d staged frame coordinates, 2 d doubles of query box, T original frame indices.
template <int DK>
__global__ void __launch_bounds__(kQB)
nearest_search_kernel(const double* __restrict__ Xs, const int* __restrict__ xperm,
                      const unsigned long long* __restrict__ xkeys, int n, const double* __restrict__ Qs,
                      const int* __restrict__ qperm, const unsigned long long* __restrict__ qkeys, int m, int d,
                      int T, int ntiles, const double* __restrict__ tbox, int64_t* __restrict__ index,
                      double* __restrict__ dist, unsigned long long* __restrict__ counters) {
  extern __shared__ double sm[];
  double* tile = sm;
  double* qlo = tile + (size_t)T * d;
  double* qhi = qlo + d;
  int* tidx = (int*)(qhi + d);
  __shared__ double red[kQB / 32];
  __shared__ unsigned s_mask[kQB / 32];
  __shared__ double s_bound;
  __shared__ int s_seed;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q0 = blockIdx.x * kQB;
  const int cntq = min(kQB, m - q0);
  const int qi = q0 + min(tid, cntq - 1);
  const bool valid = tid < cntq;
  const double* qrow = Qs + (int64_t)qi * d;
  const int D = DK > 0 ? DK : d;
  double qreg[DK > 0 ? DK : 1];
  if constexpr (DK > 0) {
#pragma unroll
    for (int f = 0; f < DK; ++f) qreg[f] = qrow[f];
  }

  for (int f = tid; f < d; f += kQB) {
    double lo = CUDART_INF, hi = -CUDART_INF;
    for (int r = 0; r < cntq; ++r) { const double v = Qs[(int64_t)(q0 + r) * d + f]; lo = fmin(lo, v); hi = fmax(hi, v); }
    qlo[f] = lo; qhi[f] = hi;
  }
  if (tid == 0) {                       // the tile at the block's middle query in the frame order
    const unsigned long long key = qkeys[q0 + cntq / 2];
    int a = 0, b = n;
    while (a < b) { const int c = (int)(((unsigned)a + (unsigned)b) >> 1); if (xkeys[c] < key) a = c + 1; else b = c; }
    s_seed = min(a, n - 1) / T;
    s_bound = CUDART_INF;
  }
  double best = CUDART_INF;
  int bi = INT_MAX;
  unsigned long long visited = 0;
  __syncthreads();

  auto visit = [&](int c) {
    const int r0 = c * T, cnt = min(T, n - r0);
    __syncthreads();                    // the previous tile is no longer read
    const double* src = Xs + (int64_t)r0 * d;
    for (int e = tid; e < cnt * d; e += kQB) tile[e] = src[e];
    for (int r = tid; r < cnt; r += kQB) tidx[r] = xperm[r0 + r];
    __syncthreads();
    if (valid) {
      const double* b = tbox + (int64_t)c * 2 * d;
      double lb = 0.0;
#pragma unroll
      for (int f = 0; f < D; ++f) {     // point-to-box bound of this query (the box bound with lo_q = hi_q = q)
        double qf;
        if constexpr (DK > 0) qf = qreg[f]; else qf = qrow[f];
        double g = __dsub_rn(b[f], qf);
        const double h = __dsub_rn(qf, b[d + f]);
        if (h > g) g = h;
        if (g < 0.0) g = 0.0;
        lb = __dadd_rn(lb, __dmul_rn(g, g));
      }
      if (!(lb > best)) {
        for (int r = 0; r < cnt; ++r) {
          const double* y = tile + r * d;
          double s = 0.0;
#pragma unroll
          for (int f = 0; f < D; ++f) {
            double qf;
            if constexpr (DK > 0) qf = qreg[f]; else qf = __ldg(qrow + f);
            const double t = __dsub_rn(qf, y[f]);
            s = __dadd_rn(s, __dmul_rn(t, t));
          }
          take(best, bi, s, tidx[r]);
        }
      }
    }
    double mx = valid ? best : -CUDART_INF;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    if (tid == 0) {
      double v = red[0];
      for (int w = 1; w < kQB / 32; ++w) v = fmax(v, red[w]);
      s_bound = v;
    }
    __syncthreads();
    ++visited;
  };

  const int seed = s_seed;
  visit(seed);
  for (int t0 = 0; t0 < ntiles; t0 += kQB) {
    const int t = t0 + tid;
    const bool cand = t < ntiles && t != seed &&
                      !(box_bound(qlo, qhi, tbox + (int64_t)t * 2 * d, tbox + (int64_t)t * 2 * d + d, d) > s_bound);
    const unsigned mk = __ballot_sync(0xffffffffu, cand);
    if (lane == 0) s_mask[warp] = mk;
    __syncthreads();
    for (int w = 0; w < kQB / 32; ++w) {
      unsigned bits = s_mask[w];
      while (bits) {
        const int c = t0 + w * 32 + __ffs(bits) - 1;
        bits &= bits - 1;
        // every thread evaluates the same bound against the same s_bound, so the branch is uniform
        if (!(box_bound(qlo, qhi, tbox + (int64_t)c * 2 * d, tbox + (int64_t)c * 2 * d + d, d) > s_bound)) visit(c);
      }
    }
    __syncthreads();                    // s_mask is rewritten by the next round
  }
  if (valid) {
    const int o = qperm[qi];
    index[o] = bi;
    dist[o] = __dsqrt_rn(best);
  }
  if (tid == 0) {
    atomicAdd(counters, visited);
    atomicAdd(counters + 1, (unsigned long long)ntiles);
  }
}

// ---- workspace layout ------------------------------------------------------------------------------------------
int tile_rows(int d) { return std::max(1, std::min(kMaxTile, kTileDoubles / d)); }

int key_bits(int dk) { return std::min(21, 63 / dk); }

struct NearLayout {
  size_t counters, box, fkeys, fkeys2, fidx, fidx2, qkeys, qkeys2, qidx, qidx2, Xs, Qs, tbox, temp, temp_bytes, total;
  int T, ntiles;
};

bool near_layout(int64_t n, int64_t m, int d, NearLayout& L) {
  if (n < 1 || m < 0 || d < 1 || d > kMaxDim || n > INT_MAX || m > INT_MAX) return false;
  const int dk = std::min(d, kKeyDims), end_bit = key_bits(dk) * dk;
  size_t ft = 0, qt = 0;
  if (cub::DeviceRadixSort::SortPairs(nullptr, ft, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                      (int*)nullptr, (int*)nullptr, (int)n, 0, end_bit) != cudaSuccess)
    return false;
  if (m > 0 && cub::DeviceRadixSort::SortPairs(nullptr, qt, (unsigned long long*)nullptr,
                                               (unsigned long long*)nullptr, (int*)nullptr, (int*)nullptr, (int)m, 0,
                                               end_bit) != cudaSuccess)
    return false;
  L.T = tile_rows(d);
  L.ntiles = (int)ceil_div(n, L.T);
  size_t o = 0;
  auto take_bytes = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 256); return at; };
  L.counters = take_bytes(2 * sizeof(unsigned long long));
  L.box = take_bytes(2 * kKeyDims * sizeof(long long));
  L.fkeys = take_bytes((size_t)n * sizeof(unsigned long long));
  L.fkeys2 = take_bytes((size_t)n * sizeof(unsigned long long));
  L.fidx = take_bytes((size_t)n * sizeof(int));
  L.fidx2 = take_bytes((size_t)n * sizeof(int));
  L.qkeys = take_bytes((size_t)m * sizeof(unsigned long long));
  L.qkeys2 = take_bytes((size_t)m * sizeof(unsigned long long));
  L.qidx = take_bytes((size_t)m * sizeof(int));
  L.qidx2 = take_bytes((size_t)m * sizeof(int));
  L.Xs = take_bytes((size_t)n * d * sizeof(double));
  L.Qs = take_bytes((size_t)m * d * sizeof(double));
  L.tbox = take_bytes((size_t)L.ntiles * 2 * d * sizeof(double));
  L.temp_bytes = std::max(ft, qt);
  L.temp = take_bytes(L.temp_bytes);
  L.total = o;
  return true;
}

size_t search_smem(int d, int T) { return ((size_t)T * d + 2 * (size_t)d) * sizeof(double) + (size_t)T * sizeof(int); }

}  // namespace
}  // namespace dcg

using namespace dcg;

extern "C" size_t dcg_nearest_frames_workspace_bytes(int64_t n, int64_t m, int d) {
  NearLayout L;
  if (!near_layout(n, m, d, L)) return 0;
  return L.total;
}

extern "C" int dcg_nearest_frames_f64(const double* X, int64_t n, int64_t ldx, const double* Q, int64_t m,
                                      int64_t ldq, int d, int64_t* index, double* dist, void* ws, size_t ws_bytes,
                                      void* stream) {
  if (n < 1 || m < 0 || d < 1 || d > kMaxDim || ldx < d || ldq < d || n > INT_MAX || m > INT_MAX) return DCG_E_SHAPE;
  if (m == 0) return 0;
  if (!X || !Q || !index || !dist) return DCG_E_NULL;
  NearLayout L;
  if (!near_layout(n, m, d, L)) {
    DCG_LAUNCH_CHECK();               // the temporary-storage query failed: report the CUDA error
    return DCG_E_SHAPE;
  }
  if (!ws || ws_bytes < L.total) return DCG_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  auto* counters = (unsigned long long*)(w + L.counters);
  auto* box = (long long*)(w + L.box);
  auto* fkeys = (unsigned long long*)(w + L.fkeys);
  auto* fkeys2 = (unsigned long long*)(w + L.fkeys2);
  auto* qkeys = (unsigned long long*)(w + L.qkeys);
  auto* qkeys2 = (unsigned long long*)(w + L.qkeys2);
  int* fidx = (int*)(w + L.fidx);
  int* fidx2 = (int*)(w + L.fidx2);
  int* qidx = (int*)(w + L.qidx);
  int* qidx2 = (int*)(w + L.qidx2);
  double* Xs = (double*)(w + L.Xs);
  double* Qs = (double*)(w + L.Qs);
  double* tbox = (double*)(w + L.tbox);
  const int ni = (int)n, mi = (int)m;
  const int dk = std::min(d, kKeyDims), bits = key_bits(dk);

  DCG_CUDA_TRY(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long), st));
  box_init_kernel<<<1, 32, 0, st>>>(box);
  DCG_LAUNCH_CHECK();
  const unsigned bgrid = (unsigned)std::min<int64_t>(ceil_div(n + m, kPrepThreads), 8 * kNumSMs);
  bbox_kernel<<<bgrid, kPrepThreads, 0, st>>>(X, ni, ldx, Q, mi, ldq, dk, box);
  DCG_LAUNCH_CHECK();
  morton_kernel<<<(unsigned)ceil_div(n, kPrepThreads), kPrepThreads, 0, st>>>(X, ni, ldx, dk, bits, box, fkeys, fidx);
  DCG_LAUNCH_CHECK();
  morton_kernel<<<(unsigned)ceil_div(m, kPrepThreads), kPrepThreads, 0, st>>>(Q, mi, ldq, dk, bits, box, qkeys, qidx);
  DCG_LAUNCH_CHECK();
  size_t tb = L.temp_bytes;
  DCG_CUDA_TRY(cub::DeviceRadixSort::SortPairs(w + L.temp, tb, fkeys, fkeys2, fidx, fidx2, ni, 0, bits * dk, st));
  tb = L.temp_bytes;
  DCG_CUDA_TRY(cub::DeviceRadixSort::SortPairs(w + L.temp, tb, qkeys, qkeys2, qidx, qidx2, mi, 0, bits * dk, st));
  const unsigned ggrid = 32 * kNumSMs;
  gather_kernel<<<ggrid, kPrepThreads, 0, st>>>(X, ldx, d, fidx2, n * d, Xs);
  DCG_LAUNCH_CHECK();
  gather_kernel<<<ggrid, kPrepThreads, 0, st>>>(Q, ldq, d, qidx2, m * d, Qs);
  DCG_LAUNCH_CHECK();
  tile_box_kernel<<<(unsigned)ceil_div((int64_t)L.ntiles * d, kPrepThreads), kPrepThreads, 0, st>>>(
      Xs, ni, d, L.T, L.ntiles, tbox);
  DCG_LAUNCH_CHECK();

  const size_t smem = search_smem(d, L.T);
  const unsigned grid = (unsigned)ceil_div(m, kQB);
  auto run = [&](auto kernel) -> int {
    DCG_CUDA_TRY(ensure_dynamic_smem((const void*)kernel, smem));
    kernel<<<grid, kQB, smem, st>>>(Xs, fidx2, fkeys2, ni, Qs, qidx2, qkeys2, mi, d, L.T, L.ntiles, tbox, index, dist,
                                    counters);
    DCG_LAUNCH_CHECK();
    return 0;
  };
  switch (d) {
    case 1: return run(nearest_search_kernel<1>);
    case 2: return run(nearest_search_kernel<2>);
    case 3: return run(nearest_search_kernel<3>);
    case 4: return run(nearest_search_kernel<4>);
    default: return run(nearest_search_kernel<0>);
  }
}
