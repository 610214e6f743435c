// Agglomerative clustering trees, identical to scikit-learn's AgglomerativeClustering (reference
// modules/statistics/statistics.py:285, hierarchical_clustering) for the four linkages it accepts.
//
// complete / average / ward: scipy's nn_chain (scipy/cluster/hierarchy, reached through
// hierarchy.linkage / hierarchy.ward when connectivity is None) on the full FP64 distance matrix:
//   1. linkage_dist_kernel   D[i][j] = sqrt(sum_f (y_i[f] - y_j[f])^2), features in ascending order with a
//                            rounded multiply and a rounded add per term (scipy pdist's arithmetic; the
//                            library is built with FMA contraction on, hence the explicit intrinsics),
//                            square matrix with rows padded to 32 doubles and +inf on the diagonal.
//   2. nn_chain_kernel       the whole merge sequence in ONE launch of one 16-CTA thread-block cluster.
//                            Every CTA owns a strip of columns; a row scan is a strip arg-min, the partials
//                            are exchanged through distributed shared memory and the phases are separated
//                            by barrier.cluster.  Every CTA replays the same chain decisions, so the chain
//                            and the cluster sizes are private to the CTA.  Retired slots are marked by
//                            +inf in their column, so a row scan reads only the row.
// single: scikit-learn's own mst_linkage_core (sklearn/cluster/_hierarchical_fast.pyx): Prim's algorithm
//   from node 0 with the distances computed on the fly (EuclideanDistance.dist, same arithmetic as above):
//   3. prim_kernel           same cluster shape, O(N) memory.
// Finish (both): a stable sort of the merges by distance (numpy mergesort semantics: a rank sort on the
// unique key (distance, merge index)), then the relabelling pass on one thread: scipy's `label`
// (union-find, smaller root first) or sklearn's `_single_linkage_label` (no swap).
//
// HDBSCAN (sklearn.cluster.HDBSCAN, algorithm "auto" on dense Euclidean data = _hdbscan_prims), O(n) memory:
//   4. core_dist_kernel      core[i] = distance from frame i to its min_samples-th nearest frame (itself
//                            included, at 0): a brute-force k-smallest selection with the arithmetic above.
//   3. prim_kernel           with `core` set: sklearn's mst_from_data_matrix, Prim from node 0 on the
//                            mutual-reachability distance max(core[c], core[j], dist(c, j)); each edge is
//                            recorded from the tree node that last strictly improved the new node.
// The edge sort (numpy's default argsort, not stable) and the union-find stay on the host.
#include <cooperative_groups.h>
#include <math_constants.h>
#include <climits>
#include "dcg_common.cuh"

namespace cg = cooperative_groups;

namespace dcg {
namespace {

constexpr int kCtas = 16;        // CTAs of the thread-block cluster that builds the tree (non-portable size)
constexpr int kThreads = 1024;
constexpr int kDistTile = 64;
constexpr int kDistChunk = 16;   // features per shared-memory stage of the distance kernel
constexpr int kSortThreads = 256;
constexpr size_t kPrimStageBytes = 200 * 1024;   // frames of a CTA's strip staged in shared memory up to this

struct Part { double v; int i; };

__device__ __forceinline__ void take(double& bv, int& bi, double v, int i) {
  if (v < bv || (v == bv && i < bi)) { bv = v; bi = i; }
}

// Arg-min over the CTA (lowest index among the minima); the result is valid in thread 0.
__device__ __forceinline__ void cta_argmin(double& bv, int& bi, Part* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_down_sync(0xffffffffu, bv, o);
    const int oi = __shfl_down_sync(0xffffffffu, bi, o);
    take(bv, bi, ov, oi);
  }
  if (lane == 0) red[warp] = Part{bv, bi};
  __syncthreads();
  if (warp == 0) {
    bv = CUDART_INF; bi = INT_MAX;
    if (lane < (int)(blockDim.x >> 5)) { bv = red[lane].v; bi = red[lane].i; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_down_sync(0xffffffffu, bv, o);
      const int oi = __shfl_down_sync(0xffffffffu, bi, o);
      take(bv, bi, ov, oi);
    }
  }
}

// Cluster-wide arg-min of the CTA partials in part[] (call after the cluster barrier); valid in thread 0.
__device__ __forceinline__ Part cluster_argmin(cg::cluster_group& cl, Part* part) {
  double bv = CUDART_INF;
  int bi = INT_MAX;
  const int lane = threadIdx.x & 31;
  if (lane < kCtas) {
    const Part q = *cl.map_shared_rank(part, lane);
    bv = q.v; bi = q.i;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_down_sync(0xffffffffu, bv, o);
    const int oi = __shfl_down_sync(0xffffffffu, bi, o);
    take(bv, bi, ov, oi);
  }
  return Part{bv, bi};
}

__device__ __forceinline__ void strip_of(int n, int rank, int& lo, int& hi) {
  const int s = (n + kCtas - 1) / kCtas;
  lo = min(n, rank * s);
  hi = min(n, lo + s);
}

// ---- 1. all-pairs distances --------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
linkage_dist_kernel(const double* __restrict__ Y, int n, int d, int64_t ld, double* __restrict__ D, int64_t ldD) {
  __shared__ double A[kDistTile][kDistChunk + 1], B[kDistTile][kDistChunk + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i0 = blockIdx.y * kDistTile, j0 = blockIdx.x * kDistTile;
  double acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
  for (int f0 = 0; f0 < d; f0 += kDistChunk) {
    const int fc = min(kDistChunk, d - f0);
    for (int e = threadIdx.x; e < kDistTile * kDistChunk; e += 256) {
      const int r = e / kDistChunk, f = e % kDistChunk;
      A[r][f] = (i0 + r < n && f < fc) ? Y[(int64_t)(i0 + r) * ld + f0 + f] : 0.0;
      B[r][f] = (j0 + r < n && f < fc) ? Y[(int64_t)(j0 + r) * ld + f0 + f] : 0.0;
    }
    __syncthreads();
    for (int f = 0; f < fc; ++f) {
      double a[4], b[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) { a[r] = A[ty + 16 * r][f]; b[r] = B[tx + 16 * r][f]; }
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const double t = __dsub_rn(a[r], b[c]);
          acc[r][c] = __dadd_rn(acc[r][c], __dmul_rn(t, t));
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = i0 + ty + 16 * r;
    if (i >= n) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int j = j0 + tx + 16 * c;
      if (j < ldD) D[(int64_t)i * ldD + j] = (i == j || j >= n) ? CUDART_INF : __dsqrt_rn(acc[r][c]);
    }
  }
}

// ---- 2. NN-chain (complete / average / ward) -----------------------------------------------------------
// Lance-Williams updates of scipy's _hierarchy_distance_update, evaluated left to right without FMA.
__device__ __forceinline__ double lance_williams(int method, double dxi, double dyi, double dxy, int nx, int ny, int ni) {
  if (method == DCG_LINK_COMPLETE) return dxi > dyi ? dxi : dyi;
  if (method == DCG_LINK_AVERAGE)
    return __ddiv_rn(__dadd_rn(__dmul_rn((double)nx, dxi), __dmul_rn((double)ny, dyi)), (double)(nx + ny));
  const double t = __ddiv_rn(1.0, (double)(nx + ny + ni));
  const double a = __dmul_rn(__dmul_rn(__dmul_rn((double)(ni + nx), t), dxi), dxi);
  const double b = __dmul_rn(__dmul_rn(__dmul_rn((double)(ni + ny), t), dyi), dyi);
  const double c = __dmul_rn(__dmul_rn(__dmul_rn((double)ni, t), dxy), dxy);
  return __dsqrt_rn(__dsub_rn(__dadd_rn(a, b), c));
}

// D: n x ldD (overwritten); zraw: (n-1) x 4 merges in chain order (slot x < slot y, distance, size);
// priv: kCtas x 2n ints (each CTA's cluster sizes and chain); phases[0] = row scans, phases[1] = merges.
__global__ void __launch_bounds__(kThreads, 1)
nn_chain_kernel(double* __restrict__ D, int n, int64_t ldD, int method, double* __restrict__ zraw,
                int* __restrict__ priv, long long* __restrict__ phases) {
  cg::cluster_group cl = cg::this_cluster();
  const int rank = (int)cl.block_rank();
  const int tid = threadIdx.x;
  int lo, hi;
  strip_of(n, rank, lo, hi);
  int* size = priv + (size_t)rank * 2 * n;
  int* chain = size + n;
  __shared__ Part red[32];
  __shared__ Part part[2];
  __shared__ int s_x, s_y, s_merge, s_done;
  __shared__ double s_dist;
  for (int i = tid; i < n; i += kThreads) size[i] = 1;
  // chain state: kept by thread 0, identical in every CTA
  int len = 0, x = 0, p = -1, first = 0, k = 0;
  long long scans = 0;
  int par = 0;
  __syncthreads();
  for (;;) {
    if (tid == 0) {
      if (len == 0) { x = first; chain[0] = x; len = 1; p = -1; }
      s_x = x;
    }
    __syncthreads();
    const double* row = D + (int64_t)s_x * ldD;
    double bv = CUDART_INF;
    int bi = INT_MAX;
    for (int j = lo + tid; j < hi; j += kThreads) {
      const double v = __ldcg(row + j);
      if (v < bv) { bv = v; bi = j; }
    }
    cta_argmin(bv, bi, red);
    if (tid == 0) part[par] = Part{bv, bi};
    cl.sync();
    if (tid < 32) {
      const Part q = cluster_argmin(cl, &part[par]);
      if (tid == 0) {
        ++scans;
        int y = q.i;
        double dist = q.v;
        int merge = 0;
        if (len > 1) {
          const double dxp = __ldcg(row + p);
          if (!(q.v < dxp)) { merge = 1; y = p; dist = dxp; }
        }
        if (!merge) {
          if (len == n || y == INT_MAX) merge = -1;     // cannot happen for finite input: stop, not overrun
          else { chain[len++] = y; p = x; x = y; }
        }
        s_y = y; s_dist = dist; s_merge = merge;
      }
    }
    par ^= 1;
    __syncthreads();
    if (s_merge < 0) break;
    if (!s_merge) continue;

    const int a = min(s_x, s_y), b = max(s_x, s_y);
    const int na = size[a], nb = size[b];
    const double dist = s_dist;
    if (rank == 0 && tid == 0) {
      double* z = zraw + (size_t)4 * k;
      z[0] = (double)a; z[1] = (double)b; z[2] = dist; z[3] = (double)(na + nb);
    }
    double* ra = D + (int64_t)a * ldD;
    double* rb = D + (int64_t)b * ldD;
    for (int i = lo + tid; i < hi; i += kThreads) {
      if (i == a) continue;
      if (i == b) { __stcg(rb + a, CUDART_INF); continue; }
      const int ni = size[i];
      if (ni == 0) continue;
      const double v = lance_williams(method, __ldcg(ra + i), __ldcg(rb + i), dist, na, nb, ni);
      __stcg(rb + i, v);
      double* ri = D + (int64_t)i * ldD;
      __stcg(ri + b, v);
      __stcg(ri + a, CUDART_INF);       // slot a is retired: no row scan may find it again
    }
    __syncthreads();
    if (tid == 0) {
      size[a] = 0;
      size[b] = na + nb;
      len -= 2;
      ++k;
      if (len >= 1) { x = chain[len - 1]; p = len >= 2 ? chain[len - 2] : -1; }
      while (first < n && size[first] == 0) ++first;
      s_done = (k == n - 1);
    }
    cl.sync();    // the updated row / columns are visible to every CTA before the next row scan
    if (s_done) break;
  }
  if (rank == 0 && tid == 0) { phases[0] = scans; phases[1] = k; }
  cl.sync();    // no CTA leaves while a peer may still read its partials
}

// ---- 3. Prim (single; HDBSCAN's mutual-reachability MST when core != nullptr) ---------------------------------
// cur: n doubles (distance of every frame to the tree, -1 once in the tree; each CTA touches its strip only).
// core == nullptr: zraw rows of 4, (current node, new node, distance, 0), in visiting order (mst_linkage_core).
// core set: src (n ints) holds the tree node that last strictly improved each frame (sklearn's
//   current_sources); zraw rows of 3, (src[new], new, distance), in visiting order (mst_from_data_matrix).
//   The CTA that owns the new node writes its row, so src is only ever read by the CTA that wrote it.
// phases[0] = phases[1] = steps.
__global__ void __launch_bounds__(kThreads, 1)
prim_kernel(const double* __restrict__ Y, int n, int d, int64_t ld, int stage, const double* __restrict__ core,
            double* __restrict__ cur, int* __restrict__ src, double* __restrict__ zraw,
            long long* __restrict__ phases) {
  extern __shared__ double ysm[];
  cg::cluster_group cl = cg::this_cluster();
  const int rank = (int)cl.block_rank();
  const int tid = threadIdx.x;
  int lo, hi;
  strip_of(n, rank, lo, hi);
  __shared__ Part red[32];
  __shared__ Part part[2];
  __shared__ int s_cur;
  const double* ys = Y + (int64_t)lo * ld;
  int64_t ys_ld = ld;
  if (stage) {
    for (int e = tid; e < (hi - lo) * d; e += kThreads) {
      const int r = e / d, f = e % d;
      ysm[e] = Y[(int64_t)(lo + r) * ld + f];
    }
    ys = ysm;
    ys_ld = d;
  }
  for (int j = lo + tid; j < hi; j += kThreads) cur[j] = CUDART_INF;
  if (core)
    for (int j = lo + tid; j < hi; j += kThreads) src[j] = 1;     // sklearn's np.ones; every frame is set before use
  if (tid == 0) s_cur = 0;
  int par = 0;
  __syncthreads();
  for (int step = 0; step < n - 1; ++step) {
    const int c = s_cur;
    const double* yc = Y + (int64_t)c * ld;
    const double core_c = core ? core[c] : 0.0;
    double bv = CUDART_INF;
    int bi = INT_MAX;
    for (int j = lo + tid; j < hi; j += kThreads) {
      double cj = cur[j];
      if (j == c) { cur[j] = -1.0; continue; }
      if (cj < 0.0) continue;
      const double* yj = ys + (int64_t)(j - lo) * ys_ld;
      double s = 0.0;
      for (int f = 0; f < d; ++f) {
        const double t = __dsub_rn(__ldg(yc + f), yj[f]);
        s = __dadd_rn(s, __dmul_rn(t, t));
      }
      double left = __dsqrt_rn(s);
      if (core) {                                   // Cython's max(core_c, core_j, dist): first of the largest
        double m = core_c;
        const double cj_core = core[j];
        if (cj_core > m) m = cj_core;
        if (left > m) m = left;
        left = m;
        if (left < cj) { cj = left; cur[j] = cj; src[j] = c; }
      } else if (left < cj) {
        cj = left; cur[j] = cj;
      }
      if (cj < bv) { bv = cj; bi = j; }
    }
    cta_argmin(bv, bi, red);
    if (tid == 0) part[par] = Part{bv, bi};
    cl.sync();
    if (tid < 32) {
      const Part q = cluster_argmin(cl, &part[par]);
      if (tid == 0) {
        const int nxt = q.i == INT_MAX ? 0 : q.i;
        if (!core && rank == 0) {
          double* z = zraw + (size_t)4 * step;
          z[0] = (double)c; z[1] = (double)nxt; z[2] = q.v; z[3] = 0.0;
        } else if (core && nxt >= lo && nxt < hi) {
          double* z = zraw + (size_t)3 * step;
          z[0] = (double)src[nxt]; z[1] = (double)nxt; z[2] = q.v;
        }
        s_cur = nxt;
      }
    }
    par ^= 1;
    __syncthreads();
  }
  if (rank == 0 && tid == 0) { phases[0] = n - 1; phases[1] = n - 1; }
  cl.sync();    // no CTA leaves while a peer may still read its partials
}

// ---- 4. HDBSCAN core distances ------------------------------------------------------------------------------
// One warp per query frame, kCoreWarps queries per CTA.  The CTA stages `rows` candidate frames at a time in
// shared memory (row stride lds, odd, so the lanes' 8-byte reads hit distinct banks); lane l scans the tile
// rows l, l + 32, ... and keeps the k smallest squared distances it has seen in a register list of KC >= k
// slots, ascending.  The KC - k bottom slots hold -1 (below every squared distance) and never move, so the
// top slot is the lane's k-th smallest and rejects any candidate that is not below it.  The 32 lane lists
// are then merged by k warp-wide pops of the smallest head; the k-th pop is the query's k-th smallest.
// Only the value is used, so ties among neighbours do not matter.
constexpr int kCoreWarps = 8;
constexpr int kCoreTileDoubles = 6144;          // 48 KB of candidate rows per stage

template <int KC>
__device__ __forceinline__ void topk_insert(double (&lst)[KC], double v) {
#pragma unroll
  for (int t = KC - 1; t > 0; --t) lst[t] = v < lst[t - 1] ? lst[t - 1] : (v < lst[t] ? v : lst[t]);
  lst[0] = v < lst[0] ? v : lst[0];
}

template <int KC>
__global__ void __launch_bounds__(kCoreWarps * 32)
core_dist_kernel(const double* __restrict__ Y, int n, int d, int64_t ld, int k, int rows, int lds,
                 double* __restrict__ core) {
  extern __shared__ double tile[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = blockIdx.x * kCoreWarps + warp;
  const double* yq = Y + (int64_t)min(q, n - 1) * ld;
  double lst[KC];
#pragma unroll
  for (int t = 0; t < KC; ++t) lst[t] = t < KC - k ? -1.0 : CUDART_INF;
  for (int j0 = 0; j0 < n; j0 += rows) {
    const int cnt = min(rows, n - j0);
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * d; e += kCoreWarps * 32) {
      const int r = e / d, f = e % d;
      tile[r * lds + f] = Y[(int64_t)(j0 + r) * ld + f];
    }
    __syncthreads();
    for (int r = lane; r < cnt; r += 32) {
      const double* yj = tile + r * lds;
      double s = 0.0;
      for (int f = 0; f < d; ++f) {
        const double t = __dsub_rn(__ldg(yq + f), yj[f]);
        s = __dadd_rn(s, __dmul_rn(t, t));
      }
      if (s < lst[KC - 1]) topk_insert(lst, s);
    }
  }
  double kth = 0.0;
  for (int p = 0; p < k; ++p) {
    double head = CUDART_INF;
#pragma unroll
    for (int t = KC - 1; t >= 0; --t)
      if (lst[t] >= 0.0) head = lst[t];
    double best = head;
    int who = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int ow = __shfl_xor_sync(0xffffffffu, who, o);
      if (ob < best || (ob == best && ow < who)) { best = ob; who = ow; }
    }
    kth = best;
    if (who == lane) {
      bool done = false;
#pragma unroll
      for (int t = 0; t < KC; ++t)
        if (!done && lst[t] >= 0.0) { lst[t] = -1.0; done = true; }
    }
  }
  if (lane == 0 && q < n) core[q] = __dsqrt_rn(kth);
}

// ---- finish: stable sort by distance + relabelling --------------------------------------------------------
__global__ void __launch_bounds__(kSortThreads)
linkage_sort_kernel(const double* __restrict__ zraw, int m, double* __restrict__ Z) {
  __shared__ double keys[kSortThreads];
  const int i = blockIdx.x * kSortThreads + threadIdx.x;
  const double di = i < m ? zraw[(size_t)4 * i + 2] : 0.0;
  int rank = 0;
  for (int j0 = 0; j0 < m; j0 += kSortThreads) {
    keys[threadIdx.x] = j0 + (int)threadIdx.x < m ? zraw[(size_t)4 * (j0 + threadIdx.x) + 2] : 0.0;
    __syncthreads();
    const int cnt = min(kSortThreads, m - j0);
    for (int jj = 0; jj < cnt; ++jj) {
      const double dj = keys[jj];
      rank += (dj < di) || (dj == di && j0 + jj < i);
    }
    __syncthreads();
  }
  if (i < m) {
#pragma unroll
    for (int c = 0; c < 4; ++c) Z[(size_t)4 * rank + c] = zraw[(size_t)4 * i + c];
  }
}

__device__ __forceinline__ int uf_find(int* parent, int v) {
  int r = v;
  while (parent[r] >= 0) r = parent[r];
  while (v != r) { const int nx = parent[v]; parent[v] = r; v = nx; }
  return r;
}

// Z (sorted, in place): children become union-find roots; node n + i is merge i; column 3 the merged size.
// smaller_first: scipy's `label` (smaller root first); otherwise sklearn's _single_linkage_label order.
__global__ void __launch_bounds__(1024)
linkage_label_kernel(double* __restrict__ Z, int n, int* __restrict__ parent, int* __restrict__ usize, int smaller_first,
                     const long long* __restrict__ phases) {
  if (phases[1] != n - 1) return;     // the tree kernel stopped early: Z is left as it is, the caller reports it
  for (int i = threadIdx.x; i < 2 * n - 1; i += blockDim.x) { parent[i] = -1; usize[i] = i < n ? 1 : 0; }
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (int i = 0; i < n - 1; ++i) {
    double* z = Z + (size_t)4 * i;
    if (!(z[0] >= 0.0 && z[0] < n + i && z[1] >= 0.0 && z[1] < n + i)) return;
    int rx = uf_find(parent, (int)z[0]), ry = uf_find(parent, (int)z[1]);
    const int s = usize[rx] + usize[ry];
    parent[rx] = n + i;
    parent[ry] = n + i;
    usize[n + i] = s;
    if (smaller_first && ry < rx) { const int t = rx; rx = ry; ry = t; }
    z[0] = (double)rx; z[1] = (double)ry; z[3] = (double)s;
  }
}

// ---- workspace layout ---------------------------------------------------------------------------------------
struct LinkLayout { size_t phases, zraw, parent, usize, priv, cur, D, total; int64_t ldD; };

bool link_layout(int64_t n, int method, LinkLayout& L) {
  if (n < 2 || n > (INT_MAX - 1) / 2) return false;
  size_t o = 0;
  auto take_bytes = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 256); return at; };
  L.phases = take_bytes(2 * sizeof(long long));
  L.zraw = take_bytes((size_t)(n - 1) * 4 * sizeof(double));
  L.parent = take_bytes((size_t)(2 * n - 1) * sizeof(int));
  L.usize = take_bytes((size_t)(2 * n - 1) * sizeof(int));
  L.ldD = (int64_t)align_up((size_t)n, 32);
  if (method == DCG_LINK_SINGLE) {
    L.cur = take_bytes((size_t)n * sizeof(double));
    L.priv = L.D = 0;
  } else {
    L.priv = take_bytes((size_t)kCtas * 2 * n * sizeof(int));
    L.D = take_bytes((size_t)n * (size_t)L.ldD * sizeof(double));
    L.cur = 0;
  }
  L.total = o;
  return true;
}

bool valid_method(int m) { return m >= DCG_LINK_SINGLE && m <= DCG_LINK_WARD; }

// HDBSCAN: step counters, the Prim distances to the tree and the Prim edge sources.
struct HdbLayout { size_t phases, cur, src, total; };

bool hdb_layout(int64_t n, HdbLayout& L) {
  if (n < 2 || n > (INT_MAX - 1) / 2) return false;
  size_t o = 0;
  auto take_bytes = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 256); return at; };
  L.phases = take_bytes(2 * sizeof(long long));
  L.cur = take_bytes((size_t)n * sizeof(double));
  L.src = take_bytes((size_t)n * sizeof(int));
  L.total = o;
  return true;
}

int core_tile_rows(int d, int& lds) {
  lds = d | 1;
  const int rows = kCoreTileDoubles / lds;
  return rows >= 32 ? rows / 32 * 32 : max(rows, 1);
}

template <typename... KArgs, typename... Args>
cudaError_t launch_cluster(void (*kernel)(KArgs...), size_t smem, cudaStream_t st, Args... args) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e != cudaSuccess) return e;
  if (smem > 0) {
    e = ensure_dynamic_smem((const void*)kernel, smem);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(kCtas);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCtas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

}  // namespace
}  // namespace dcg

using namespace dcg;

extern "C" size_t dcg_linkage_workspace_bytes(int64_t n, int d, int method) {
  LinkLayout L;
  if (d < 1 || !valid_method(method) || !link_layout(n, method, L)) return 0;
  return L.total;
}

extern "C" int dcg_linkage_f64(const double* Y, int64_t n, int d, int64_t ld, int method, double* Z,
                               void* ws, size_t ws_bytes, void* stream) {
  LinkLayout L;
  if (n < 2 || n > (INT_MAX - 1) / 2 || d < 1 || ld < d) return DCG_E_SHAPE;
  if (!valid_method(method)) return DCG_E_MODE;
  link_layout(n, method, L);
  if (!Y || !Z) return DCG_E_NULL;
  if (!ws || ws_bytes < L.total) return DCG_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  long long* phases = (long long*)(w + L.phases);
  double* zraw = (double*)(w + L.zraw);
  const int ni = (int)n;
  if (method == DCG_LINK_SINGLE) {
    const int s = (ni + kCtas - 1) / kCtas;
    const size_t stage_bytes = (size_t)s * d * sizeof(double);
    const int stage = stage_bytes <= kPrimStageBytes;
    DCG_CUDA_TRY(launch_cluster(prim_kernel, stage ? stage_bytes : 0, st, Y, ni, d, ld, stage,
                                (const double*)nullptr, (double*)(w + L.cur), (int*)nullptr, zraw, phases));
  } else {
    double* D = (double*)(w + L.D);
    const dim3 grid((unsigned)ceil_div(L.ldD, kDistTile), (unsigned)ceil_div(n, kDistTile));
    linkage_dist_kernel<<<grid, 256, 0, st>>>(Y, ni, d, ld, D, L.ldD);
    DCG_LAUNCH_CHECK();
    DCG_CUDA_TRY(launch_cluster(nn_chain_kernel, 0, st, D, ni, L.ldD, method, zraw, (int*)(w + L.priv), phases));
  }
  linkage_sort_kernel<<<(unsigned)ceil_div(n - 1, kSortThreads), kSortThreads, 0, st>>>(zraw, ni - 1, Z);
  DCG_LAUNCH_CHECK();
  linkage_label_kernel<<<1, 1024, 0, st>>>(Z, ni, (int*)(w + L.parent), (int*)(w + L.usize),
                                           method != DCG_LINK_SINGLE, phases);
  DCG_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t dcg_hdbscan_workspace_bytes(int64_t n, int d, int min_samples) {
  HdbLayout L;
  if (d < 1 || min_samples < 1 || min_samples > DCG_HDBSCAN_MAX_MIN_SAMPLES || min_samples > n ||
      !hdb_layout(n, L))
    return 0;
  return L.total;
}

extern "C" int dcg_core_distances_f64(const double* Y, int64_t n, int d, int64_t ld, int min_samples, double* core,
                                      void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;           // no workspace today; the argument keeps the HDBSCAN entry points alike
  if (n < 2 || n > (INT_MAX - 1) / 2 || d < 1 || ld < d) return DCG_E_SHAPE;
  if (min_samples < 1 || min_samples > DCG_HDBSCAN_MAX_MIN_SAMPLES || min_samples > n) return DCG_E_SHAPE;
  if (!Y || !core) return DCG_E_NULL;
  int lds;
  const int rows = core_tile_rows(d, lds);
  const size_t smem = (size_t)rows * lds * sizeof(double);
  if (smem > kPrimStageBytes) return DCG_E_SHAPE;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)ceil_div(n, kCoreWarps);
  const int ni = (int)n;
  auto run = [&](auto kernel) -> int {
    DCG_CUDA_TRY(ensure_dynamic_smem((const void*)kernel, smem));
    kernel<<<grid, kCoreWarps * 32, smem, st>>>(Y, ni, d, ld, min_samples, rows, lds, core);
    DCG_LAUNCH_CHECK();
    return 0;
  };
  if (min_samples <= 8) return run(core_dist_kernel<8>);
  if (min_samples <= 16) return run(core_dist_kernel<16>);
  if (min_samples <= 32) return run(core_dist_kernel<32>);
  return run(core_dist_kernel<64>);
}

extern "C" int dcg_mreach_mst_f64(const double* Y, int64_t n, int d, int64_t ld, const double* core, double* mst,
                                  void* ws, size_t ws_bytes, void* stream) {
  HdbLayout L;
  if (n < 2 || n > (INT_MAX - 1) / 2 || d < 1 || ld < d) return DCG_E_SHAPE;
  hdb_layout(n, L);
  if (!Y || !core || !mst) return DCG_E_NULL;
  if (!ws || ws_bytes < L.total) return DCG_E_WORKSPACE;
  char* w = (char*)ws;
  const int ni = (int)n;
  const int s = (ni + kCtas - 1) / kCtas;
  const size_t stage_bytes = (size_t)s * d * sizeof(double);
  const int stage = stage_bytes <= kPrimStageBytes;
  DCG_CUDA_TRY(launch_cluster(prim_kernel, stage ? stage_bytes : 0, (cudaStream_t)stream, Y, ni, d, ld, stage,
                              core, (double*)(w + L.cur), (int*)(w + L.src), mst, (long long*)(w + L.phases)));
  return 0;
}
