// Eigen stage of TICA (linalg.py): inverses of the diagonal blocks of chol(K) for its explicit inverse.
// The rest of the shift-and-invert iteration is cuSOLVER / cuBLAS calls and dcg_gen_eig_small_f64 (ticacov.cu).
#include "dcg_common.cuh"

// ---- inverses of the diagonal blocks of a lower-triangular matrix -----------------------------------------
// The explicit inverse of the Cholesky factor of K (linalg._tri_inv_lower) is assembled bottom-up from the
// inverses of its diagonal blocks of <= 128 rows.  cuBLAS inverts such a block in ~56 us (trsm with 125
// right-hand sides, panel-serial, and its batched form loops over the blocks: 0.45 ms for the 8 blocks of
// F = 1000); here one CTA per block does it by forward substitution with NO synchronisation at all: thread j
// owns column j of the inverse, x_i = (delta_ij - sum_{k<i} L_ik x_k) / L_ii, its x_k sit in its own
// shared-memory column, and every thread of a warp reads the same L_ik (one broadcast load from L1 / L2).
// n^2 / 2 dependent-free FMAs per thread: ~20 us for all blocks together.
__global__ void __launch_bounds__(128, 1)
tri_inv_blocks_kernel(const double* __restrict__ L, double* __restrict__ out, int bs, int64_t srow, int64_t scol,
                      int64_t sbatch, int64_t orow, int64_t ocol, int64_t obatch) {
  extern __shared__ double tri_x[];                      // [k][j], j fastest: thread j's column, conflict-free
  const int j = threadIdx.x;
  const double* Lb = L + (size_t)blockIdx.y * sbatch + (size_t)blockIdx.x * bs * (srow + scol);
  double* Ob = out + (size_t)blockIdx.y * obatch + (size_t)blockIdx.x * bs * (orow + ocol);
  if (j >= bs) return;
  for (int i = 0; i < bs; ++i) {
    const double* Li = Lb + (size_t)i * srow;
    double a0 = (i == j) ? 1.0 : 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int k = 0;
    for (; k + 3 < i; k += 4) {                           // x_k = 0 for k < j: the loop is the same for all threads
      a0 = fma(-__ldg(Li + (size_t)k * scol), tri_x[k * bs + j], a0);
      a1 = fma(-__ldg(Li + (size_t)(k + 1) * scol), tri_x[(k + 1) * bs + j], a1);
      a2 = fma(-__ldg(Li + (size_t)(k + 2) * scol), tri_x[(k + 2) * bs + j], a2);
      a3 = fma(-__ldg(Li + (size_t)(k + 3) * scol), tri_x[(k + 3) * bs + j], a3);
    }
    for (; k < i; ++k) a0 = fma(-__ldg(Li + (size_t)k * scol), tri_x[k * bs + j], a0);
    const double x = j <= i ? ((a0 + a1) + (a2 + a3)) / __ldg(Li + (size_t)i * scol) : 0.0;
    tri_x[i * bs + j] = x;
    Ob[(size_t)i * orow + (size_t)j * ocol] = x;
  }
}

extern "C" int dcg_tri_inv_blocks_f64(const double* L, double* out, int batch, int nblk, int bs,
                                      int64_t srow, int64_t scol, int64_t sbatch,
                                      int64_t orow, int64_t ocol, int64_t obatch, void* stream) {
  if (!L || !out) return DCG_E_NULL;
  if (batch < 1 || nblk < 1 || bs < 1 || bs > 128) return DCG_E_SHAPE;
  const size_t smem = (size_t)bs * bs * sizeof(double);
  DCG_CUDA_TRY(dcg::ensure_dynamic_smem((const void*)tri_inv_blocks_kernel, smem));
  tri_inv_blocks_kernel<<<dim3((unsigned)nblk, (unsigned)batch), 128, smem, (cudaStream_t)stream>>>(
      L, out, bs, srow, scol, sbatch, orow, ocol, obatch);
  DCG_LAUNCH_CHECK();
  return 0;
}
