/*
 * dcg.h -- C-ABI of libdcg_b200.so: the B200 (sm_100a) kernels behind deep_cartograph's
 * data-parallel collective-variable hot path.
 *
 * Conventions (SURVEY.md section 8b):
 *   - plain C symbols, `int` return: 0 = ok, -1..-999 = -(cudaError_t), <= -1000 = argument errors
 *     (see DCG_E_*); no exceptions, no stdout.
 *   - every data pointer is a DEVICE pointer owned by the caller (e.g. torch tensor .data_ptr());
 *     `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - calls are asynchronous with respect to `stream`; the caller synchronises before reading
 *     results on the host;
 *   - scratch memory is caller-provided: `ws` / `ws_bytes`, sized by the matching
 *     *_workspace_bytes() query; the library keeps no mutable global state;
 *   - no CPU fallback: without a CUDA device every compute entry point returns an error.
 *
 * Each entry point cites the reference interface (paths under /root/reference/deep_cartograph/)
 * whose arithmetic it replaces.
 */
#ifndef DCG_H_
#define DCG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCG_VERSION 100 /* 0.1.0 */

/* argument errors */
#define DCG_E_NULL      (-1000) /* required pointer is NULL */
#define DCG_E_SHAPE     (-1001) /* n/f/d/k/lag/ld out of range */
#define DCG_E_WORKSPACE (-1002) /* ws too small or NULL */
#define DCG_E_ALIGN     (-1003) /* pointer alignment */
#define DCG_E_ARCH      (-1004) /* device is not sm_100 (tensor-core path) */
#define DCG_E_MODE      (-1005) /* unknown precision / mode flag */

/* covariance contraction engines (dcg_cov_lag_f32 `engine`) */
#define DCG_COV_SIMT_F32   0 /* CUDA-core FP32 FMA tiles, FP64 flush (validation engine)        */
#define DCG_COV_TC_3XTF32  1 /* tcgen05 kind::tf32, split precision hi*hi + hi*lo + lo*hi       */
#define DCG_COV_TC_1XTF32  2 /* tcgen05 kind::tf32, single pass (fast, ~1e-3 relative)          */
#define DCG_COV_TC_3XF16   3 /* tcgen05 kind::f16, FP16 split hi*hi + hi*lo + lo*hi: same 11-bit
                                pieces as 3xTF32 at half the MMA count; needs |z| < 65504 (i.e.
                                standardised inputs)                                            */

int dcg_version(void);
const char* dcg_error_string(int code);
/* sm count / compute capability of the current device; returns 0 or an error */
int dcg_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- A2: per-feature statistics -------------------------------------------------------------
 * Replaces `training_df.agg(['mean','std','min','max'])`
 * (modules/cv_learning/cv_calculator.py:295-297).  Single pass over X (n x f, row stride ld
 * floats): per-thread shifted FP32 sums promoted to FP64, FP64 Welford/Chan merge.  Outputs: mean[f], m2[f] (sum of squared
 * deviations from the mean; std(ddof=1) = sqrt(m2/(n-1))), minv[f], maxv[f].                  */
size_t dcg_colstats_workspace_bytes(int64_t n, int f);
int dcg_colstats_f32(const float* X, int64_t n, int f, int64_t ld,
                     double* mean, double* m2, float* minv, float* maxv,
                     void* ws, size_t ws_bytes, void* stream);

/* ---- A2 across frame shards (SURVEY 8e) --------------------------------------------------------
 * The reference computes the statistics over the concatenated trajectories (cv_calculator.py:295-297);
 * with the frames sharded over GPUs every rank contributes one packed record
 * [n | mean f | m2 f | min f | max f] (doubles) to ONE all-gather, and dcg_stats_merge combines the
 * `world` records (Chan's parallel update, FP64; ranks with n = 0 are skipped).  n_total may be NULL. */
int dcg_stats_pack(double n, const double* mean, const double* m2, const float* minv, const float* maxv,
                   int f, double* packed, void* stream);
int dcg_stats_merge(const double* all_packed, int world, int f, double* mean, double* m2,
                    float* minv, float* maxv, double* n_total, void* stream);

/* ---- small all-reduce over NVLink peer memory (SURVEY 8e) ----------------------------------------
 * The frame-sharded path exchanges a few KB per Lloyd iteration ([sums | counts | stats], reference
 * statistics.py:189-195 run on shards), per projection pass (the CV min / max of normalize_cv,
 * cv_calculator.py:974-991) and per KMeans set-up.  These are ONE kernel per GPU working on peer memory:
 * every rank stores its vector into its slot of every peer's inbox, releases a flag, waits for the `world`
 * flags of its own inbox and reduces the slots in rank order (bitwise identical results on all ranks).
 * One process per GPU: dcg_p2p_alloc makes this rank's inbox (dcg_p2p_buffer_bytes) and its 64-byte CUDA IPC
 * handle, dcg_p2p_open maps a peer's; `peer_bases` (host array, world entries, own inbox at [rank]);
 * `seq` = 1, 2, 3, ... identical on all ranks; op 0 = sum, 1 = max; n <= slot_doubles; in place allowed.   */
size_t dcg_p2p_buffer_bytes(int world, int64_t slot_doubles);
int dcg_p2p_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int dcg_p2p_open(const unsigned char* handle64, void** ptr);
int dcg_p2p_close(void* ptr, int opened);
int dcg_p2p_allreduce_f64(const double* v, double* out, int n, int op, int rank, int world,
                          void* const* peer_bases, int64_t slot_doubles, uint64_t seq, void* stream);

/* ---- A4: in-place standardisation ------------------------------------------------------------
 * Replaces `LinearCalculator.normalize_data` (cv_calculator.py:806-837): x = (x - mean[j]) /
 * range[j] with IEEE float32 subtraction and division.  Also used for the CV normalisation of
 * projected data (cv_calculator.py:966-970) with f = d.                                        */
int dcg_standardize_f32(float* X, int64_t n, int f, int64_t ld,
                        const float* mean, const float* range, void* stream);

/* ---- A11/A12 feeder: gathered, standardised minibatch ------------------------------------------
 * Z[i, :] = (X[idx[i] + offset, :] - mean) / range for i < nb (IEEE float32 subtraction and
 * division, as mlcolvar `Normalization.forward`, the `norm_in` layer of the DeepTICA model built at
 * cv_calculator.py:2569-2590) in one pass instead of a gather and two read+write passes.  idx is
 * int64 (device), every idx[i] + offset must lie in [0, n) (not checked); Z is nb x f, row-major,
 * contiguous.                                                                                    */
int dcg_gather_standardize_f32(const float* X, int64_t n, int f, int64_t ld,
                               const int64_t* idx, int64_t nb, int64_t offset,
                               const float* mean, const float* range, float* Z, void* stream);

/* ---- A5/A6/A7/A8: fused standardise + C0 / C_tau accumulation -------------------------------
 * Replaces mlcolvar `create_timelagged_dataset` + `TICA.compute`'s correlation sums
 * (cv_calculator.py:2244-2261, 2306-2378) and sklearn PCA's Gram (cv_calculator.py:2204-2210).
 * With z_t = (x_t - mean)/range (mean/range NULL: X is used as is), rows t = 0..n_rows-1 and
 * M = n_rows - lag pairs:
 *     S0[i,j]   = sum_{t<M} z_t[i] z_t[j]        (upper triangle i<=j is valid; lower undefined)
 *     St[i,j]   = sum_{t<M} z_t[i] z_{t+lag}[j]  (full, not symmetrised; NULL to skip; lag=0 skips)
 *     colsum_t  = sum_{t<M} z_t ,  colsum_lag = sum_{t>=lag} z_t
 * all FP64, row-major f x f.  `block` > 0 restricts both matrices to the diagonal blocks of that
 * width (hTICA level 1, cv_calculator.py:2331-2354); entries outside are left untouched.
 * For a frame shard, pass own rows + the `lag` halo rows of the next shard (SURVEY 8e).
 * Outputs are OVERWRITTEN (not accumulated).                                                    */
size_t dcg_cov_workspace_bytes(int64_t n_rows, int f, int lag, int block, int engine);
int dcg_cov_lag_f32(const float* X, int64_t n_rows, int f, int64_t ld, int lag,
                    const float* mean, const float* range, int block,
                    double* S0, double* St, double* colsum_t, double* colsum_lag,
                    int engine, void* ws, size_t ws_bytes, void* stream);

/* ---- A5/A6/A7/A8, exact engine: integer tensor cores ---------------------------------------------
 * Same sums as dcg_cov_lag_f32 (same reference call sites), computed EXACTLY on the int8 tensor
 * cores (tcgen05 kind::i8, int32 accumulation): every value is first rounded to 23-bit fixed point
 * relative to its column's range, q = rint((x - mean[j]) * 2^e_j) -- the float32 resolution of the
 * data -- split into three int8 digit planes in the K-major layout of the contraction (one HBM-bound
 * pass), and the planes are contracted by TMA-staged integer MMAs: the digit products are exact (all
 * but d0 d0, which is left out), and only the FP64 scaling and adds of the int32 partial sums round
 * (csrc/cov_i8.cu).  `xmin` / `xmax` (f, float32, device): per-column bounds of X over ALL n_rows rows
 * (the column statistics, dcg_colstats_f32); values outside them may be clamped to |q| <= 4161536.
 * `info[0]` (int32, device, may be NULL) is nonzero if and only if some value was clamped; its value
 * counts groups of values and depends on the kernel path.  The digit planes of a window of frames live
 * in `ws`.                                                                                            */
#define DCG_COV_TC_I8X3    4 /* tcgen05 kind::i8 on three int8 digit planes: exact accumulation    */
size_t dcg_cov_i8_workspace_bytes(int64_t n_rows, int f, int lag, int block);
int dcg_cov_lag_i8_f32(const float* X, int64_t n_rows, int f, int64_t ld, int lag,
                       const float* mean, const float* range, const float* xmin, const float* xmax,
                       int block, double* S0, double* St, double* colsum_t, double* colsum_lag,
                       int* info, void* ws, size_t ws_bytes, void* stream);

/* Device timing of the exact engine's two kernels (diagnostics for bench.py's roofline): when switched
 * on, every window's quantise and contraction launches are bracketed by CUDA events on the launching
 * stream (up to 64 windows between reads); dcg_cov_i8_get_timing synchronises on them and returns the
 * summed durations in ms and the number of contraction launches since the last read.  One stream, one
 * host thread.                                                                                        */
int dcg_cov_i8_set_timing(int on);
int dcg_cov_i8_get_timing(float* quantize_ms, float* contract_ms, int* launches);

/* ---- A9/A10: projection ----------------------------------------------------------------------
 * Replaces `LinearCalculator.normalize_cv` + `project_data` (cv_calculator.py:918-991):
 * P[t,:] = ((x_t - mean)/range) @ W  (mean/range NULL: no standardisation), W is f x d row-major
 * float32, P is n x d row-major float32.  pmin/pmax (d, float32, may be NULL) receive the
 * per-column min / max of P (for cv_norm_mean / cv_norm_range).  1 <= d <= 64.                  */
size_t dcg_project_workspace_bytes(int64_t n, int f, int d);
int dcg_project_f32(const float* X, int64_t n, int f, int64_t ld,
                    const float* mean, const float* range,
                    const float* W, int d, float* P, float* pmin, float* pmax,
                    void* ws, size_t ws_bytes, void* stream);

/* ---- A8: hTICA level-1 projections, all diagonal blocks in one pass ------------------------------
 * Replaces the per-subspace `data @ V_b` loop of `HTICACalculator.compute_cv`
 * (cv_calculator.py:2331-2371; the block-diagonal T1 of :2367).  Feature block c covers columns
 * [c*block, min(f, (c+1)*block)) (torch.split semantics: the last block may be narrower) and
 * projects only them:  P[t, c*s + j] = sum_i ((x_t[i] - mean[i]) / range[i]) * W[i, j],
 * i in block c, j < min(s, width of block c).  W is f x s row-major: row i holds the s weights
 * of feature i within its own block.  P is n x p_ld row-major float32.  Needs 16-byte aligned
 * rows (X % 16 == 0, ld % 4 == 0; else DCG_E_ALIGN), 1 <= s <= 16, block <= 1018.               */
size_t dcg_project_blocks_workspace_bytes(int64_t n, int f, int block);
int dcg_project_blocks_f32(const float* X, int64_t n, int f, int64_t ld,
                           const float* mean, const float* range,
                           const float* W, int block, int s, float* P, int64_t p_ld,
                           void* ws, size_t ws_bytes, void* stream);

/* ---- K1: KMeans E-step + M-step sums ---------------------------------------------------------
 * Replaces one sklearn `lloyd_iter` as triggered by `statistics.kmeans_clustering`
 * (modules/statistics/statistics.py:159-197; sklearn/cluster/_k_means_lloyd.pyx:193-214):
 * label = argmin_j ||c_j||^2 - 2 y.c_j, lowest index wins ties.  Y is n x d (row stride ld),
 * `dtype_bytes` wide (4 = float32, 8 = float64); centers is k x d FP64 (the Lloyd driver owns the
 * centres in FP64).  Scores are screened in FP32 and near-ties re-evaluated in FP64, so the label is
 * the FP64 argmin.  labels (int32, n) is read (previous labels, -1 initially) and overwritten.  Outputs (overwritten): sums[k*d], counts[k] FP64;
 * stats[0] = number of labels that changed, stats[1] = inertia sum ||y - c_label||^2,
 * stats[2] = number of exact ties (FP64 second-best == best).  gap (n, may be NULL) receives
 * second-best minus best score per frame in `dtype_bytes` precision.  Limits: 1 <= d <= 32,
 * k*(pad4(d)+1)*4 bytes <= 200 KB (centres live in shared memory).
 * update_sums = 0 skips sums/counts (final E-step, _kmeans.py:742-754).
 * y_absmax (device pointer to one double, may be NULL): a bound |Y[t,q]| <= *y_absmax over the
 * frames of this call.  With it the per-CTA partial sums are accumulated in 64-bit fixed point
 * (native 32-bit shared-memory integer adds instead of FP64 compare-and-swap loops): exact integer
 * sums, order-independent, each value rounded at <= 2^-45 * y_absmax (for <= 128 k frames per CTA),
 * i.e. below the run-to-run noise of FP64 summation order.  NULL keeps FP64 atomics.
 * With y_absmax, d <= 15 and 256 <= k <= 2048 (or k >= 64 and d >= 8) the scores are screened
 * on the tensor cores (FP16-split GEMM, operands scaled into [-1, 1] by the bound; kmeans_mma.cu)
 * with the same rigorous near-tie test and FP64 refine: the labels are unchanged, k = 1000 is
 * twice as fast.  Env DCG_KMEANS_TC=0 forces the CUDA-core kernel.                             */
size_t dcg_kmeans_workspace_bytes(int64_t n, int d, int k, int dtype_bytes);
int dcg_kmeans_step(const void* Y, int64_t n, int d, int64_t ld, int dtype_bytes,
                    const double* centers, int k, int32_t* labels,
                    double* sums, double* counts, double* stats, void* gap,
                    int update_sums, const double* y_absmax, void* ws, size_t ws_bytes, void* stream);

/* ---- K1: M-step finish ------------------------------------------------------------------------
 * Replaces sklearn `_average_centers` + the centre-shift test of `_kmeans_single_lloyd`
 * (sklearn/cluster/_k_means_common.pyx, _kmeans.py:703-740) as reached from
 * statistics.kmeans_clustering (statistics.py:159-197).  info[0] = number of empty clusters
 * (counts == 0).  If there is none: centers[j] = sums[j] * (1 / counts[j]) in place and
 * info[1] = sum_j ||c_new - c_old||^2; otherwise centers are left untouched (the caller relocates
 * the empty clusters first, sklearn/cluster/_k_means_common.pyx:167-211).  All FP64.            */
int dcg_kmeans_update(const double* sums, const double* counts, int k, int d,
                      double* centers, double* info, void* stream);

/* ---- K1: one whole Lloyd iteration on one device ----------------------------------------------
 * dcg_kmeans_step (E-step + FP64 sums) followed by dcg_kmeans_update (M-step finish) in one call.
 * `work` holds k*d + k + 5 doubles: [sums k*d | counts k | stats 3 | info 2] (overwritten); see the
 * two entry points above for their meaning.  `centers` is updated in place unless a cluster came
 * out empty (info[0] > 0).  Sharded runs call the two halves around their all-reduce instead.   */
int dcg_kmeans_iterate(const void* Y, int64_t n, int d, int64_t ld, int dtype_bytes,
                       double* centers, int k, int32_t* labels, double* work,
                       const double* y_absmax, void* ws, size_t ws_bytes, void* stream);

/* ---- K1: up to `iters` Lloyd iterations on one device without a host round trip -------------------
 * The Lloyd driver of statistics.kmeans_clustering (reference statistics.py:159-197, scikit-learn's
 * lloyd loop) reads (changed, empty, shift) after every iteration.  Here the tests run on the device:
 * `work` holds k*d + k + 8 doubles [sums | counts | stats 3 | info 2 | ctl 3]; ctl = [stop, done, tol].
 * The iterations are all enqueued; after the one in which a cluster came out empty, no label changed or
 * the centre shift is <= tol, the remaining launches return at once, so `work`, `centers` and `labels`
 * hold exactly the state dcg_kmeans_iterate would have left at that iteration and ctl[1] says which.  */
int dcg_kmeans_iterate_n(const void* Y, int64_t n, int d, int64_t ld, int dtype_bytes,
                         double* centers, int k, int32_t* labels, double* work,
                         const double* y_absmax, int iters, double tol,
                         void* ws, size_t ws_bytes, void* stream);

/* ---- K3: nearest sample to each centre -------------------------------------------------------
 * Replaces `statistics.find_centroids` (statistics.py:370-377): argmin_t ||y_t - c_j||_2 per
 * centre j, first index on ties, evaluated in FP64.  argmin is int64[k].                        */
size_t dcg_nearest_workspace_bytes(int64_t n, int d, int k);
int dcg_nearest_to_centers(const void* Y, int64_t n, int d, int64_t ld, int dtype_bytes,
                           const double* centers, int k, int64_t* argmin,
                           void* ws, size_t ws_bytes, void* stream);

/* ---- A11: DeepTICA minibatch covariance ------------------------------------------------------
 * Replaces the correlation sums inside mlcolvar `DeepTICA.training_step` (driven from
 * cv_calculator.py:1508-1524).  f, g are B x d float32 network outputs (row-major), w / wl the
 * per-sample weights (NULL = 1).  Outputs FP64 raw sums (overwritten), accumulated in FP64 from
 * the first row (each w f_i f_j is rounded once), since they are not mean-free:
 *   out[0]            = sum w,          out[1] = sum wl
 *   out[2 .. 2+d)     = sum w f
 *   then d*d each     : sum w f f^T,  sum wl f g^T,  then d each: sum wl f, sum wl g
 * The caller forms mean-free C0 / C_tau in FP64 (see host code).  1 <= d <= 32.  The result is
 * deterministic: the per-CTA partial sums go to ws (dcg_ticacov_workspace_bytes(B, d) bytes, no
 * initialisation needed) and are added in a fixed order by a second launch.                      */
size_t dcg_ticacov_out_doubles(int d);
size_t dcg_ticacov_workspace_bytes(int64_t B, int d);
int dcg_ticacov_f32(const float* f, const float* g, const float* w, const float* wl,
                    int64_t B, int d, double* out, void* ws, size_t ws_bytes, void* stream);

/* ---- A11: DeepTICA eigen-loss and its gradient ------------------------------------------------
 * Replaces mlcolvar `cholesky_eigh` + `ReduceEigenvaluesLoss(mode='sum2')` and their autograd
 * backward inside `DeepTICA.training_step` (driven from cv_calculator.py:1508-1524): from the raw
 * sums of dcg_ticacov_f32 (after an all-reduce when the minibatch is sharded) one launch forms the
 * mean-free symmetrised C0 / C_tau, B = C0 + reg I, L = chol(B), the eigenvalues of
 * L^-1 C_tau L^-T (descending) and loss = -sum_{i < n_eig} lambda_i^2 (n_eig <= 0: all), together
 * with dLoss/dC0 and dLoss/dC_tau (symmetric d x d).
 * res (doubles): [0] loss, [1] status (0 ok, 1: B not positive definite or a sum, mean or
 * covariance not finite -- then loss and evals are NaN and G0 = Gt = 0), [2] sum w, [3] sum wl,
 * evals[d], mu[d] (weighted mean of f), G0[d*d], Gt[d*d].                                        */
size_t dcg_ticaloss_out_doubles(int d);
int dcg_ticaloss_f64(const double* sums, int d, double reg, int n_eig, double* res, void* stream);

/* ---- eigen stage: small generalised symmetric eigenproblem -------------------------------------
 * H s = theta G s for `batch` independent b x b pencils (b <= 32, G symmetric positive definite,
 * row-major FP64; only the symmetric parts are used): theta[batch][b] DESCENDING, S[batch][b][b]
 * with the G-orthonormal eigenvectors as columns in the same order, status[batch] (0 ok, 1: G not
 * positive definite).  The Rayleigh-Ritz step of the top-d solver that stands in for mlcolvar
 * `cholesky_eigh` as called from TICA.compute (cv_calculator.py:2257-2261): one launch instead of
 * cholesky_ex + solve_triangular + GEMMs + eigh (whose error check synchronises the host).        */
int dcg_gen_eig_small_f64(const double* H, const double* G, int b, int batch,
                          double* theta, double* S, double* status, void* stream);

/* Inverses of the `nblk` diagonal blocks (bs x bs, bs <= 128) of `batch` lower-triangular matrices, written to
 * the same blocks of `out`; element (i, j) of matrix m at m * sbatch + i * srow + j * scol (any layout).  One CTA
 * per block, forward substitution, no synchronisation (part of the explicit inverse of chol(K) in the
 * shift-and-invert iteration that replaces mlcolvar's cholesky_eigh, cv_calculator.py:2257-2261).            */
int dcg_tri_inv_blocks_f64(const double* L, double* out, int batch, int nblk, int bs,
                           int64_t srow, int64_t scol, int64_t sbatch,
                           int64_t orow, int64_t ocol, int64_t obatch, void* stream);

/* ---- N1: dispersion sums for the clustering scores -------------------------------------------------
 * For sklearn's calinski_harabasz_score / davies_bouldin_score as called at
 * modules/statistics/statistics.py:73-74: per cluster c (labels int32 in [0, k), means k x d FP64 =
 * the means of the members), ssq[c] = sum ||y_t - m_c||^2 and sdist[c] = sum ||y_t - m_c|| over the
 * members, FP64, in one pass over Y (n x d, float32 or float64).  Outputs are overwritten.           */
int dcg_cluster_dispersion(const void* Y, int64_t n, int d, int64_t ld, int dtype_bytes, const int* labels,
                           const double* means, int k, double* ssq, double* sdist, void* stream);

/* ---- N1: exact silhouette of L labelings in one pass over all frame pairs ------------------------------
 * For sklearn's silhouette_score(metric="euclidean") as called at modules/statistics/statistics.py:75, for
 * L labelings of the same n frames Y (n x d FP64, row stride ld) at once (csrc/silhouette.cu).  Per labeling
 * l, with its labels encoded 0..k_l - 1 (as LabelEncoder does):
 *   a_i = (sum of d(i, j) over i's own cluster) / (n_own - 1),
 *   b_i = min over the other clusters c of (sum of d(i, j) over c) / |c|,
 *   s_i = (b_i - a_i) / max(a_i, b_i), NaN -> 0 (singletons; a = b = 0), scores[l] = mean of s_i.
 * d(i, j) = sqrt(sum_f (y_i[f] - y_j[f])^2), features ascending, a rounded subtract, multiply and add per term,
 * then one sqrt (pdist's arithmetic, as dcg_linkage_f64 and dcg_nearest_frames_f64).  Each distance is computed
 * once and feeds every labeling; each cluster sum of m distances is within m u / (1 - m u) of exact (u = 2^-53).
 * A labeling's results are bitwise the same whether it is scored alone or with others, and from run to run
 * (fixed-order sums, no floating-point atomics).
 * Inputs (device): labels L x n int32 (labeling l at labels + l n); offsets L + 1 int32, labeling l owns slots
 * offsets[l] .. offsets[l+1] - 1, offsets[0] = 0, offsets[L] = K = sum_l k_l; sizes K int32, the member count
 * of every slot.  Outputs: scores (L doubles); samples (L x n doubles, s_i of labeling l at samples + l n; may
 * be NULL).  A label outside 0..k_l - 1 touches no slot: that labeling's score is NaN, as is s_i of its frame.
 * Limits: every slot has one FP64 accumulator per row of a CTA in shared memory, so K <= 384
 * (DCG_SILHOUETTE_MAX_SLOTS: 192 KB of the 227 KB a CTA may use), L <= 32, d <= 2048; callers split larger
 * sets of labelings into groups.  Memory is O(n (d + L)): the workspace holds n (4 + 2 L) bytes of label
 * codes and masks and 8 L doubles per 64 frames, no n x n or chunk x n buffer.  O(n^2 (d + L)) work.
 * Errors: DCG_E_SHAPE for n < 3, n > INT_MAX, d < 1, d > 2048, ld < d, L < 1, L > 32, K < 2 L or K > 384;
 * DCG_E_NULL (samples may be NULL); DCG_E_WORKSPACE.  The workspace query returns 0 for an invalid shape.    */
#define DCG_SILHOUETTE_MAX_SLOTS     384
#define DCG_SILHOUETTE_MAX_LABELINGS 32
size_t dcg_silhouette_workspace_bytes(int64_t n, int L, int K);
int dcg_silhouette_f64(const double* Y, int64_t n, int d, int64_t ld, const int32_t* labels, int L,
                       const int32_t* offsets, const int32_t* sizes, int K, double* scores, double* samples,
                       void* ws, size_t ws_bytes, void* stream);

/* ---- N2: agglomerative clustering tree ----------------------------------------------------------------
 * Replaces sklearn AgglomerativeClustering(n_clusters, linkage).fit_predict as called from
 * `hierarchical_clustering` (modules/statistics/statistics.py:285): the full merge tree of the n frames of
 * Y (n x d FP64, row stride ld, Euclidean), bitwise identical to sklearn's.  Z is (n-1) x 4 FP64, exactly
 * scipy.cluster.hierarchy.linkage's output, i.e. sklearn's children_ (columns 0-1), distances_ (column 2)
 * and the merged cluster sizes (column 3); node n + i is the cluster formed by row i.
 *   complete / average / ward: scipy's nn_chain on the full FP64 distance matrix (8 n^2 bytes of ws);
 *   single: sklearn's mst_linkage_core (Prim from frame 0, distances on the fly, O(n) ws).
 * The first 16 bytes of ws receive two int64 counters of the tree kernel (row scans, merges).  Errors:
 * DCG_E_SHAPE for n < 2, d < 1 or ld < d; DCG_E_MODE for an unknown method.                           */
#define DCG_LINK_SINGLE   0
#define DCG_LINK_COMPLETE 1
#define DCG_LINK_AVERAGE  2
#define DCG_LINK_WARD     3
size_t dcg_linkage_workspace_bytes(int64_t n, int d, int method);
int dcg_linkage_f64(const double* Y, int64_t n, int d, int64_t ld, int method, double* Z,
                    void* ws, size_t ws_bytes, void* stream);

/* ---- N3: HDBSCAN single-linkage tree (core distances + mutual-reachability MST) -----------------------
 * Replaces the device-side half of sklearn.cluster.HDBSCAN(metric="euclidean").fit on dense finite data,
 * i.e. _hdbscan_prims (sklearn/cluster/_hdbscan/hdbscan.py) with its KD-tree.  O(n) memory, no n x n matrix.
 * Distances are sqrt(sum_f (y_i[f] - y_j[f])^2), features ascending, a rounded multiply and a rounded add
 * per term: the arithmetic of the KD-tree's and of EuclideanDistance.dist, so both results are bitwise
 * sklearn's.
 * dcg_core_distances_f64 replaces NearestNeighbors(n_neighbors=min_samples).kneighbors(X)[0][:, -1]:
 *   core (n FP64) = distance of every frame to its min_samples-th nearest frame, the frame itself counted
 *   at distance 0.  1 <= min_samples <= min(n, DCG_HDBSCAN_MAX_MIN_SAMPLES).  ws may be NULL.
 * dcg_mreach_mst_f64 replaces sklearn/cluster/_hdbscan/_linkage.pyx mst_from_data_matrix (alpha = 1):
 *   Prim from frame 0 on max(core[c], core[j], dist(c, j)); mst is (n-1) x 3 FP64 rows
 *   (source node, new node, distance) in visiting order, the source being the tree node that last strictly
 *   improved the new node.  The first 16 bytes of ws receive two int64 step counters.
 * The edge sort (numpy's default argsort) and make_single_linkage are left to the caller.
 * Errors: DCG_E_SHAPE for n < 2, d < 1, ld < d or min_samples out of range; DCG_E_NULL; DCG_E_WORKSPACE. */
#define DCG_HDBSCAN_MAX_MIN_SAMPLES 64
size_t dcg_hdbscan_workspace_bytes(int64_t n, int d, int min_samples);
int dcg_core_distances_f64(const double* Y, int64_t n, int d, int64_t ld, int min_samples, double* core,
                           void* ws, size_t ws_bytes, void* stream);
int dcg_mreach_mst_f64(const double* Y, int64_t n, int d, int64_t ld, const double* core, double* mst,
                       void* ws, size_t ws_bytes, void* stream);

/* ---- N5: nearest clustered frame of supplementary frames ----------------------------------------------
 * Replaces the NearestNeighbors(n_neighbors=1).fit(X).kneighbors(Q) of the reference's assign_closest_cluster
 * (tools/traj_cluster/traj_cluster_workflow.py:207-238): for each of the m queries Q (row stride ldq) the
 * nearest of the n frames X (row stride ldx), all d features, FP64 (csrc/nearest.cu).
 * rdist = sum_f (q_f - x_f)^2, features ascending, a rounded subtract, multiply and add per term, then one
 * sqrt: the arithmetic of scikit-learn's KD-tree, which its `auto` algorithm picks for d <= 15; the device
 * keeps it for every d (for d > 15 scikit-learn switches to brute force with the GEMM expansion).
 * index[i] (int64) = the lexicographic minimum of (rdist, frame index), i.e. the lowest-indexed frame among
 * exact ties; dist[i] = sqrt(rdist).  The frames are put in Morton order and cut into tiles whose boxes
 * prune the search exactly (the bound uses the same rounded arithmetic; see nearest.cu).  Memory is
 * O((n + m) d), no n x m buffer.  The first 16 bytes of ws receive two uint64 counters: tiles visited and
 * tiles considered (query blocks x tiles).  The workspace query needs a CUDA device (it sizes the radix
 * sort) and returns 0 without one or for an invalid shape.  m = 0 is a no-op.  Every coordinate of X and Q
 * must be finite (ops.nearest_frames checks it): with NaN in a query's row no frame compares below its best, and
 * its index and dist are then not defined.
 * Errors: DCG_E_SHAPE for n < 1, m < 0, d < 1, d > 8192, ldx < d, ldq < d or n or m above INT_MAX;
 * DCG_E_NULL; DCG_E_WORKSPACE.                                                                         */
size_t dcg_nearest_frames_workspace_bytes(int64_t n, int64_t m, int d);
int dcg_nearest_frames_f64(const double* X, int64_t n, int64_t ldx, const double* Q, int64_t m, int64_t ldq,
                           int d, int64_t* index, double* dist, void* ws, size_t ws_bytes, void* stream);

/* ---- N4: free-energy surface by binned kernel density estimation ---------------------------------
 * Replaces mlcolvar.utils.fes.compute_fes(backend="KDEpy") as called at modules/figures/figures.py:95
 * (from tools/train_colvars/train_colvars_workflow.py:146-182).  KDEpy's FFTKDE = linear binning onto
 * the evaluation grid + convolution with the sampled kernel:
 *   dcg_fes_bin_f32    P is n x ld float32 (the projected frames); column c0 is x, column c1 is y
 *                      (c1 < 0: 1-D).  Frames are split into `blocks` contiguous blocks
 *                      (numpy.array_split); block b's linear-binning weights land in
 *                      hist[b][iy][ix] (FP64, G x G or G nodes spanning [lo, hi] per axis, overwritten).
 *                      Frames outside the bounds are skipped and counted in *n_outside (device, may be NULL).
 *   dcg_fes_smooth_f64 density[b] = (hist[b] / block_frames[b]) convolved with a Gaussian of standard
 *                      deviation `bandwidth` sampled at the grid offsets (step0, step1 = grid spacing);
 *                      block_frames NULL: no normalisation.  tmp: blocks*G*G doubles (dim 2 only).     */
int dcg_fes_bin_f32(const float* P, int64_t n, int64_t ld, int c0, int c1,
                    double lo0, double hi0, double lo1, double hi1, int G, int blocks,
                    double* hist, int64_t* n_outside, void* stream);
int dcg_fes_smooth_f64(const double* hist, int blocks, int G, int dim, double step0, double step1,
                       double bandwidth, const double* block_frames, double* density, double* tmp,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DCG_H_ */
