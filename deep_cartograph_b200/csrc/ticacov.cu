// A11: DeepTICA minibatch correlation sums (weighted), FP64 outputs.
// Replaces the correlation sums inside mlcolvar DeepTICA.training_step / TICA.compute as driven
// from reference cv_calculator.py:1508-1524.  B x d network outputs (d <= 32): a memory/latency-
// bound reduction, not a tensor-core contraction (SURVEY 8a row A11).
#include "dcg_common.cuh"

namespace dcg {

// out layout (doubles): [0]=sum w, [1]=sum wl, [2..2+d)=sum w f, then d*d sum w f f^T,
// d*d sum wl f g^T, d sum wl f, d sum wl g.
// A CTA stages kTcRowsPerCta rows (f row, g row, w, wl) in shared memory; thread e < d*d owns the
// matrix entry (i, j) = (e / d, e % d) of BOTH matrices, thread d*d + i the three vector entries of
// component i, thread d*d + d the two weight sums -- uniform code inside each class, rows unrolled
// by 4, FP64 throughout.  The sums are raw, not mean-free, and the mean of the network outputs is
// free to drift (the loss does not depend on it): C0 = sff/sw - mu mu^T then cancels |mu|^2 / var
// digits, which FP32 partial sums (2^-24 of |mu|^2 per add) do not have to spare.  w * f_i of two
// floats is exact in FP64, so each row costs one rounding per entry.
// The result is deterministic: CTA k takes tiles k, k + G, k + 2G, ... (G = min(tiles, kTcMaxCtas))
// and adds them in that order into its own column part[entry][k]; ticacov_reduce_kernel then sums
// the G columns of each entry in a fixed order.  (FP64 atomics across CTAs would round differently
// from run to run, since FP64 partial sums, unlike FP32 ones, do not add exactly.)
constexpr int kTcThreads = 256;
constexpr int kTcRowsPerCta = 128;
constexpr int64_t kTcMaxCtas = 1024;

static inline int64_t ticacov_ctas(int64_t B) { return min(ceil_div(B, kTcRowsPerCta), kTcMaxCtas); }

__global__ void __launch_bounds__(kTcThreads)
ticacov_kernel(const float* __restrict__ f, const float* __restrict__ g, const float* __restrict__ w,
               const float* __restrict__ wl, int64_t B, int d, double* __restrict__ part, int G) {
  extern __shared__ float sm[];              // [rows][2*d + 2] : f row, g row, w, wl
  const int stride = 2 * d + 2;
  const int dd = d * d;
  // part[idx][k]: this CTA's running sum of output entry idx
  double* col = part + blockIdx.x;
  const int64_t n_tiles = (B + kTcRowsPerCta - 1) / kTcRowsPerCta;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const bool first = (t == (int64_t)blockIdx.x);
    auto put = [&](int idx, double v) {
      double* p = col + (size_t)idx * G;
      *p = first ? v : *p + v;
    };
    const int64_t r0 = t * kTcRowsPerCta;
    const int rows = (int)min((int64_t)kTcRowsPerCta, B - r0);
    __syncthreads();                         // the previous tile's rows are no longer read
    for (int i = threadIdx.x; i < rows * d; i += kTcThreads) {
      const int r = i / d, q = i - r * d;
      sm[r * stride + q] = f[(r0 + r) * d + q];
      sm[r * stride + d + q] = g[(r0 + r) * d + q];
    }
    for (int r = threadIdx.x; r < rows; r += kTcThreads) {
      sm[r * stride + 2 * d] = w ? w[r0 + r] : 1.f;
      sm[r * stride + 2 * d + 1] = wl ? wl[r0 + r] : 1.f;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < dd + d + 1; e += kTcThreads) {
      if (e < dd) {
        const int i = e / d, j = e - i * d;
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 4
        for (int r = 0; r < rows; ++r) {
          const float* row = sm + r * stride;
          const double fi = row[i];
          a0 = fma((double)row[2 * d] * fi, (double)row[j], a0);
          a1 = fma((double)row[2 * d + 1] * fi, (double)row[d + j], a1);
        }
        put(2 + d + e, a0);                  // sum w f f^T
        put(2 + d + dd + e, a1);             // sum wl f g^T
      } else if (e < dd + d) {
        const int i = e - dd;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
#pragma unroll 4
        for (int r = 0; r < rows; ++r) {
          const float* row = sm + r * stride;
          a0 = fma((double)row[2 * d], (double)row[i], a0);
          a1 = fma((double)row[2 * d + 1], (double)row[i], a1);
          a2 = fma((double)row[2 * d + 1], (double)row[d + i], a2);
        }
        put(2 + i, a0);                      // sum w f
        put(2 + d + 2 * dd + i, a1);         // sum wl f
        put(2 + 2 * d + 2 * dd + i, a2);     // sum wl g
      } else {
        double a0 = 0.0, a1 = 0.0;
        for (int r = 0; r < rows; ++r) { a0 += sm[r * stride + 2 * d]; a1 += sm[r * stride + 2 * d + 1]; }
        put(0, a0);
        put(1, a1);
      }
    }
  }
}

// out[e] = sum over k of part[e][k], one warp per entry, in a fixed order (strided lane sums, then the
// butterfly of warp_sum)
__global__ void __launch_bounds__(kTcThreads)
ticacov_reduce_kernel(const double* __restrict__ part, int G, int n_out, double* __restrict__ out) {
  const int e = blockIdx.x * (kTcThreads / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (e >= n_out) return;                    // warp-uniform
  const double* p = part + (size_t)e * G;
  double s = 0.0;
  for (int k = lane; k < G; k += 32) s += p[k];
  s = warp_sum(s);
  if (lane == 0) out[e] = s;
}

// ---- A11: the d x d eigen-loss and its gradient in ONE launch ------------------------------------
// From the raw sums: mean-free symmetrised C0 / C_tau, B = C0 + reg I, L = chol(B),
// A = L^-1 C_tau L^-T, eigenvalues (cyclic Jacobi, FP64), loss = -sum_{i < n_eig} lambda_i^2
// (mlcolvar ReduceEigenvaluesLoss(mode='sum2') on cholesky_eigh, driven from reference
// cv_calculator.py:1508-1524), and the gradients with respect to the (symmetric) C0 and C_tau.
// With the B-normalised generalised eigenvectors v_i = L^-T u_i:
//     d lambda_i = v_i^T (dC_tau - lambda_i dC0) v_i
//  => dLoss/dC_tau = -2 sum lambda_i v_i v_i^T,   dLoss/dC0 = +2 sum lambda_i^2 v_i v_i^T.
// In torch this is ~40 tiny launches (cholesky, two triangular solves, eigvalsh and their
// backward); here one warp does it in shared memory (d <= 32).
// res layout (doubles): [0] loss, [1] status (0 ok, 1 = B not positive definite or a sum not finite;
// then loss and evals are NaN and G0 = Gt = 0), [2] sum w, [3] sum wl, then evals[d] (descending),
// mu[d], G0[d*d], Gt[d*d].
__global__ void __launch_bounds__(32)
ticaloss_kernel(const double* __restrict__ sums, int d, double reg, int n_eig, double* __restrict__ res) {
  __shared__ double C0[32][33], Ct[32][33], L[32][33], A[32][33], V[32][33];
  double (*Li)[33] = C0;               // C0 is dead once its Cholesky factor exists
  __shared__ double mu[32], nu[32], xi[32], ev[32];
  __shared__ int order[32];
  __shared__ int s_bad;
  const int lane = threadIdx.x;
  const int dd = d * d;
  const double sw = sums[0], swl = sums[1];
  const double* swf = sums + 2;
  const double* sff = sums + 2 + d;
  const double* sfg = sff + dd;
  const double* slf = sfg + dd;
  const double* slg = slf + d;
  if (lane == 0) s_bad = 0;
  if (lane < d) { mu[lane] = swf[lane] / sw; nu[lane] = slg[lane] / swl; xi[lane] = slf[lane] / swl; }
  __syncwarp();
  // lane i builds row i (symmetrised afterwards)
  if (lane < d) {
    const int i = lane;
    for (int j = 0; j < d; ++j) {
      L[i][j] = sff[i * d + j] / sw - mu[i] * mu[j];                                    // C0 raw
      A[i][j] = sfg[i * d + j] / swl - mu[i] * nu[j] - xi[i] * mu[j] + mu[i] * mu[j];   // Ct raw
    }
  }
  __syncwarp();
  if (lane < d) {
    const int i = lane;
    for (int j = 0; j < d; ++j) {
      C0[i][j] = 0.5 * (L[i][j] + L[j][i]);
      Ct[i][j] = 0.5 * (A[i][j] + A[j][i]);
    }
    // a NaN / Inf anywhere in the sums (a diverged network, sum w = 0 or sum wl = 0) reaches mu, nu, xi, C0
    // or C_tau, except an infinite sum w / sum wl, which zeroes what it divides: flag all of it here, as the
    // Cholesky below only sees C0's pivots
    bool fin = isfinite(sw) && isfinite(swl) && isfinite(mu[i]) && isfinite(nu[i]) && isfinite(xi[i]);
    for (int j = 0; j < d; ++j) fin = fin && isfinite(C0[i][j]) && isfinite(Ct[i][j]);
    if (!fin) s_bad = 1;
  }
  __syncwarp();
  // Cholesky of B = C0 + reg I (column by column; lanes own rows)
  for (int j = 0; j < d; ++j) {
    if (lane == j) {
      double s = C0[j][j] + reg;
      for (int k = 0; k < j; ++k) s -= L[j][k] * L[j][k];
      if (!(s > 0.0)) { s_bad = 1; s = 1.0; }
      L[j][j] = sqrt(s);
    }
    __syncwarp();
    if (lane > j && lane < d) {
      double s = C0[lane][j];
      for (int k = 0; k < j; ++k) s -= L[lane][k] * L[j][k];
      L[lane][j] = s / L[j][j];
    }
    if (lane < j) L[lane][j] = 0.0;
    __syncwarp();
  }
  // Li = L^-1 (lane c solves L x = e_c)
  if (lane < d) {
    const int c = lane;
    for (int i = 0; i < d; ++i) {
      double s = (i == c) ? 1.0 : 0.0;
      for (int k = c; k < i; ++k) s -= L[i][k] * Li[k][c];
      Li[i][c] = (i < c) ? 0.0 : s / L[i][i];
    }
  }
  __syncwarp();
  // A = Li Ct Li^T (lane i: row i of T = Li Ct into V, then row i of A = T Li^T), symmetrised
  if (lane < d) {
    const int i = lane;
    for (int j = 0; j < d; ++j) {
      double s = 0.0;
      for (int k = 0; k <= i; ++k) s += Li[i][k] * Ct[k][j];
      V[i][j] = s;
    }
  }
  __syncwarp();
  if (lane < d) {
    const int i = lane;
    for (int j = 0; j < d; ++j) {
      double s = 0.0;
      for (int k = 0; k <= j; ++k) s += V[i][k] * Li[j][k];
      A[i][j] = s;
    }
  }
  __syncwarp();
  if (lane < d) {
    const int i = lane;
    for (int j = i + 1; j < d; ++j) { const double m = 0.5 * (A[i][j] + A[j][i]); A[i][j] = m; }
  }
  __syncwarp();
  if (lane < d) {
    const int i = lane;
    for (int j = 0; j < i; ++j) A[i][j] = A[j][i];
    for (int j = 0; j < d; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;       // eigenvectors accumulate here
  }
  __syncwarp();
  // cyclic Jacobi: A <- J^T A J, V <- V J; lanes own the index k of the updated rows / columns
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, diag = 0.0;
    if (lane < d) {
      for (int j = 0; j < d; ++j) { if (j != lane) off += A[lane][j] * A[lane][j]; }
      diag = A[lane][lane] * A[lane][lane];
    }
    off = warp_sum(off);
    diag = warp_sum(diag);
    if (off <= 1e-32 * diag || off == 0.0) break;
    for (int p = 0; p < d - 1; ++p)
      for (int q = p + 1; q < d; ++q) {
        const double apq = A[p][q];
        if (apq != 0.0) {                                        // warp-uniform
          const double app = A[p][p], aqq = A[q][q];
          const double theta = (aqq - app) / (2.0 * apq);
          const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
          const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
          __syncwarp();
          if (lane < d) {
            const int k = lane;
            if (k != p && k != q) {
              const double akp = A[k][p], akq = A[k][q];
              const double np_ = c * akp - sn * akq, nq_ = sn * akp + c * akq;
              A[k][p] = np_; A[p][k] = np_;
              A[k][q] = nq_; A[q][k] = nq_;
            }
            const double vkp = V[k][p], vkq = V[k][q];
            V[k][p] = c * vkp - sn * vkq;
            V[k][q] = sn * vkp + c * vkq;
          }
          if (lane == 0) {
            A[p][p] = app - t * apq;
            A[q][q] = aqq + t * apq;
            A[p][q] = 0.0; A[q][p] = 0.0;
          }
          __syncwarp();
        }
      }
  }
  // eigenvalues descending (rank by counting; ties broken by index).  A permutation only if every key
  // compares, so NaN ranks as -inf, as in gen_eig_small_kernel: otherwise ranks collide and order[] keeps
  // unwritten slots that index V below
  if (lane < d) {
    const double mine = A[lane][lane];
    const double km = (mine == mine) ? mine : -INFINITY;
    int r = 0;
    for (int j = 0; j < d; ++j) {
      const double o = (A[j][j] == A[j][j]) ? A[j][j] : -INFINITY;
      r += (o > km) || (o == km && j < lane);
    }
    order[r] = lane;
    ev[r] = mine;
  }
  __syncwarp();
  // generalised eigenvectors W = Li^T U (columns in descending order) into L (reused)
  if (lane < d) {
    const int i = lane;
    for (int r = 0; r < d; ++r) {
      const int col = order[r];
      double s = 0.0;
      for (int k = i; k < d; ++k) s += Li[k][i] * V[k][col];
      L[i][r] = s;
    }
  }
  __syncwarp();
  const int used = (n_eig > 0 && n_eig < d) ? n_eig : d;
  if (lane == 0) {
    double loss = 0.0;
    for (int r = 0; r < used; ++r) loss -= ev[r] * ev[r];
    res[0] = s_bad ? NAN : loss;
    res[1] = (double)s_bad;
    res[2] = sw;
    res[3] = swl;
  }
  double* o_ev = res + 4;
  double* o_mu = o_ev + d;
  double* o_g0 = o_mu + d;
  double* o_gt = o_g0 + dd;
  if (lane < d) {
    const int i = lane;
    o_ev[i] = s_bad ? NAN : ev[i];
    o_mu[i] = mu[i];
    for (int j = 0; j < d; ++j) {
      double g0 = 0.0, gt = 0.0;
      for (int r = 0; r < used; ++r) {
        const double vv = L[i][r] * L[j][r];
        g0 += 2.0 * ev[r] * ev[r] * vv;
        gt -= 2.0 * ev[r] * vv;
      }
      o_g0[i * d + j] = s_bad ? 0.0 : g0;           // a singular batch contributes no gradient
      o_gt[i * d + j] = s_bad ? 0.0 : gt;
    }
  }
}

// ---- small generalised symmetric eigenproblem  H s = theta G s  (b <= 32, G SPD), batched ---------
// The Rayleigh-Ritz step of the shift-and-invert eigen stage (linalg.py) and of any other small
// pencil: Cholesky of G, A = L^-1 H L^-T, cyclic Jacobi, S = L^-T U with the eigenvalues in
// DESCENDING order -- one launch per batch instead of cholesky_ex + solve_triangular + two GEMMs +
// eigh (whose error check is a host synchronisation) + flips.  One warp per pencil.
__global__ void __launch_bounds__(32)
gen_eig_small_kernel(const double* __restrict__ Hm, const double* __restrict__ Gm, int b,
                     double* __restrict__ theta, double* __restrict__ Sm, double* __restrict__ status) {
  __shared__ double G[32][33], H[32][33], L[32][33], A[32][33], V[32][33];
  __shared__ int order[32];
  __shared__ int s_bad;
  const int lane = threadIdx.x;
  const size_t base = (size_t)blockIdx.x * b * b;
  double (*Li)[33] = G;                                  // G is dead once factorised
  if (lane == 0) s_bad = 0;
  if (lane < b)
    for (int j = 0; j < b; ++j) {
      G[lane][j] = 0.5 * (Gm[base + lane * b + j] + Gm[base + j * b + lane]);
      H[lane][j] = 0.5 * (Hm[base + lane * b + j] + Hm[base + j * b + lane]);
    }
  __syncwarp();
  for (int j = 0; j < b; ++j) {
    if (lane == j) {
      double s = G[j][j];
      for (int k = 0; k < j; ++k) s -= L[j][k] * L[j][k];
      if (!(s > 0.0)) { s_bad = 1; s = 1.0; }
      L[j][j] = sqrt(s);
    }
    __syncwarp();
    if (lane > j && lane < b) {
      double s = G[lane][j];
      for (int k = 0; k < j; ++k) s -= L[lane][k] * L[j][k];
      L[lane][j] = s / L[j][j];
    }
    if (lane < j) L[lane][j] = 0.0;
    __syncwarp();
  }
  if (lane < b) {
    const int c = lane;
    for (int i = 0; i < b; ++i) {
      double s = (i == c) ? 1.0 : 0.0;
      for (int k = c; k < i; ++k) s -= L[i][k] * Li[k][c];
      Li[i][c] = (i < c) ? 0.0 : s / L[i][i];
    }
  }
  __syncwarp();
  if (lane < b)
    for (int j = 0; j < b; ++j) {
      double s = 0.0;
      for (int k = 0; k <= lane; ++k) s += Li[lane][k] * H[k][j];
      V[lane][j] = s;
    }
  __syncwarp();
  if (lane < b)
    for (int j = 0; j < b; ++j) {
      double s = 0.0;
      for (int k = 0; k <= j; ++k) s += V[lane][k] * Li[j][k];
      A[lane][j] = s;
    }
  __syncwarp();
  if (lane < b)
    for (int j = lane + 1; j < b; ++j) A[lane][j] = 0.5 * (A[lane][j] + A[j][lane]);
  __syncwarp();
  if (lane < b) {
    for (int j = 0; j < lane; ++j) A[lane][j] = A[j][lane];
    for (int j = 0; j < b; ++j) V[lane][j] = (lane == j) ? 1.0 : 0.0;
  }
  __syncwarp();
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, diag = 0.0;
    if (lane < b) {
      for (int j = 0; j < b; ++j) { if (j != lane) off += A[lane][j] * A[lane][j]; }
      diag = A[lane][lane] * A[lane][lane];
    }
    off = warp_sum(off);
    diag = warp_sum(diag);
    if (off <= 1e-32 * diag || off == 0.0) break;
    for (int p = 0; p < b - 1; ++p)
      for (int q = p + 1; q < b; ++q) {
        const double apq = A[p][q];
        if (apq != 0.0) {
          const double app = A[p][p], aqq = A[q][q];
          const double th = (aqq - app) / (2.0 * apq);
          const double t = (th >= 0.0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0));
          const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
          __syncwarp();
          if (lane < b) {
            const int k = lane;
            if (k != p && k != q) {
              const double akp = A[k][p], akq = A[k][q];
              const double np_ = c * akp - sn * akq, nq_ = sn * akp + c * akq;
              A[k][p] = np_; A[p][k] = np_;
              A[k][q] = nq_; A[q][k] = nq_;
            }
            const double vkp = V[k][p], vkq = V[k][q];
            V[k][p] = c * vkp - sn * vkq;
            V[k][q] = sn * vkp + c * vkq;
          }
          if (lane == 0) {
            A[p][p] = app - t * apq;
            A[q][q] = aqq + t * apq;
            A[p][q] = 0.0; A[q][p] = 0.0;
          }
          __syncwarp();
        }
      }
  }
  if (lane < b) {
    // rank by value, ties by index: a permutation only if every key compares, so NaN (a pencil that is not
    // definite, e.g. from a failed factorisation upstream; flagged through the residuals) ranks as -inf --
    // otherwise ranks collide and order[] keeps unwritten slots that index V below
    const double mine = A[lane][lane];
    const double km = (mine == mine) ? mine : -INFINITY;
    int r = 0;
    for (int j = 0; j < b; ++j) {
      const double o = (A[j][j] == A[j][j]) ? A[j][j] : -INFINITY;
      r += (o > km) || (o == km && j < lane);
    }
    order[r] = lane;
    theta[(size_t)blockIdx.x * b + r] = mine;
  }
  __syncwarp();
  if (lane < b)
    for (int r = 0; r < b; ++r) {
      const int col = order[r];
      double s = 0.0;
      for (int k = lane; k < b; ++k) s += Li[k][lane] * V[k][col];
      Sm[base + lane * b + r] = s;
    }
  if (lane == 0) status[blockIdx.x] = (double)s_bad;
}

}  // namespace dcg

using namespace dcg;

extern "C" int dcg_gen_eig_small_f64(const double* H, const double* G, int b, int batch,
                                     double* theta, double* S, double* status, void* stream) {
  if (!H || !G || !theta || !S || !status) return DCG_E_NULL;
  if (b < 1 || b > 32 || batch < 1) return DCG_E_SHAPE;
  gen_eig_small_kernel<<<batch, 32, 0, (cudaStream_t)stream>>>(H, G, b, theta, S, status);
  DCG_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t dcg_ticaloss_out_doubles(int d) {
  if (d < 1 || d > 32) return 0;
  return (size_t)(4 + 2 * d + 2 * d * d);
}

extern "C" int dcg_ticaloss_f64(const double* sums, int d, double reg, int n_eig, double* res, void* stream) {
  if (!sums || !res) return DCG_E_NULL;
  if (d < 1 || d > 32) return DCG_E_SHAPE;
  ticaloss_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(sums, d, reg, n_eig, res);
  DCG_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t dcg_ticacov_out_doubles(int d) {
  if (d < 1 || d > 32) return 0;
  return (size_t)(2 + d + 2 * d * d + 2 * d);
}

extern "C" size_t dcg_ticacov_workspace_bytes(int64_t B, int d) {
  if (B <= 0 || d < 1 || d > 32) return 0;
  return (size_t)ticacov_ctas(B) * dcg_ticacov_out_doubles(d) * sizeof(double);
}

extern "C" int dcg_ticacov_f32(const float* f, const float* g, const float* w, const float* wl,
                               int64_t B, int d, double* out, void* ws, size_t ws_bytes, void* stream) {
  if (!f || !g || !out) return DCG_E_NULL;
  if (B <= 0 || d < 1 || d > 32) return DCG_E_SHAPE;
  if (!ws || ws_bytes < dcg_ticacov_workspace_bytes(B, d)) return DCG_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int G = (int)ticacov_ctas(B);
  const int n_out = (int)dcg_ticacov_out_doubles(d);
  const size_t smem = (size_t)kTcRowsPerCta * (2 * d + 2) * sizeof(float);
  DCG_CUDA_TRY(ensure_dynamic_smem((const void*)ticacov_kernel, (size_t)(smem)));
  ticacov_kernel<<<G, kTcThreads, smem, st>>>(f, g, w, wl, B, d, (double*)ws, G);
  DCG_LAUNCH_CHECK();
  ticacov_reduce_kernel<<<(unsigned)ceil_div(n_out, kTcThreads / 32), kTcThreads, 0, st>>>((const double*)ws, G,
                                                                                          n_out, out);
  DCG_LAUNCH_CHECK();
  return 0;
}
