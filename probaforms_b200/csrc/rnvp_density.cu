// Predictive log scores of k draws per row (probaforms_b200/predictive.py predictive_density): the Gaussian-KDE log
// score, the Dawid-Sebastiani score and the per-feature 1-D KDE log scores of an observation y.  The draws arrive as a
// row block laid out d_draws[(j * rows + r) * D + d], as for rnvp_draw_joint.
//
// One CTA of 256 threads per row, everything in fp64 on the float32 draws:
//   1. the mean, thread (s, d) summing draws s, s + S, ... (S = 256 / D slices), thread d adding the slices in order;
//   2. S = sum_j (x_j - mean)(x_j - mean)^T / (k - 1): chunks of 64 centred draws in shared memory, thread (ty, tx) of
//      a 16 x 16 grid owns the pairs (ty + 16 a, tx + 16 b), b <= a < TR (TR = ceil(D / 16) rounded to a power of two),
//      so only the lower triangle of 16 x 16 blocks is formed;
//   3. the 1-D KDE of each feature (online max-shifted logsumexp, slices merged in order);
//   4. S = L L^T, right-looking Cholesky on the packed lower triangle; a pivot L_ii^2 <= 1e-12 S_ii is degenerate;
//   5. L^-1, one column per thread by forward substitution, stored transposed with an odd row stride; the DSS;
//   6. q_j = ||L^-1 (y - x_j)||^2: chunks of 64 draws, thread (ty, tx) owns draws ty + 16 a (a < 4) and outputs
//      tx + 16 b (b < TR); the 16-column blocks above the diagonal of L^-1 are skipped.  The 16 partial squares of a
//      draw are summed by a fixed shuffle tree, and 16 threads keep online logsumexps that are merged in order.
// Every sum has a fixed order and a row's arithmetic does not depend on its position in the block, so repeated calls
// and any split into row blocks give the same bits.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/rnvp.h"

int rnvp_fail(int code, const char* msg);

namespace {

constexpr int K_THREADS = 256;
constexpr int K_CHUNK = 64;                 // draws per staged chunk of the covariance and whitening passes
constexpr int K_SMEM_MAX = 232448;          // opt-in dynamic shared memory per CTA on sm_100 (227 KB)
constexpr double LOG_2PI = 1.8378770664093454836;
constexpr double DEGENERATE = 1e-12;        // Cholesky pivot L_ii^2 <= DEGENERATE * S_ii: the row's S is degenerate
constexpr unsigned FULL = 0xffffffffu;

struct DensityArgs {
  const float* draws;
  const float* y;
  double* log_score;
  double* dss;
  double* marginal;
  int64_t k, rows;
  int D;
  double log_f, inv_f2, log_f1, f1;
};

__device__ __forceinline__ int pk(int i, int j) { return i * (i + 1) / 2 + j; }   // packed lower triangle, j <= i

// running max-shifted sum of exp: (m, s) stands for log(s) + m
__device__ __forceinline__ void lse_add(double& m, double& s, double v) {
  if (!(v > -INFINITY)) return;
  if (v > m) {
    s = __fma_rn(s, exp(__dsub_rn(m, v)), 1.0);
    m = v;
  } else {
    s = __dadd_rn(s, exp(__dsub_rn(v, m)));
  }
}
__device__ __forceinline__ void lse_merge(double& m, double& s, double m2, double s2) {
  if (!(m2 > -INFINITY)) return;
  if (!(m > -INFINITY)) { m = m2; s = s2; return; }
  if (m2 > m) {
    s = __fma_rn(s, exp(__dsub_rn(m, m2)), s2);
    m = m2;
  } else {
    s = __fma_rn(s2, exp(__dsub_rn(m2, m)), s);
  }
}

// Shared memory (doubles): s_mean, s_y, s_diag [D]; s_m, s_s [K_THREADS]; region A: max(D (D + 1) / 2, K_CHUNK Dp);
// region B: max(Dp (Dp + 1), K_CHUNK Dp), Dp = 16 TR.  A holds S, then L (packed), then the whitening chunks; B holds
// the covariance chunks, then L^-1 transposed (row l, column i at l * (Dp + 1) + i).
__host__ __device__ inline int64_t density_smem_doubles(int D, int TR) {
  const int64_t Dp = 16 * TR;
  const int64_t a = max((int64_t)D * (D + 1) / 2, K_CHUNK * Dp), b = max(Dp * (Dp + 1), K_CHUNK * Dp);
  return 3 * (int64_t)D + 2 * K_THREADS + a + b;
}

template <int TR>
__global__ void __launch_bounds__(K_THREADS) density_kernel(const DensityArgs a) {
  extern __shared__ double s_dyn[];
  __shared__ int s_flag;
  constexpr int Dp = 16 * TR, LD = Dp + 1, JA = K_CHUNK / 16;
  const int D = a.D, t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t r = blockIdx.x, k = a.k;
  double* s_mean = s_dyn;
  double* s_y = s_mean + D;
  double* s_diag = s_y + D;
  double* s_m = s_diag + D;
  double* s_s = s_m + K_THREADS;
  double* A = s_s + K_THREADS;
  double* B = A + max(D * (D + 1) / 2, K_CHUNK * Dp);
  const float* xr = a.draws + r * D;
  const int64_t xs = a.rows * D;             // stride between draws of one row
  const float* y = a.y + r * D;
  double* marg = a.marginal ? a.marginal + r * D : nullptr;

  // 1. mean; any non-finite draw or y makes the whole row NaN
  const int S = K_THREADS / D;
  double sum = 0.0;
  bool bad = false;
  if (t < S * D) {
    const int s = t / D, d = t - s * D;
    for (int64_t j = s; j < k; j += S) {
      const float x = xr[j * xs + d];
      bad |= !isfinite(x);
      sum = __dadd_rn(sum, (double)x);
    }
  }
  for (int d = t; d < D; d += K_THREADS) {
    s_y[d] = (double)y[d];
    bad |= !isfinite(y[d]);
  }
  s_m[t] = sum;
  if (__syncthreads_or(bad)) {
    if (t == 0) a.log_score[r] = a.dss[r] = (double)NAN;
    if (marg)
      for (int d = t; d < D; d += K_THREADS) marg[d] = (double)NAN;
    return;
  }
  if (t < D) {
    double tot = 0.0;
    for (int s = 0; s < S; ++s) tot = __dadd_rn(tot, s_m[s * D + t]);
    s_mean[t] = __ddiv_rn(tot, (double)k);
  }
  __syncthreads();

  // 2. covariance (ddof = 1), lower 16 x 16 blocks only; chunks staged in B as [jj][Dp], zero-padded
  {
    double acc[TR][TR];
#pragma unroll
    for (int u = 0; u < TR; ++u)
#pragma unroll
      for (int v = 0; v < TR; ++v) acc[u][v] = 0.0;
    for (int64_t j0 = 0; j0 < k; j0 += K_CHUNK) {
      const int nj = (int)min((int64_t)K_CHUNK, k - j0);
      for (int i = t; i < K_CHUNK * Dp; i += K_THREADS) {
        const int jj = i / Dp, d = i - jj * Dp;
        B[i] = jj < nj && d < D ? __dsub_rn((double)xr[(j0 + jj) * xs + d], s_mean[d]) : 0.0;
      }
      __syncthreads();
      for (int jj = 0; jj < nj; ++jj) {
        const double* c = B + jj * Dp;
        double ca[TR], cb[TR];
#pragma unroll
        for (int u = 0; u < TR; ++u) {
          ca[u] = c[ty + 16 * u];
          cb[u] = c[tx + 16 * u];
        }
#pragma unroll
        for (int u = 0; u < TR; ++u)
#pragma unroll
          for (int v = 0; v <= u; ++v) acc[u][v] = __fma_rn(ca[u], cb[v], acc[u][v]);
      }
      __syncthreads();
    }
    const double km1 = (double)(k - 1);
#pragma unroll
    for (int u = 0; u < TR; ++u)
#pragma unroll
      for (int v = 0; v <= u; ++v) {
        const int d = ty + 16 * u, e = tx + 16 * v;
        if (d < D && e <= d) {
          const double c = __ddiv_rn(acc[u][v], km1);
          A[pk(d, e)] = c;
          if (e == d) s_diag[d] = c;
        }
      }
  }
  __syncthreads();

  // 3. per-feature 1-D KDE, bandwidth f1 sigma_d; NaN for a constant feature
  if (marg) {
    double m = -INFINITY, s = 0.0;
    if (t < S * D) {
      const int sl = t / D, d = t - sl * D;
      const double inv_h = __drcp_rn(__dmul_rn(a.f1, sqrt(s_diag[d])));
      for (int64_t j = sl; j < k; j += S) {
        const double u = __dmul_rn(__dsub_rn(s_y[d], (double)xr[j * xs + d]), inv_h);
        lse_add(m, s, __dmul_rn(-0.5, __dmul_rn(u, u)));
      }
    }
    s_m[t] = m;
    s_s[t] = s;
    __syncthreads();
    if (t < D) {
      double mm = -INFINITY, ss = 0.0;
      for (int sl = 0; sl < S; ++sl) lse_merge(mm, ss, s_m[sl * D + t], s_s[sl * D + t]);
      const double lse = __dadd_rn(mm, log(ss));
      const double log_h = __dadd_rn(a.log_f1, 0.5 * log(s_diag[t]));
      marg[t] = s_diag[t] > 0.0 ? -(lse - log((double)k) - log_h - 0.5 * LOG_2PI) : (double)NAN;
    }
    __syncthreads();
  }

  // 4. Cholesky S = L L^T in place (packed)
  if (t == 0) s_flag = 0;
  __syncthreads();
  for (int j = 0; j < D; ++j) {
    if (t == 0) {
      const double p = A[pk(j, j)];
      if (!(p > DEGENERATE * s_diag[j])) s_flag = 1;
      else A[pk(j, j)] = sqrt(p);
    }
    __syncthreads();
    if (s_flag) break;
    const double ljj = A[pk(j, j)];
    for (int i = j + 1 + t; i < D; i += K_THREADS) A[pk(i, j)] = __ddiv_rn(A[pk(i, j)], ljj);
    __syncthreads();
    const int m = D - j - 1;
    for (int e = t; e < m * m; e += K_THREADS) {
      const int i = j + 1 + e / m, l = j + 1 + e % m;
      if (l <= i) A[pk(i, l)] = __fma_rn(-A[pk(i, j)], A[pk(l, j)], A[pk(i, l)]);
    }
    __syncthreads();
  }
  if (s_flag) {
    if (t == 0) a.log_score[r] = a.dss[r] = (double)NAN;
    return;
  }

  // 5. log det L, L^-1 (column c by thread c, written as row c of B), then the DSS
  double logdet = 0.0;
  if (t == 0)
    for (int i = 0; i < D; ++i) logdet = __dadd_rn(logdet, log(A[pk(i, i)]));
  if (t < Dp) {
    double* col = B + t * LD;
    for (int i = 0; i < Dp; ++i) col[i] = 0.0;
    if (t < D) {
      col[t] = __drcp_rn(A[pk(t, t)]);
      for (int i = t + 1; i < D; ++i) {
        double s = 0.0;
        for (int l = t; l < i; ++l) s = __fma_rn(A[pk(i, l)], col[l], s);
        col[i] = -__ddiv_rn(s, A[pk(i, i)]);
      }
    }
  }
  __syncthreads();
  if (t < D) {
    double w = 0.0;
    for (int l = 0; l <= t; ++l) w = __fma_rn(B[l * LD + t], __dsub_rn(s_y[l], s_mean[l]), w);
    s_m[t] = __dmul_rn(w, w);
  }
  __syncthreads();
  if (t == 0) {
    double q = 0.0;
    for (int i = 0; i < D; ++i) q = __dadd_rn(q, s_m[i]);
    a.dss[r] = __fma_rn(2.0, logdet, q);
    s_s[0] = logdet;
  }
  __syncthreads();
  logdet = s_s[0];

  // 6. whitening of y - x_j and the KDE's logsumexp; chunks staged in A as [jj][Dp], zero-padded
  double m = -INFINITY, s = 0.0;
  for (int64_t j0 = 0; j0 < k; j0 += K_CHUNK) {
    const int nj = (int)min((int64_t)K_CHUNK, k - j0);
    __syncthreads();
    for (int i = t; i < K_CHUNK * Dp; i += K_THREADS) {
      const int jj = i / Dp, d = i - jj * Dp;
      A[i] = jj < nj && d < D ? __dsub_rn(s_y[d], (double)xr[(j0 + jj) * xs + d]) : 0.0;
    }
    __syncthreads();
    double acc[JA][TR];
#pragma unroll
    for (int u = 0; u < JA; ++u)
#pragma unroll
      for (int v = 0; v < TR; ++v) acc[u][v] = 0.0;
#pragma unroll
    for (int lb = 0; lb < TR; ++lb) {
#pragma unroll 4
      for (int l16 = 0; l16 < 16; ++l16) {
        const int l = 16 * lb + l16;
        double va[JA], li[TR];
#pragma unroll
        for (int u = 0; u < JA; ++u) va[u] = A[(ty + 16 * u) * Dp + l];
#pragma unroll
        for (int v = lb; v < TR; ++v) li[v] = B[l * LD + tx + 16 * v];
#pragma unroll
        for (int u = 0; u < JA; ++u)
#pragma unroll
          for (int v = lb; v < TR; ++v) acc[u][v] = __fma_rn(li[v], va[u], acc[u][v]);
      }
    }
#pragma unroll
    for (int u = 0; u < JA; ++u) {
      double q = 0.0;
#pragma unroll
      for (int v = 0; v < TR; ++v) q = __fma_rn(acc[u][v], acc[u][v], q);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) q = __dadd_rn(q, __shfl_xor_sync(FULL, q, o));
      if (tx == 0 && ty + 16 * u < nj) lse_add(m, s, __dmul_rn(-0.5 * a.inv_f2, q));
    }
  }
  if (tx == 0) {
    s_m[ty] = m;
    s_s[ty] = s;
  }
  __syncthreads();
  if (t == 0) {
    double mm = -INFINITY, ss = 0.0;
    for (int i = 0; i < 16; ++i) lse_merge(mm, ss, s_m[i], s_s[i]);
    const double lse = __dadd_rn(mm, log(ss));
    a.log_score[r] = -(lse - log((double)k) - D * a.log_f - logdet - 0.5 * D * LOG_2PI);
  }
}

template <int TR>
int launch_density(const DensityArgs& a, cudaStream_t st) {
  const int smem = (int)(density_smem_doubles(a.D, TR) * sizeof(double));
  if (smem > K_SMEM_MAX) return rnvp_fail(RNVP_ESHAPE, "rnvp_draw_density: shared memory");
  cudaError_t e = cudaFuncSetAttribute(density_kernel<TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_draw_density: cudaFuncSetAttribute");
  density_kernel<TR><<<(unsigned)a.rows, K_THREADS, smem, st>>>(a);
  e = cudaGetLastError();
  return e == cudaSuccess ? 0 : rnvp_fail((int)e, "density_kernel");
}

}  // namespace

extern "C" int rnvp_draw_density(const float* d_draws, int64_t k, int64_t rows, int D, const float* d_y, double factor,
                                 double factor1, double* d_log_score, double* d_dss, double* d_marginal,
                                 void* stream) {
  if (D < 1 || D > RNVP_JOINT_MAX_D) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: D must be in [1, 128]");
  if (k <= D || k > RNVP_SUMMARY_MAX_DRAWS) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: k must be in (D, 8192]");
  if (rows < 0) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: rows must be >= 0");
  if (!(factor > 0.0) || !isfinite(factor)) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: factor must be > 0");
  if (d_marginal && (!(factor1 > 0.0) || !isfinite(factor1)))
    return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: factor1 must be > 0");
  if (rows == 0) return 0;
  if (!d_draws || !d_y || !d_log_score || !d_dss)
    return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: null d_draws, d_y, d_log_score or d_dss");
  if (rows > 0x7fffffff) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_density: too many rows");

  DensityArgs a{};
  a.draws = d_draws;
  a.y = d_y;
  a.log_score = d_log_score;
  a.dss = d_dss;
  a.marginal = d_marginal;
  a.k = k;
  a.rows = rows;
  a.D = D;
  a.log_f = log(factor);
  a.inv_f2 = 1.0 / (factor * factor);
  a.f1 = factor1;
  a.log_f1 = d_marginal ? log(factor1) : 0.0;
  cudaStream_t st = (cudaStream_t)stream;
  if (D <= 16) return launch_density<1>(a, st);
  if (D <= 32) return launch_density<2>(a, st);
  if (D <= 64) return launch_density<4>(a, st);
  return launch_density<8>(a, st);
}
