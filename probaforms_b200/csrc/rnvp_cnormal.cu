// ConditionalNormal (reference probaforms/models/cnormal.py): an MLP from the conditions C to the two heads mu and
// log_sigma of a Gaussian over x, trained on mean((z - mu)^2 / (2 sigma^2) + log sigma) with z = x (independent
// covariance) or z = (x - b_out) M, M = (W_out^T)^-1 (full covariance).  FP32 FMA throughout.
//
// A CTA owns a tile of up to R rows of a step's batch and keeps every activation of the tile in shared memory (row-major
// with an odd row stride, so that both the row-parallel and the column-parallel loops below are free of bank
// conflicts).  The fit sweep runs forward, loss and backward over its tile and writes per-CTA partial sums of every
// weight gradient (plus the loss); mlp_reduce_kernel adds the partials of all CTAs in CTA order and cn_tail applies
// what only the whole batch can: dW_out = -M G_M^T M, db_out = -M sum g_z, Adam, the loss hand-off, and in full mode the
// Gauss-Jordan inverse for the next step.  A batch of at most R rows is one launch (cn_step_kernel).
//
// A zero pivot in the inverse writes the index (+1) of the first step that cannot run to *status; every later kernel
// of the fit returns at once, so the parameters and losses stay those of the steps before it.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>

#include "../../include/rnvp.h"
#include "rnvp_adam.cuh"
#include "rnvp_mlp.cuh"
#include "rnvp_philox.cuh"

namespace {

struct CnShape {
  int D, Cd, nh, act, indep, R;
  int h[MLP_MAX_HIDDEN];
  int w[MLP_MAX_HIDDEN], b[MLP_MAX_HIDDEN];           // float offsets of model.model.{2k}.weight / .bias
  int mu_w, mu_b, ls_w, ls_b, out_w, out_b, P;
  int stride;                                         // floats of one CTA's partial record (P gradients + loss)
  int sweep_smem, tail_smem;
};

// shared-memory layout of one tile: C | H_0 .. H_{nh-1} | MU | LS | Z | XB, each [R][odd stride]
struct CnTile {
  float *c, *h[MLP_MAX_HIDDEN], *mu, *ls, *z, *xb;
  int ldc, ldh[MLP_MAX_HIDDEN], ldd;
};

__host__ __device__ inline int tile_floats(const CnShape& s, int R) {
  int f = R * odd_ld(s.Cd) + 4 * R * odd_ld(s.D);
  for (int k = 0; k < s.nh; ++k) f += R * odd_ld(s.h[k]);
  return f + 64;                                      // + the block reduction scratch
}

__device__ __forceinline__ CnTile carve(const CnShape& s, float* sm) {
  CnTile t;
  const int R = s.R;
  t.ldc = odd_ld(s.Cd);
  t.c = sm; sm += R * t.ldc;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {
    t.ldh[k] = k < s.nh ? odd_ld(s.h[k]) : 0;
    t.h[k] = sm;
    sm += R * t.ldh[k];
  }
  t.ldd = odd_ld(s.D);
  t.mu = sm; sm += R * t.ldd;
  t.ls = sm; sm += R * t.ldd;
  t.z = sm; sm += R * t.ldd;
  t.xb = sm;
  return t;
}

__device__ __forceinline__ void load_tile(const CnShape& s, const CnTile& t, const float* __restrict__ params,
                                 const float* __restrict__ X, const float* __restrict__ C,
                                 const int64_t* __restrict__ idx, int64_t row0, int nr) {
  for (int e = threadIdx.x; e < nr * s.Cd; e += blockDim.x) {
    const int r = e / s.Cd, j = e - r * s.Cd;
    const int64_t row = idx ? idx[row0 + r] : row0 + r;
    t.c[r * t.ldc + j] = C[row * s.Cd + j];
  }
  if (X)
    for (int e = threadIdx.x; e < nr * s.D; e += blockDim.x) {
      const int r = e / s.D, j = e - r * s.D;
      const int64_t row = idx ? idx[row0 + r] : row0 + r;
      const float x = X[row * s.D + j];
      if (s.indep) t.z[r * t.ldd + j] = x;
      else t.xb[r * t.ldd + j] = x - params[s.out_b + j];
    }
  __syncthreads();
}

// hidden layers and both heads (LS holds log sigma); in full mode with X, Z = XB M
__device__ __forceinline__ void forward_tile(const CnShape& s, const CnTile& t, const float* __restrict__ params,
                                    const float* __restrict__ M, bool want_z, int nr) {
  const float* in = t.c;
  int ldi = t.ldc, ni = s.Cd;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {          // unrolled: the per-layer arrays are indexed statically
    if (k >= s.nh) break;
    dense_rows(in, ldi, ni, params + s.w[k], params + s.b[k], t.h[k], t.ldh[k], s.h[k], nr, s.act);
    __syncthreads();
    in = t.h[k]; ldi = t.ldh[k]; ni = s.h[k];
  }
  const int D = s.D;
  const int nout = (want_z ? 3 : 2) * D;
  for (int e = threadIdx.x; e < nr * nout; e += blockDim.x) {
    const int i = e / nr, r = e - i * nr;
    float acc;
    if (i < 2 * D) {
      const int hd = i < D ? 0 : 1, k = i - hd * D;
      const float* w = params + (hd ? s.ls_w : s.mu_w) + (size_t)k * ni;
      const float* x = in + r * ldi;
      acc = params[(hd ? s.ls_b : s.mu_b) + k];
      for (int j = 0; j < ni; ++j) acc = fmaf(x[j], __ldg(w + j), acc);
      (hd ? t.ls : t.mu)[r * t.ldd + k] = acc;
    } else {
      const int k = i - 2 * D;
      const float* x = t.xb + r * t.ldd;
      acc = 0.0f;
      for (int j = 0; j < D; ++j) acc = fmaf(x[j], M[j * D + k], acc);
      t.z[r * t.ldd + k] = acc;
    }
  }
  __syncthreads();
}

// forward, loss and backward of one tile; writes the tile's gradient partials g[0..P) (the out slots hold G_M and
// sum g_z in full mode and are left alone in independent mode) and the tile's loss sum to g[P]
__device__ __forceinline__ void sweep_tile(const CnShape& s, float* sm, const float* __restrict__ params, const float* __restrict__ M,
                           const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx,
                           int64_t row0, int nr, float inv_bd, float* __restrict__ g) {
  const CnTile t = carve(s, sm);
  float* scratch = t.xb + s.R * t.ldd;                 // the 64 floats after the tile (tile_floats)
  load_tile(s, t, params, X, C, idx, row0, nr);
  forward_tile(s, t, params, M, !s.indep, nr);
  const int D = s.D;
  float lsum = 0.0f;
  for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
    const int r = e / D, k = e - r * D, o = r * t.ldd + k;
    const float mu = t.mu[o], ls = t.ls[o], is2 = expf(-2.0f * ls);
    const float d = t.z[o] - mu, dd = d * is2;
    lsum += fmaf(0.5f * d, dd, ls);
    t.mu[o] = -dd * inv_bd;                              // d loss / d mu
    t.ls[o] = fmaf(-d, dd, 1.0f) * inv_bd;               // d loss / d log_sigma
    if (!s.indep) t.z[o] = dd * inv_bd;                  // d loss / d z
  }
  const float tot = block_sum(lsum, scratch);
  if (threadIdx.x == 0) g[s.P] = tot;
  int hl = 0, ldl = 0;
  float* Hl = nullptr;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k)
    if (k == s.nh - 1) { hl = s.h[k]; Hl = t.h[k]; ldl = t.ldh[k]; }
  wgrad(t.mu, t.ldd, D, Hl, ldl, hl, nr, g + s.mu_w, g + s.mu_b);
  wgrad(t.ls, t.ldd, D, Hl, ldl, hl, nr, g + s.ls_w, g + s.ls_b);
  if (!s.indep) wgrad(t.xb, t.ldd, D, t.z, t.ldd, D, nr, g + s.out_w, nullptr);   // G_M[j][k] = sum_r xb[r][j] gz[r][k]
  if (!s.indep)
    for (int k = threadIdx.x; k < D; k += blockDim.x) {
      float acc = 0.0f;
      for (int r = 0; r < nr; ++r) acc += t.z[r * t.ldd + k];
      g[s.out_b + k] = acc;
    }
  __syncthreads();
  // d loss / d H_last through both heads
  for (int e = threadIdx.x; e < nr * hl; e += blockDim.x) {
    const int j = e / nr, r = e - j * nr;
    const float *gm = t.mu + r * t.ldd, *gl = t.ls + r * t.ldd;
    float acc = 0.0f;
    for (int i = 0; i < D; ++i)
      acc = fmaf(gm[i], __ldg(params + s.mu_w + (size_t)i * hl + j), fmaf(gl[i], __ldg(params + s.ls_w + (size_t)i * hl + j), acc));
    Hl[r * ldl + j] = acc * act_d(s.act, Hl[r * ldl + j]);
  }
  __syncthreads();
#pragma unroll
  for (int k = MLP_MAX_HIDDEN - 1; k >= 0; --k) {
    if (k >= s.nh) continue;
    const float* in = k ? t.h[k - 1] : t.c;
    const int ldi = k ? t.ldh[k - 1] : t.ldc, ni = k ? s.h[k - 1] : s.Cd;
    wgrad(t.h[k], t.ldh[k], s.h[k], in, ldi, ni, nr, g + s.w[k], g + s.b[k]);
    __syncthreads();
    if (k) {
      back_rows(t.h[k], t.ldh[k], s.h[k], params + s.w[k], t.h[k - 1], t.ldh[k - 1], ni, nr, s.act);
      __syncthreads();
    }
  }
}

// M = (W_out^T)^-1 by Gauss-Jordan with partial pivoting in shared memory (aug [D][2D]); false on an exact-zero pivot
// params is read after the same kernel's Adam update (cn_step_kernel): plain loads, no read-only path
__device__ __forceinline__ bool invert_out(const CnShape& s, const float* params, float* __restrict__ M, float* sm) {
  const int D = s.D, W2 = 2 * D;
  float* A = sm;
  float* f = sm + D * W2;
  __shared__ int piv;
  __shared__ float pval;
  for (int e = threadIdx.x; e < D * W2; e += blockDim.x) {
    const int r = e / W2, c = e - r * W2;
    A[e] = c < D ? params[s.out_w + c * D + r] : (c - D == r ? 1.0f : 0.0f);   // W^T | I
  }
  __syncthreads();
  for (int c = 0; c < D; ++c) {
    if (threadIdx.x < 32) {
      int best = c;
      float bv = -1.0f;
      for (int r = c + threadIdx.x; r < D; r += 32) {
        const float a = fabsf(A[r * W2 + c]);
        if (a > bv) { bv = a; best = r; }
      }
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int ob = __shfl_xor_sync(0xffffffffu, best, o);
        if (ov > bv || (ov == bv && ob < best)) { bv = ov; best = ob; }
      }
      if (threadIdx.x == 0) { piv = best; pval = A[best * W2 + c]; }
    }
    __syncthreads();
    if (pval == 0.0f) return false;                    // uniform: every thread reads the same shared value
    const int p = piv;
    const float ip = 1.0f / pval;
    for (int e = threadIdx.x; e < W2; e += blockDim.x) {
      const float a = A[p * W2 + e], b = A[c * W2 + e];
      A[c * W2 + e] = a * ip;
      if (p != c) A[p * W2 + e] = b;
    }
    __syncthreads();
    for (int r = threadIdx.x; r < D; r += blockDim.x) f[r] = A[r * W2 + c];
    __syncthreads();
    for (int e = threadIdx.x; e < D * W2; e += blockDim.x) {
      const int r = e / W2, col = e - r * W2;
      if (r != c) A[e] = fmaf(-f[r], A[c * W2 + col], A[e]);
    }
    __syncthreads();
  }
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) M[e] = A[(e / D) * W2 + D + e % D];
  __syncthreads();
  return true;
}

struct CnStep {
  RnvpAdamCoef k;
  float inv_bd;
  int adam;                       // 0: gradient only (rnvp_cn_grad)
  long long step;                 // index of this step within the fit (0-based), for *status
};

// what needs the whole batch's gradient g (reduced, P + 1 floats): out-layer chain rule, Adam, loss, next inverse
__device__ __forceinline__ void cn_tail(const CnShape& s, float* sm, float* __restrict__ params, float* __restrict__ m,
                        float* __restrict__ v, float* __restrict__ M, float* __restrict__ g, float* __restrict__ gflat,
                        float* loss_dst, int* status, const CnStep& st) {
  const int D = s.D;
  if (!s.indep) {
    float* T = sm;                                     // T = G_M^T M
    float* db = sm + D * D;
    for (int e = threadIdx.x; e < D * D; e += blockDim.x) {
      const int a = e / D, b = e - a * D;
      float acc = 0.0f;
      for (int j = 0; j < D; ++j) acc = fmaf(g[s.out_w + j * D + a], M[j * D + b], acc);
      T[e] = acc;
    }
    for (int a = threadIdx.x; a < D; a += blockDim.x) {
      float acc = 0.0f;
      for (int j = 0; j < D; ++j) acc = fmaf(M[a * D + j], g[s.out_b + j], acc);
      db[a] = -acc;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < D * D; e += blockDim.x) {
      const int a = e / D, b = e - a * D;
      float acc = 0.0f;
      for (int j = 0; j < D; ++j) acc = fmaf(M[a * D + j], T[j * D + b], acc);
      g[s.out_w + e] = -acc;
    }
    for (int a = threadIdx.x; a < D; a += blockDim.x) g[s.out_b + a] = db[a];
    __syncthreads();
  }
  const int n_upd = s.indep ? s.out_w : s.P;          // the out tensors are last; without a gradient Adam skips them
  if (threadIdx.x == 0 && loss_dst) *loss_dst = g[s.P] * st.inv_bd;
  if (!st.adam) {
    for (int i = threadIdx.x; i < s.P; i += blockDim.x) gflat[i] = i < n_upd ? g[i] : 0.0f;
    return;
  }
  for (int i = threadIdx.x; i < n_upd; i += blockDim.x) {
    float mi = m[i], vi = v[i];
    params[i] = rnvp_adam_update(g[i], params[i], mi, vi, st.k);
    m[i] = mi; v[i] = vi;
  }
  if (s.indep) return;
  __syncthreads();
  if (!invert_out(s, params, M, sm) && threadIdx.x == 0) *status = (int)(st.step + 2);   // step+1 cannot run
}

__global__ void __launch_bounds__(MLP_THREADS) cn_sweep_kernel(CnShape s, const float* __restrict__ params,
    const float* __restrict__ M, const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx,
    int64_t nb, float inv_bd, float* __restrict__ partials, const int* status) {
  if (status && *status) return;
  extern __shared__ __align__(16) float smem[];
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(nb - row0 < s.R ? nb - row0 : s.R);
  sweep_tile(s, smem, params, M, X, C, idx, row0, nr, inv_bd, partials + (size_t)blockIdx.x * s.stride);
}

__global__ void __launch_bounds__(MLP_TAIL_THREADS) cn_tail_kernel(CnShape s, float* params, float* m, float* v,
                                                                  float* M, float* g, float* gflat, float* loss_dst,
                                                                  int* status, CnStep st) {
  if (status && *status) return;
  extern __shared__ __align__(16) float smem[];
  cn_tail(s, smem, params, m, v, M, g, gflat, loss_dst, status, st);
}

// a whole step of a batch that fits one tile
__global__ void __launch_bounds__(MLP_TAIL_THREADS) cn_step_kernel(CnShape s, float* params, float* m, float* v,
    float* M, const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx, int nb,
    float* g, float* gflat, float* loss_dst, int* status, CnStep st) {
  if (status && *status) return;
  extern __shared__ __align__(16) float smem[];
  sweep_tile(s, smem, params, M, X, C, idx, 0, nb, st.inv_bd, g);
  __syncthreads();                                     // g (global) is read back by other threads of this CTA
  cn_tail(s, smem, params, m, v, M, g, gflat, loss_dst, status, st);
}

__global__ void cn_inverse_kernel(CnShape s, const float* params, float* M, int* status) {
  extern __shared__ __align__(16) float smem[];
  if (!invert_out(s, params, M, smem) && threadIdx.x == 0) *status = 1;
}

// Net.forward for inference: mu, sigma, x_tilde (noise from Philox keyed on (seed, row_offset + row, j), or eps),
// inv = (X - b_out) M; every output may be NULL
__global__ void __launch_bounds__(MLP_THREADS) cn_forward_kernel(CnShape s, const float* __restrict__ params,
    const float* __restrict__ M, const float* __restrict__ X, const float* __restrict__ C, int64_t N,
    unsigned long long seed, long long row_offset, const float* __restrict__ eps, float* mu_o, float* sigma_o,
    float* xt_o, float* inv_o) {
  extern __shared__ __align__(16) float smem[];
  const CnTile t = carve(s, smem);
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(N - row0 < s.R ? N - row0 : s.R);
  const bool want_inv = inv_o && X;
  CnShape sf = s;
  sf.indep = 0;                                        // X - b_out goes to XB in both modes
  load_tile(sf, t, params, want_inv ? X : nullptr, C, nullptr, row0, nr);
  forward_tile(s, t, params, M, want_inv, nr);
  const int D = s.D;
  for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
    const int r = e / D, k = e - r * D, o = r * t.ldd + k;
    const int64_t row = row0 + r;
    const float mu = t.mu[o], sg = expf(t.ls[o]);
    if (mu_o) mu_o[row * D + k] = mu;
    if (sigma_o) sigma_o[row * D + k] = sg;
    if (want_inv) inv_o[row * D + k] = t.z[o];
    const float ep = eps ? eps[row * D + k] : rnvp_rng::normal1(seed, row_offset + row, k);
    t.ls[o] = fmaf(ep, sg, mu);                        // x_tilde before the out layer
  }
  if (!xt_o) return;
  __syncthreads();
  for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
    const int r = e / D, k = e - r * D;
    float y = t.ls[r * t.ldd + k];
    if (!s.indep) {
      const float* x = t.ls + r * t.ldd;
      y = params[s.out_b + k];
      for (int j = 0; j < D; ++j) y = fmaf(x[j], __ldg(params + s.out_w + k * D + j), y);
    }
    xt_o[(row0 + r) * D + k] = y;
  }
}

// log|det W_out| and M64 = (W_out^T)^-1 in fp64 for the exact log-density: LU of A = W_out^T in shared memory with the
// partial pivoting of invert_out (largest |a| in the column, the lowest row on a tie), then column c of A^-1 by thread
// c, forward and back substitution through ws.  ws[0] = sum_c log|u_cc| in column order, ws[1 + j * D + c] =
// M64[j][c]; *status = 1 on an exact-zero pivot.
__global__ void cn_logdet_kernel(CnShape s, const float* __restrict__ params, double* ws, int* status) {
  extern __shared__ __align__(16) double smd[];
  __shared__ int piv, perm[MLP_MAX_D];
  __shared__ double pval;
  const int D = s.D;
  double* A = smd;
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) {
    const int r = e / D, c = e - r * D;
    A[e] = (double)params[s.out_w + c * D + r];        // W^T
  }
  for (int r = threadIdx.x; r < D; r += blockDim.x) perm[r] = r;
  __syncthreads();
  for (int c = 0; c < D; ++c) {
    if (threadIdx.x < 32) {
      int best = c;
      double bv = -1.0;
      for (int r = c + threadIdx.x; r < D; r += 32) {
        const double a = fabs(A[r * D + c]);
        if (a > bv) { bv = a; best = r; }
      }
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int ob = __shfl_xor_sync(0xffffffffu, best, o);
        if (ov > bv || (ov == bv && ob < best)) { bv = ov; best = ob; }
      }
      if (threadIdx.x == 0) { piv = best; pval = A[best * D + c]; }
    }
    __syncthreads();
    if (pval == 0.0) {                                 // uniform: every thread reads the same shared value
      if (threadIdx.x == 0) *status = 1;
      return;
    }
    const int p = piv;
    if (p != c) {
      for (int e = threadIdx.x; e < D; e += blockDim.x) {
        const double a = A[p * D + e];
        A[p * D + e] = A[c * D + e];
        A[c * D + e] = a;
      }
      if (threadIdx.x == 0) { const int q = perm[p]; perm[p] = perm[c]; perm[c] = q; }
    }
    __syncthreads();
    for (int r = c + 1 + threadIdx.x; r < D; r += blockDim.x) A[r * D + c] = __ddiv_rn(A[r * D + c], pval);
    __syncthreads();
    const int m = D - c - 1;
    for (int e = threadIdx.x; e < m * m; e += blockDim.x) {
      const int r = c + 1 + e / m, col = c + 1 + e % m;
      A[r * D + col] = __fma_rn(-A[r * D + c], A[c * D + col], A[r * D + col]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double ld = 0.0;
    for (int c = 0; c < D; ++c) ld = __dadd_rn(ld, log(fabs(A[c * D + c])));
    ws[0] = ld;
  }
  const int c = threadIdx.x;
  if (c < D) {                                         // P A = L U: L U x = P e_c, x = column c of A^-1
    double* x = ws + 1 + c;
    for (int i = 0; i < D; ++i) {
      double v = perm[i] == c ? 1.0 : 0.0;
      for (int l = 0; l < i; ++l) v = __fma_rn(-A[i * D + l], x[l * D], v);
      x[i * D] = v;
    }
    for (int i = D - 1; i >= 0; --i) {
      double v = x[i * D];
      for (int l = i + 1; l < D; ++l) v = __fma_rn(-A[i * D + l], x[l * D], v);
      x[i * D] = __ddiv_rn(v, A[i * D + i]);
    }
  }
}

// exact log-density of X given C: the fp32 net of cn_forward_kernel (mu and log_sigma with the same bits), then one
// warp per row in fp64: u = (x - b_out) M64 (u = x in independent mode), sum_d ((u_d - mu_d) / sigma_d)^2 and sum_d
// log_sigma_d lane-strided and summed by a fixed shuffle tree
__global__ void __launch_bounds__(MLP_THREADS) cn_log_prob_kernel(CnShape s, const float* __restrict__ params,
    const double* __restrict__ ws, const float* __restrict__ X, const float* __restrict__ C, int64_t N,
    double* __restrict__ logp, const int* status) {
  if (status && *status) return;
  extern __shared__ __align__(16) float smem[];
  const CnTile t = carve(s, smem);
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(N - row0 < s.R ? N - row0 : s.R);
  CnShape sx = s;
  sx.indep = 1;                                        // raw X goes to Z in both modes
  load_tile(sx, t, params, X, C, nullptr, row0, nr);
  forward_tile(s, t, params, nullptr, false, nr);
  const int D = s.D, lane = threadIdx.x & 31;
  const double* M = ws + 1;
  for (int r = threadIdx.x >> 5; r < nr; r += MLP_THREADS / 32) {
    const float* x = t.z + r * t.ldd;
    double q = 0.0, ls = 0.0;
    for (int c = lane; c < D; c += 32) {
      double u = x[c];
      if (!s.indep) {
        u = 0.0;
        for (int j = 0; j < D; ++j)
          u = __fma_rn(__dsub_rn((double)x[j], (double)params[s.out_b + j]), M[j * D + c], u);
      }
      const double l = t.ls[r * t.ldd + c];
      const double z = __dmul_rn(__dsub_rn(u, (double)t.mu[r * t.ldd + c]), exp(-l));
      q = __fma_rn(z, z, q);
      ls = __dadd_rn(ls, l);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      q = __dadd_rn(q, __shfl_down_sync(0xffffffffu, q, o));
      ls = __dadd_rn(ls, __shfl_down_sync(0xffffffffu, ls, o));
    }
    if (lane == 0) {
      double lp = -0.5 * q - ls - 0.5 * D * 1.8378770664093454836;   // log 2 pi
      if (!s.indep) lp -= ws[0];
      logp[row0 + r] = lp;
    }
  }
}

}  // namespace

struct rnvp_cn_desc {
  CnShape s;
};

namespace {

int check_cn(const rnvp_cn_desc* d) { return d ? 0 : rnvp_fail(RNVP_EINVAL, "null ConditionalNormal descriptor"); }

void launch_step(const rnvp_cn_desc* d, float* params, float* m, float* v, float* M, const float* X,
                 const float* C, const int64_t* idx, int64_t nb, float* gflat, float* loss_dst, int* status,
                 const CnStep& st, float* ws, cudaStream_t stream) {
  const CnShape& s = d->s;
  const int64_t nt = n_tiles(s.R, nb);
  float* g = ws;                                       // reduced gradient + loss (stride floats), then the partials
  if (nt == 1) {
    cn_step_kernel<<<1, MLP_TAIL_THREADS, std::max(s.sweep_smem, s.tail_smem), stream>>>(
        s, params, m, v, M, X, C, idx, (int)nb, g, gflat, loss_dst, status, st);
    return;
  }
  float* partials = ws + s.stride;
  cn_sweep_kernel<<<(unsigned)nt, MLP_THREADS, s.sweep_smem, stream>>>(s, params, M, X, C, idx, nb, st.inv_bd,
                                                                      partials, status);
  // the gradients and the loss; in independent mode the out slots (last) have no gradient
  launch_reduce(partials, (int)nt, s.stride, s.P, 0, s.indep ? s.out_w : s.P, 1, g, status, stream);
  cn_tail_kernel<<<1, MLP_TAIL_THREADS, s.tail_smem, stream>>>(s, params, m, v, M, g, gflat, loss_dst, status, st);
}

}  // namespace

extern "C" {

int rnvp_cn_desc_create(int D, int Cd, int n_hidden, const int* hidden, int act, int independent, rnvp_cn_desc** out) {
  if (!out) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_desc_create: out is null");
  *out = nullptr;
  if (!hidden || D < 1 || Cd < 1 || n_hidden < 1) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_desc_create: bad shape");
  if (act != RNVP_ACT_TANH && act != RNVP_ACT_RELU && act != RNVP_ACT_SIGMOID)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_desc_create: act must be RNVP_ACT_TANH, _RELU or _SIGMOID");
  if (D > MLP_MAX_D) return rnvp_fail(RNVP_ESHAPE, "ConditionalNormal: var_size D must be <= 128");
  if (Cd > MLP_MAX_CD) return rnvp_fail(RNVP_ESHAPE, "ConditionalNormal: cond_size must be <= 256");
  if (n_hidden > MLP_MAX_HIDDEN) return rnvp_fail(RNVP_ESHAPE, "ConditionalNormal: at most 4 hidden layers");
  CnShape s{};
  s.D = D; s.Cd = Cd; s.nh = n_hidden; s.act = act; s.indep = independent ? 1 : 0;
  int64_t off = 0;
  if (int rc = hidden_layout(n_hidden, hidden, Cd, s.h, s.w, s.b, off, "ConditionalNormal", "rnvp_cn_desc_create"))
    return rc;
  const int hl = hidden[n_hidden - 1];
  linear_layout(s.mu_w, s.mu_b, hl, D, off);
  linear_layout(s.ls_w, s.ls_b, hl, D, off);
  linear_layout(s.out_w, s.out_b, D, D, off);
  s.P = (int)off;
  s.stride = (s.P + 1 + 3) & ~3;
  s.R = rows_per_tile(s);
  s.sweep_smem = tile_floats(s, s.R) * 4;
  s.tail_smem = (2 * D * D + D) * 4;
  if (int rc = opt_in_smem({(const void*)cn_sweep_kernel, (const void*)cn_tail_kernel, (const void*)cn_step_kernel,
                            (const void*)cn_inverse_kernel, (const void*)cn_forward_kernel,
                            (const void*)cn_log_prob_kernel},
                           std::max(s.sweep_smem, s.tail_smem), "ConditionalNormal", "rnvp_cn_desc_create"))
    return rc;
  *out = new rnvp_cn_desc{s};
  return 0;
}

void rnvp_cn_desc_destroy(rnvp_cn_desc* d) { delete d; }

int64_t rnvp_cn_param_count(const rnvp_cn_desc* d) { return d ? d->s.P : -1; }

int64_t rnvp_cn_workspace_bytes(const rnvp_cn_desc* d, int64_t N) {
  if (!d || N < 0) return -1;
  const int64_t nt = n_tiles(d->s.R, N);
  return 4 * (int64_t)d->s.stride * (1 + (nt > 1 ? nt : 0));
}

int rnvp_cn_inverse(const rnvp_cn_desc* d, const float* d_params, float* d_M, int* d_status, void* stream) {
  if (check_cn(d)) return RNVP_EINVAL;
  if (!d_params || !d_M || !d_status) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_inverse: null buffer");
  cn_inverse_kernel<<<1, MLP_TAIL_THREADS, d->s.tail_smem, (cudaStream_t)stream>>>(d->s, d_params, d_M, d_status);
  return launched("cn_inverse_kernel launch");
}

int rnvp_cn_forward(const rnvp_cn_desc* d, const float* d_params, const float* d_M, const float* d_X, const float* d_C,
                    int64_t N, uint64_t seed, int64_t row_offset, const float* d_eps, float* d_mu, float* d_sigma,
                    float* d_xtilde, float* d_inv, void* stream) {
  if (check_cn(d)) return RNVP_EINVAL;
  if (!d_params || !d_C || N < 0 || (d_inv && (!d_X || !d_M)))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_forward: bad argument");
  if (N == 0) return 0;
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_forward: too many rows");
  cn_forward_kernel<<<(unsigned)n_tiles(d->s.R, N), MLP_THREADS, d->s.sweep_smem, (cudaStream_t)stream>>>(
      d->s, d_params, d_M, d_X, d_C, N, seed, row_offset, d_eps, d_mu, d_sigma, d_xtilde, d_inv);
  return launched("cn_forward_kernel launch");
}

int rnvp_cn_log_prob(const rnvp_cn_desc* d, const float* d_params, const float* d_X, const float* d_C, int64_t N,
                     double* d_logp, double* d_workspace, int* d_status, void* stream) {
  if (check_cn(d)) return RNVP_EINVAL;
  const bool full = !d->s.indep;
  if (!d_params || !d_X || !d_C || !d_logp || N < 0 || (full && (!d_workspace || !d_status)))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_log_prob: bad argument");
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_log_prob: too many rows");
  cudaStream_t st = (cudaStream_t)stream;
  if (full) {
    const int smem = d->s.D * d->s.D * (int)sizeof(double);
    const cudaError_t e = cudaFuncSetAttribute(cn_logdet_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_cn_log_prob: cudaFuncSetAttribute");
    cn_logdet_kernel<<<1, MLP_TAIL_THREADS, smem, st>>>(d->s, d_params, d_workspace, d_status);
    if (int rc = launched("cn_logdet_kernel launch")) return rc;
  }
  if (N == 0) return 0;
  cn_log_prob_kernel<<<(unsigned)n_tiles(d->s.R, N), MLP_THREADS, d->s.sweep_smem, st>>>(
      d->s, d_params, full ? d_workspace : nullptr, d_X, d_C, N, d_logp, full ? d_status : nullptr);
  return launched("cn_log_prob_kernel launch");
}

int rnvp_cn_grad(const rnvp_cn_desc* d, const float* d_params, const float* d_M, const float* d_X, const float* d_C,
                 const int64_t* d_idx, int64_t N, float* d_gflat, float* d_loss, void* d_workspace,
                 int64_t workspace_bytes, void* stream) {
  if (check_cn(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || !d_C || !d_gflat || N < 1 || (!d->s.indep && !d_M))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_grad: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_cn_workspace_bytes(d, N))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_grad: workspace smaller than rnvp_cn_workspace_bytes(N)");
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_grad: too many rows");
  CnStep st{};
  st.inv_bd = (float)(1.0 / ((double)N * d->s.D));
  st.adam = 0;
  launch_step(d, const_cast<float*>(d_params), nullptr, nullptr, const_cast<float*>(d_M), d_X, d_C, d_idx, N, d_gflat,
              d_loss, nullptr, st, (float*)d_workspace, (cudaStream_t)stream);
  return launched("ConditionalNormal gradient launch");
}

int rnvp_cn_fit_epoch(const rnvp_cn_desc* d, float* d_params, float* d_exp_avg, float* d_exp_avg_sq, float* d_M,
                      const float* d_X, const float* d_C, const int64_t* d_perm, int64_t n, int64_t batch_size,
                      double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step0,
                      float* d_losses, int* d_status, void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_cn(d)) return RNVP_EINVAL;
  if (!d_params || !d_exp_avg || !d_exp_avg_sq || !d_M || !d_X || !d_C || !d_perm || !d_losses || !d_status || n < 0 ||
      batch_size < 1 || step0 < 0)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_fit_epoch: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_cn_workspace_bytes(d, std::min(n, batch_size)))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cn_fit_epoch: workspace smaller than rnvp_cn_workspace_bytes(batch_size)");
  int64_t s = 0;
  for (int64_t b0 = 0; b0 < n; b0 += batch_size, ++s) {
    const int64_t nb = std::min(batch_size, n - b0);
    CnStep st{};
    st.k = adam_coef(lr, beta1, beta2, eps, weight_decay, step0 + s + 1);
    st.inv_bd = (float)(1.0 / ((double)nb * d->s.D));
    st.adam = 1;
    st.step = step0 + s;
    launch_step(d, d_params, d_exp_avg, d_exp_avg_sq, d_M, d_X, d_C, d_perm + b0, nb, nullptr, d_losses + s, d_status,
                st, (float*)d_workspace, (cudaStream_t)stream);
    if (int rc = launched("ConditionalNormal fit step launch")) return rc;
  }
  return 0;
}

// torch's CPU generator state (get_state() bytes: legacy mt19937 pod, then the cached normals) advanced by `words`
// 32-bit draws of at::mt19937: operator() decrements left_, regenerates the 624-word block when it reaches 0, then
// reads state_[next_++]
int rnvp_cn_rng_advance(uint8_t* state, int64_t state_bytes, int64_t numel) {
  constexpr int N = 624, Mm = 397;
  if (!state || state_bytes != 5056) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_rng_advance: not a torch CPU generator state");
  if (numel < 16) return rnvp_fail(RNVP_EINVAL, "rnvp_cn_rng_advance: numel < 16 takes torch's cached double path");
  int32_t left;
  uint64_t next, st64[N];
  memcpy(&left, state + 8, 4);
  memcpy(&next, state + 16, 8);
  memcpy(st64, state + 24, sizeof(st64));
  uint32_t mt[N];
  for (int i = 0; i < N; ++i) mt[i] = (uint32_t)st64[i];
  auto regen = [&]() {
    auto twist = [](uint32_t u, uint32_t v) {
      return (((u & 0x80000000u) | (v & 0x7fffffffu)) >> 1) ^ ((v & 1u) ? 0x9908b0dfu : 0u);
    };
    int k = 0;
    for (; k < N - Mm; ++k) mt[k] = mt[k + Mm] ^ twist(mt[k], mt[k + 1]);
    for (; k < N - 1; ++k) mt[k] = mt[k + Mm - N] ^ twist(mt[k], mt[k + 1]);
    mt[N - 1] = mt[Mm - 1] ^ twist(mt[N - 1], mt[0]);
  };
  int64_t words = numel + (numel % 16 ? 16 : 0);
  while (words > 0) {
    if (words < left) {                                // no regeneration: left stays >= 1
      left -= (int32_t)words; next += (uint64_t)words;
      break;
    }
    words -= left;                                     // left - 1 plain draws, then the draw that regenerates
    regen();
    left = N;
    next = 1;
  }
  for (int i = 0; i < N; ++i) st64[i] = mt[i];
  memcpy(state + 8, &left, 4);
  memcpy(state + 16, &next, 8);
  memcpy(state + 24, st64, sizeof(st64));
  return 0;
}

}  // extern "C"
