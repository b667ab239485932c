// Per-feature bootstrap metrics (probaforms/metrics/ks1d.py, div1d.py): KS, Cramer-von Mises, ROC AUC, Anderson-Darling,
// histogram KL / JS and KDE KL / JS.
//
// A bootstrap draw of a column is the original column with per-row counts c (bincount of the resampled indices).  The
// pooled column [x; y] of each feature is sorted once (by the caller); d_src holds each sorted position's row (< n: x).
// For draw b, a position contributes c_b[src] to the x or the y side.  Equal values form a tie group, and every
// statistic except the KDE pair is a function of, per tie group with a nonzero count, the cumulative x and y counts
// before the group (Bx, By) and the group's own counts (gx, gy):
//   KS     max(clip(-min d, 0, 1), max d),  d = F_x - F_y at the group end, F_x = linspace(0, 1, n + 1)[Bx + gx]
//   CvM    U = n sum_i (r_i - i)^2 + m sum_j (r_j - j)^2 with midranks r: over the x indices Bx+1..Bx+gx of a group
//          the sum is closed-form, kept as 4U in 128-bit integers (exact for every n + m < 2^31)
//   AUC    Mann-Whitney with half-weight ties: 2U = sum (2 gy Bx + gx gy)
//   AD     A2kN of scipy's midrank variant: sum over groups of lj/N (N M - B n)^2 / (B (N - B) - N lj / 4)
//   hist   bin k of np.histogram against edges linspace(lo, hi, bins + 1) of the draw's pooled range: the count of
//          values < e_k is the cumulative count at the first sorted position whose bin reaches k
// rank_kernel does one chunked block scan per (draw, feature) over the sorted positions: an int64 sum-scan of the packed
// (x << 32 | y) counts, and a max-scan that carries the cumulative count at the latest group start across chunks.
// kde_kernel sums c_i exp(-(g_k - x_i)^2 / (2 h^2)) over the sorted column for every grid point, in fp64.
// All reductions run in a fixed order, so repeated calls give identical bits.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/rnvp.h"

int rnvp_fail(int code, const char* msg);

namespace {

typedef unsigned long long u64;
typedef __int128 i128;

constexpr int R_THREADS = 256;              // rank_kernel: one CTA per (feature, draw)
constexpr int R_ITEMS = 8;                  // consecutive sorted positions per thread and chunk
constexpr int R_CHUNK = R_THREADS * R_ITEMS;
constexpr int R_WARPS = R_THREADS / 32;
constexpr int K_THREADS = 256;              // kde_kernel: G grid points x (K_THREADS / G) position slices per CTA
constexpr int K_STAGE = 1024;               // sorted positions staged in shared memory per step

// np.linspace(lo, hi, num)[k] of NumPy 2.x (endpoint=True): k * step + lo with step = (hi - lo) / (num - 1), the last
// point exactly hi; a zero step (subnormal range) multiplies k / (num - 1) by the range instead.  No FMA contraction.
__device__ double linspace_at(int64_t k, double lo, double hi, int64_t num) {
  if (num > 1 && k == num - 1) return hi;
  const double delta = __dsub_rn(hi, lo);
  if (num <= 1) return __dadd_rn(__dmul_rn((double)k, delta), lo);
  const double step = __ddiv_rn(delta, (double)(num - 1));
  if (step == 0.0) return __dadd_rn(__dmul_rn(__ddiv_rn((double)k, (double)(num - 1)), delta), lo);
  return __dadd_rn(__dmul_rn((double)k, step), lo);
}

// np.histogram's bin of v against edges e_0..e_bins: the largest k < bins with e_k <= v ([e_k, e_k+1), the last bin
// closed).  Values outside [e_0, e_bins] carry a zero count here; they are clamped to the first or last bin.
__device__ int bin_of(double v, double lo, double hi, int bins, double inv_step) {
  if (!(v >= lo)) return 0;
  if (v >= hi) return bins - 1;
  const double t = floor(__dmul_rn(__dsub_rn(v, lo), inv_step));
  int k = t >= 0.0 ? (t < (double)(bins - 1) ? (int)t : bins - 1) : 0;   // NaN (zero range) -> 0
  while (k > 0 && linspace_at(k, lo, hi, (int64_t)bins + 1) > v) --k;
  while (k + 1 < bins && linspace_at(k + 1, lo, hi, (int64_t)bins + 1) <= v) ++k;
  return k;
}

// The draw's pooled min and max: the values at the first and the last sorted positions with a nonzero count.
__device__ void draw_range(const double* v, const int* src, const uint16_t* cnt, int64_t N, double* s_lo, double* s_hi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    for (int64_t base = 0;; base += 32) {
      const int64_t p = base + lane;
      const unsigned nz = __ballot_sync(0xffffffffu, p < N && cnt[src[p]] != 0);
      if (nz) {
        if (lane == 0) *s_lo = v[base + __ffs(nz) - 1];
        break;
      }
    }
  } else if (warp == 1) {
    for (int64_t base = N - 1;; base -= 32) {
      const int64_t p = base - lane;
      const unsigned nz = __ballot_sync(0xffffffffu, p >= 0 && cnt[src[p]] != 0);
      if (nz) {
        if (lane == 0) *s_hi = v[base - (__ffs(nz) - 1)];
        break;
      }
    }
  }
  __syncthreads();
}

struct SumOp {
  __device__ u64 operator()(u64 a, u64 b) const { return a + b; }
};
struct MaxOp {
  __device__ u64 operator()(u64 a, u64 b) const { return a > b ? a : b; }
};

// Exclusive block scan of one value per thread (identity 0 for both ops); *total gets the reduction of all threads.
template <class Op>
__device__ u64 block_exclusive(u64 x, Op op, u64* s_warp, u64* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  u64 inc = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u64 y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc = op(inc, y);
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    u64 w = lane < R_WARPS ? s_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < R_WARPS; o <<= 1) {
      const u64 y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w = op(w, y);
    }
    if (lane < R_WARPS) s_warp[lane] = w;
  }
  __syncthreads();
  u64 ex = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) ex = 0;
  if (warp > 0) ex = op(s_warp[warp - 1], ex);
  *total = s_warp[R_WARPS - 1];
  __syncthreads();                       // s_warp is reused by the next scan
  return ex;
}

// Fixed-order tree reduction of one double per thread of a CTA of R_THREADS; the result is returned to every thread.
template <class F>
__device__ double block_reduce(double x, double* s_red, F op) {
  s_red[threadIdx.x] = x;
  __syncthreads();
  for (int s = R_THREADS / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) s_red[threadIdx.x] = op(s_red[threadIdx.x], s_red[threadIdx.x + s]);
    __syncthreads();
  }
  const double r = s_red[0];
  __syncthreads();
  return r;
}

__device__ double dadd(double a, double b) { return __dadd_rn(a, b); }

// A nonnegative 128-bit integer as a double: correctly rounded below 2^64, within one ulp above.
__device__ double i128_to_double(i128 v) {
  const u64 hi = (u64)(v >> 64), lo = (u64)v;
  if (hi == 0) return (double)lo;
  return __dadd_rn(__dmul_rn((double)hi, 18446744073709551616.0), (double)lo);
}

// Adds 4 sum_{j=1..g} (A/2 - j)^2 = g A^2 - 2 A g (g + 1) + 4 g (g + 1) (2 g + 1) / 6 of one tie group (A > 0) to the
// 128-bit accumulator (hi, lo), exactly.  The usual group (g < 2^16, A < 2^23) has every product below 2^62 and takes
// int64 arithmetic; any other (g, A < 2^33) is formed in 128 bits.
__device__ void add_cvm_group4(u64& lo, u64& hi, long long A, long long g) {
  u64 tlo, thi;
  if (g < (1LL << 16) && A < (1LL << 23)) {
    tlo = (u64)(g * A * A - 2 * A * g * (g + 1) + 4 * (g * (g + 1) * (2 * g + 1) / 6));
    thi = 0;
  } else {
    const i128 a = A, G = g;
    const i128 t = G * a * a - 2 * a * G * (G + 1) + 4 * (G * (G + 1) * (2 * G + 1) / 6);
    tlo = (u64)t;
    thi = (u64)(t >> 64);
  }
  lo += tlo;
  hi += thi + (lo < tlo ? 1 : 0);
}

struct RankArgs {
  const double* vals;       // [D][N] sorted pooled columns
  const int* src;           // [D][N] row of each sorted position
  const uint16_t* counts;   // [n_draws][N]
  int64_t n, m;
  int D, bins;
  double eps;
  double* stats;            // [n_draws][D][RNVP_RANK_NSTAT]
  int* slots;               // [n_draws][D][bins + 1][2] cumulative x, y counts below each histogram edge
};

__global__ void __launch_bounds__(R_THREADS) rank_kernel(RankArgs a) {
  const int d = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int64_t n = a.n, m = a.m, N = n + m;
  const double* v = a.vals + (size_t)d * N;
  const int* src = a.src + (size_t)d * N;
  const uint16_t* cnt = a.counts + (size_t)b * N;
  int* slot = a.slots + ((size_t)b * a.D + d) * (size_t)(a.bins + 1) * 2;
  const int bins = a.bins;

  __shared__ double s_lo, s_hi;
  __shared__ u64 s_warp[R_WARPS];
  __shared__ double s_red[R_THREADS];
  __shared__ i128 s_ired[R_THREADS];

  draw_range(v, src, cnt, N, &s_lo, &s_hi);
  double lo = s_lo, hi = s_hi;
  if (lo == hi) {                        // np.histogram widens an empty range to +-0.5
    lo = __dsub_rn(lo, 0.5);
    hi = __dadd_rn(hi, 0.5);
  }
  const double inv_step = (double)bins / __dsub_rn(hi, lo);   // first guess only; bin_of checks the exact edges
  const double nd = (double)n, md = (double)m;

  u64 carry_cum = 0, carry_start = 0;
  double dmax = -INFINITY, dmin = INFINITY, adx = 0.0, ady = 0.0;
  u64 cvx_lo = 0, cvx_hi = 0, cvy_lo = 0, cvy_hi = 0;   // 4 U of each sample, 128 bits: past 2^63 from n = m ~ 1.3e6
  long long u2 = 0, ndist = 0;

  for (int64_t c0 = 0; c0 < N; c0 += R_CHUNK) {
    const int64_t p0 = c0 + (int64_t)tid * R_ITEMS;
    double vv[R_ITEMS];
    u64 pk[R_ITEMS];
    bool st[R_ITEMS];
    const double prev = (p0 > 0 && p0 < N) ? v[p0 - 1] : 0.0;
#pragma unroll
    for (int i = 0; i < R_ITEMS; ++i) {
      const int64_t p = p0 + i;
      if (p < N) {
        vv[i] = v[p];
        const int s = src[p];
        const u64 c = cnt[s];
        pk[i] = s < n ? (c << 32) : c;
        st[i] = p == 0 || vv[i] != (i ? vv[i - 1] : prev);
      } else {
        vv[i] = 0.0;
        pk[i] = 0;
        st[i] = false;
      }
    }
    // cumulative counts up to and including each position
    u64 loc[R_ITEMS], run = 0;
#pragma unroll
    for (int i = 0; i < R_ITEMS; ++i) loc[i] = (run += pk[i]);
    u64 tot;
    const u64 ex = block_exclusive(run, SumOp(), s_warp, &tot) + carry_cum;
    carry_cum += tot;
    // cumulative count before the start of each position's tie group
    u64 gs[R_ITEMS], mrun = 0;
#pragma unroll
    for (int i = 0; i < R_ITEMS; ++i) {
      if (st[i]) mrun = ex + loc[i] - pk[i];
      gs[i] = mrun;
    }
    u64 mtot;
    const u64 mex = block_exclusive(mrun, MaxOp(), s_warp, &mtot);
    const u64 carry_in = mex > carry_start ? mex : carry_start;
    carry_start = mtot > carry_start ? mtot : carry_start;

    int bprev = 0;
    if (p0 > 0 && p0 < N) bprev = bin_of(prev, lo, hi, bins, inv_step);
#pragma unroll
    for (int i = 0; i < R_ITEMS; ++i) {
      const int64_t p = p0 + i;
      if (p >= N) break;
      const u64 incl = ex + loc[i];
      const u64 before = gs[i] > carry_in ? gs[i] : carry_in;
      const int bcur = bin_of(vv[i], lo, hi, bins, inv_step);
      if (st[i]) {
        const u64 excl = incl - pk[i];
        for (int k = bprev + 1; k <= bcur; ++k) {
          slot[2 * k] = (int)(excl >> 32);
          slot[2 * k + 1] = (int)(excl & 0xffffffffu);
        }
      }
      bprev = bcur;
      const bool en = p == N - 1 || vv[i] != (i + 1 < R_ITEMS ? vv[i + 1] : v[p + 1]);
      if (!en) continue;
      const long long ax = (long long)(incl >> 32), ay = (long long)(incl & 0xffffffffu);
      const long long bx = (long long)(before >> 32), by = (long long)(before & 0xffffffffu);
      const long long gx = ax - bx, gy = ay - by, t = gx + gy;
      if (t == 0) continue;                // no row of this value was drawn
      ++ndist;
      // KS: ECDFs as scipy's ks_2samp takes them, linspace(0, 1, n + 1)[count]
      const double dd = __dsub_rn(linspace_at(ax, 0.0, 1.0, n + 1), linspace_at(ay, 0.0, 1.0, m + 1));
      dmax = fmax(dmax, dd);
      dmin = fmin(dmin, dd);
      // CvM: 4 sum_{j=1..g} (r - (B + j))^2 with midrank r = P + (t + 1) / 2, A = 2r - 2B
      const long long P = bx + by;
      add_cvm_group4(cvx_lo, cvx_hi, 2 * P + t + 1 - 2 * bx, gx);
      add_cvm_group4(cvy_lo, cvy_hi, 2 * P + t + 1 - 2 * by, gy);
      // AUC (y scored above x): pairs with y above x count 2, tied pairs 1
      u2 += 2 * gy * bx + gx * gy;
      // AD midrank: lj / N * (N * M - B * n_i)^2 / (B * (N - B) - N * lj / 4), M = cumulative count - g / 2
      const double Nd = (double)N, lj = (double)t;
      const double Bj = __dadd_rn((double)P, __ddiv_rn(lj, 2.0));
      const double den = __dsub_rn(__dmul_rn(Bj, __dsub_rn(Nd, Bj)), __ddiv_rn(__dmul_rn(Nd, lj), 4.0));
      const double w = __ddiv_rn(lj, Nd);
      const double Mx = __dsub_rn((double)ax, __ddiv_rn((double)gx, 2.0));
      const double My = __dsub_rn((double)ay, __ddiv_rn((double)gy, 2.0));
      const double ex_ = __dsub_rn(__dmul_rn(Nd, Mx), __dmul_rn(Bj, nd));
      const double ey_ = __dsub_rn(__dmul_rn(Nd, My), __dmul_rn(Bj, md));
      adx = __dadd_rn(adx, __ddiv_rn(__dmul_rn(w, __dmul_rn(ex_, ex_)), den));
      ady = __dadd_rn(ady, __ddiv_rn(__dmul_rn(w, __dmul_rn(ey_, ey_)), den));
    }
  }
  // edges that no position reached: the last bins hold nothing beyond the draw's max
  if (tid == 0) {
    slot[0] = 0;
    slot[1] = 0;
    for (int k = bin_of(v[N - 1], lo, hi, bins, inv_step) + 1; k <= bins; ++k) {
      slot[2 * k] = (int)(carry_cum >> 32);
      slot[2 * k + 1] = (int)(carry_cum & 0xffffffffu);
    }
  }

  dmax = block_reduce(dmax, s_red, [](double x, double y) { return fmax(x, y); });
  dmin = block_reduce(dmin, s_red, [](double x, double y) { return fmin(x, y); });
  adx = block_reduce(adx, s_red, dadd);
  ady = block_reduce(ady, s_red, dadd);
  i128 isum[4] = {((i128)cvx_hi << 64) | cvx_lo, ((i128)cvy_hi << 64) | cvy_lo, u2, ndist};
  for (int j = 0; j < 4; ++j) {          // integer sums: exact in any order
    s_ired[tid] = isum[j];
    __syncthreads();
    for (int s = R_THREADS / 2; s > 0; s >>= 1) {
      if (tid < s) s_ired[tid] += s_ired[tid + s];
      __syncthreads();
    }
    isum[j] = s_ired[0];
    __syncthreads();
  }

  // histogram KL / JS of p = h_x / n + eps and q = h_y / m + eps
  double kl = 0.0, j1 = 0.0, j2 = 0.0;
  for (int k = tid; k < bins; k += R_THREADS) {
    const double p = __dadd_rn(__ddiv_rn((double)(slot[2 * k + 2] - slot[2 * k]), nd), a.eps);
    const double q = __dadd_rn(__ddiv_rn((double)(slot[2 * k + 3] - slot[2 * k + 1]), md), a.eps);
    const double mm = __dmul_rn(0.5, __dadd_rn(p, q));
    kl = __dadd_rn(kl, __dmul_rn(p, log(__ddiv_rn(p, q))));
    j1 = __dadd_rn(j1, __dmul_rn(p, log(__ddiv_rn(p, mm))));
    j2 = __dadd_rn(j2, __dmul_rn(q, log(__ddiv_rn(q, mm))));
  }
  kl = block_reduce(kl, s_red, dadd);
  j1 = block_reduce(j1, s_red, dadd);
  j2 = block_reduce(j2, s_red, dadd);

  if (tid == 0) {
    double* out = a.stats + ((size_t)b * a.D + d) * RNVP_RANK_NSTAT;
    const double min_s = fmin(fmax(-dmin, 0.0), 1.0);
    out[0] = dmax > min_s ? dmax : min_s;
    if (n < 2 || m < 2) {
      out[1] = NAN;                      // cramervonmises_2samp needs two observations per sample
    } else {
      const double u = __dadd_rn(__dmul_rn(nd, i128_to_double(isum[0]) * 0.25),
                                 __dmul_rn(md, i128_to_double(isum[1]) * 0.25));
      const long long k = n * m;         // < 2^60 for n + m < 2^31; k N can exceed 2^63
      out[1] = __dsub_rn(__ddiv_rn(u, i128_to_double((i128)k * N)), __ddiv_rn((double)(4 * k - 1), (double)(6 * N)));
    }
    const double auc = __ddiv_rn(i128_to_double(isum[2]), (double)(2 * n * m));
    out[2] = __dadd_rn(fabs(__dsub_rn(auc, 0.5)), 0.5);
    out[3] = __dmul_rn(__dadd_rn(__ddiv_rn(adx, nd), __ddiv_rn(ady, md)),
                       __ddiv_rn((double)N - 1.0, (double)N));
    out[4] = kl;
    out[5] = __dadd_rn(__dmul_rn(0.5, j1), __dmul_rn(0.5, j2));
    out[6] = i128_to_double(isum[3]);
  }
}

struct KdeArgs {
  const double* vals;
  const int* src;
  const uint16_t* counts;
  int64_t n, m;
  int D, bins;
  double cx, cy;            // 1 / (2 h^2) of the x and the y sample
  double* sums;             // [n_draws][D][2][bins]
  int G;                    // grid points per CTA: bins split evenly over ceil(bins / K_THREADS) CTAs
};

// Grid points per kde_kernel CTA.  A CTA's threads are (grid point, slice) pairs packed densely, so bins = 101 keeps 202
// of 256 threads busy (two slices) instead of rounding the grid up to whole warps of points.  Launches with fewer than
// K_MIN_CTAS CTAs split the grid further (down to 32 points per CTA, more slices each) so the device fills.  The split
// depends on the sizes only, so a given call sums in the same order on every device.
constexpr int K_MIN_CTAS = 1024;
int kde_grid_per_cta(int bins, int64_t features_x_draws) {
  int tiles = (bins + K_THREADS - 1) / K_THREADS;
  int G = (bins + tiles - 1) / tiles;
  while (G > 32 && features_x_draws * tiles < K_MIN_CTAS) {
    tiles *= 2;
    G = (bins + tiles - 1) / tiles;
  }
  return G;
}

__global__ void __launch_bounds__(K_THREADS) kde_kernel(KdeArgs a) {
  const int d = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
  const int64_t n = a.n, N = a.n + a.m;
  const double* v = a.vals + (size_t)d * N;
  const int* src = a.src + (size_t)d * N;
  const uint16_t* cnt = a.counts + (size_t)b * N;

  __shared__ double s_lo, s_hi;
  __shared__ double s_v[K_STAGE];
  __shared__ int s_w[K_STAGE];             // count of the position, negative for a y row
  __shared__ double s_part[K_THREADS][2];

  draw_range(v, src, cnt, N, &s_lo, &s_hi);
  const int G = a.G, slices = K_THREADS / G;
  const int gk = blockIdx.x * G + tid % G, slice = tid / G;
  const bool active = slice < slices && gk < a.bins;
  const double g = active ? linspace_at(gk, s_lo, s_hi, a.bins) : s_lo;

  double sx = 0.0, sy = 0.0;
  for (int64_t c0 = 0; c0 < N; c0 += K_STAGE) {
    __syncthreads();
    for (int j = tid; j < K_STAGE; j += K_THREADS) {
      const int64_t p = c0 + j;
      int w = 0;
      if (p < N) {
        const int s = src[p];
        w = s < n ? (int)cnt[s] : -(int)cnt[s];
        s_v[j] = v[p];
      }
      s_w[j] = w;
    }
    __syncthreads();
    const int lim = active ? (int)(N - c0 < K_STAGE ? N - c0 : K_STAGE) : 0;
    for (int j = slice; j < lim; j += slices) {
      const int w = s_w[j];                // one or two values of j across a warp
      if (w == 0) continue;
      const double t = __dsub_rn(g, s_v[j]);
      const double e = exp(-__dmul_rn(__dmul_rn(t, t), w > 0 ? a.cx : a.cy));
      if (w > 0) sx = __dadd_rn(sx, __dmul_rn((double)w, e));
      else sy = __dadd_rn(sy, __dmul_rn((double)-w, e));
    }
  }
  s_part[tid][0] = sx;
  s_part[tid][1] = sy;
  __syncthreads();
  if (slice == 0 && active) {
    double tx = 0.0, ty = 0.0;
    for (int s = 0; s < slices; ++s) {      // slice order: fixed
      tx = __dadd_rn(tx, s_part[s * G + tid][0]);
      ty = __dadd_rn(ty, s_part[s * G + tid][1]);
    }
    double* out = a.sums + ((size_t)b * a.D + d) * 2 * a.bins;
    out[gk] = tx;
    out[a.bins + gk] = ty;
  }
}

int launch_fail(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return 0;
  return rnvp_fail((int)e, what);
}

int check_sizes(int64_t n, int64_t m, int D, int n_draws, int bins, const char* what) {
  if (n < 1 || m < 1 || D < 1 || n_draws < 1 || bins < 1) return rnvp_fail(RNVP_EINVAL, what);
  if (n + m > 0x7fffffff || D > 65535 || n_draws > 65535) return rnvp_fail(RNVP_EINVAL, what);
  return 0;
}

}  // namespace

extern "C" {

int64_t rnvp_rank_workspace_bytes(int D, int n_draws, int bins) {
  if (D < 1 || n_draws < 1 || bins < 1) return rnvp_fail(RNVP_EINVAL, "rnvp_rank_workspace_bytes: bad sizes");
  return (int64_t)n_draws * D * ((int64_t)bins + 1) * 2 * (int64_t)sizeof(int);
}

int rnvp_rank_draws(const double* d_sorted, const int32_t* d_src, int64_t n, int64_t m, int D, const uint16_t* d_counts,
                    int n_draws, int bins, double eps, double* d_stats, void* d_workspace, int64_t workspace_bytes,
                    void* stream) {
  if (int rc = check_sizes(n, m, D, n_draws, bins, "rnvp_rank_draws: bad sizes")) return rc;
  if (!d_sorted || !d_src || !d_counts || !d_stats || !d_workspace)
    return rnvp_fail(RNVP_EINVAL, "rnvp_rank_draws: null buffer");
  if (workspace_bytes < rnvp_rank_workspace_bytes(D, n_draws, bins))
    return rnvp_fail(RNVP_EINVAL, "rnvp_rank_draws: workspace too small (see rnvp_rank_workspace_bytes)");
  RankArgs a{d_sorted, d_src, d_counts, n, m, D, bins, eps, d_stats, (int*)d_workspace};
  rank_kernel<<<dim3((unsigned)D, (unsigned)n_draws), R_THREADS, 0, (cudaStream_t)stream>>>(a);
  return launch_fail("rank_kernel");
}

int rnvp_kde_draws(const double* d_sorted, const int32_t* d_src, int64_t n, int64_t m, int D, const uint16_t* d_counts,
                   int n_draws, int bins, double h_x, double h_y, double* d_sums, void* stream) {
  if (int rc = check_sizes(n, m, D, n_draws, bins, "rnvp_kde_draws: bad sizes")) return rc;
  if (!d_sorted || !d_src || !d_counts || !d_sums) return rnvp_fail(RNVP_EINVAL, "rnvp_kde_draws: null buffer");
  if (!(h_x > 0.0) || !(h_y > 0.0)) return rnvp_fail(RNVP_EINVAL, "rnvp_kde_draws: bandwidths must be positive");
  const int G = kde_grid_per_cta(bins, (int64_t)D * n_draws);
  KdeArgs a{d_sorted, d_src, d_counts, n, m, D, bins, 0.5 / (h_x * h_x), 0.5 / (h_y * h_y), d_sums, G};
  kde_kernel<<<dim3((unsigned)((bins + G - 1) / G), (unsigned)D, (unsigned)n_draws), K_THREADS, 0,
               (cudaStream_t)stream>>>(a);
  return launch_fail("kde_kernel");
}

}  // extern "C"
