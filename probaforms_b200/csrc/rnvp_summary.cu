// Per-cell summaries of k draws (probaforms_b200/predictive.py): mean, std, numpy 'linear' quantiles, ensemble CRPS and
// the PIT rank of an observation.
//
// The draws of one request are laid out d_draws[j * cells + c] (draw j, cell c = row * D + feature).  A CTA owns G
// adjacent cells and has one warp per cell.  It reads every draw's G cells as one coalesced G * 4-byte access, writes
// them transposed into shared memory as G columns of k order-preserving uint32 keys (padded to k_pad = next power of two
// with the largest key), and after one __syncthreads each warp works on its own column alone: a bitonic sort in shared
// memory (__syncwarp between stages), then two passes over the sorted column (the fp64 sum; then sum (x - mean)^2,
// the CRPS spread sum on centred values, sum |x - y| and #{x < y}) and one lane per quantile.  Every sum has a fixed
// order (lane-strided partial sums, then a shuffle tree), and a cell's arithmetic does not depend on its position in
// the group, so results do not depend on how a request is split into launches.
//
// Quantiles follow numpy 2.3's np.quantile(draws, q, axis=0) for float32 draws bit for bit: virtual index (k - 1) q in
// fp64; prev = floor, next = prev + 1, or both the last element with gamma = index + 1 when index >= k - 1; the
// neighbours' difference b - a is taken in float32 (numpy subtracts in the input's dtype), the rest in fp64 without FMA
// contraction: a + diff g, or b - diff (1 - g) when g >= 0.5.  A cell with a NaN draw gives NaN for every quantile.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/rnvp.h"

int rnvp_fail(int code, const char* msg);

namespace {

constexpr int S_MAX_G = 8;                  // cells per CTA: 8 x 4 bytes fill a 32-byte sector per draw
constexpr int S_PAD = 4;                    // column stride k_pad + 4: the transposed stores of a warp hit 32 banks
constexpr int S_SMEM_MAX = 232448;          // opt-in dynamic shared memory per CTA on sm_100 (227 KB)
constexpr unsigned FULL = 0xffffffffu;

struct SummaryArgs {
  const float* draws;
  const float* y;
  double* mean;
  double* std;
  double* quant;
  double* crps;
  int32_t* rank;
  int64_t k, cells, q_stride;
  int k_pad, stride, G, nq;
  double q[RNVP_SUMMARY_MAX_QUANTILES];
};

// float -> uint32 whose unsigned order is the float order (-NaN < -inf < ... < -0 < +0 < ... < +inf < +NaN)
__device__ __forceinline__ uint32_t f2key(float f) {
  const uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t key) {
  return __uint_as_float(key ^ ((key >> 31) ? 0x80000000u : 0xffffffffu));
}

// fixed-order warp sum (tree on lane 0, then broadcast): every lane gets the same bits
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_down_sync(FULL, v, o));
  return __shfl_sync(FULL, v, 0);
}

__global__ void __launch_bounds__(32 * S_MAX_G) draw_summary_kernel(const SummaryArgs a) {
  extern __shared__ uint32_t s_keys[];
  const int G = a.G, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t k = a.k, cells = a.cells;
  const int64_t c0 = (int64_t)blockIdx.x * G;

  // coalesced read of G adjacent cells per draw, transposed into G columns of keys; blockDim = 32 G, so one pass of the
  // CTA covers 32 draws
  {
    const int g = tid % G;
    const int64_t c = c0 + g;
    uint32_t* col = s_keys + g * a.stride;
    if (c < cells) {
      const float* src = a.draws + c;
      int64_t j = tid / G;
      for (; j + 96 < k; j += 128) {
        const float v0 = __ldcs(src + j * cells), v1 = __ldcs(src + (j + 32) * cells);
        const float v2 = __ldcs(src + (j + 64) * cells), v3 = __ldcs(src + (j + 96) * cells);
        col[j] = f2key(v0);
        col[j + 32] = f2key(v1);
        col[j + 64] = f2key(v2);
        col[j + 96] = f2key(v3);
      }
      for (; j < k; j += 32) col[j] = f2key(__ldcs(src + j * cells));
    }
  }
  __syncthreads();

  const int64_t c = c0 + warp;
  if (c >= cells) return;
  uint32_t* col = s_keys + warp * a.stride;
  const uint32_t P = (uint32_t)a.k_pad;
  for (uint32_t i = (uint32_t)k + lane; i < P; i += 32) col[i] = 0xffffffffu;    // padding sorts last
  __syncwarp();

  // bitonic sort of the column, ascending
  for (uint32_t size = 2; size <= P; size <<= 1) {
    for (uint32_t j = size >> 1; j > 0; j >>= 1) {
      for (uint32_t p = lane; p < P / 2; p += 32) {
        const uint32_t i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
        const uint32_t x = col[i], y = col[i + j];
        const uint32_t lo = min(x, y), hi = max(x, y);
        const bool up = (i & size) == 0;
        col[i] = up ? lo : hi;
        col[i + j] = up ? hi : lo;
      }
      __syncwarp();
    }
  }

  // pass 1: sum and NaN flag
  double sum = 0.0;
  bool nan = false;
  for (int64_t i = lane; i < k; i += 32) {
    const float x = key2f(col[i]);
    nan |= isnan(x);
    sum = __dadd_rn(sum, (double)x);
  }
  nan = __any_sync(FULL, nan);
  const double mean = __ddiv_rn(warp_sum(sum), (double)k);

  // pass 2: sum (x - mean)^2, sum (2 i + 1 - k) (x_(i) - mean) over the sorted column (i from 0), sum |x - y|, #{x < y}
  const bool has_y = a.y != nullptr;
  const float yf = has_y ? a.y[c] : 0.0f;
  const double yd = (double)yf;
  double ss = 0.0, spread = 0.0, absdev = 0.0;
  int below = 0;
  for (int64_t i = lane; i < k; i += 32) {
    const float xf = key2f(col[i]);
    const double dx = __dsub_rn((double)xf, mean);
    ss = __fma_rn(dx, dx, ss);
    spread = __fma_rn((double)(2 * i + 1 - k), dx, spread);
    if (has_y) {
      absdev = __dadd_rn(absdev, fabs(__dsub_rn((double)xf, yd)));
      below += xf < yf;
    }
  }
  ss = warp_sum(ss);
  spread = warp_sum(spread);
  absdev = warp_sum(absdev);
  below = __reduce_add_sync(FULL, below);
  const double kd = (double)k;

  if (lane == 0) {
    if (a.mean) a.mean[c] = mean;
    if (a.std) a.std[c] = sqrt(__ddiv_rn(ss, kd));
    // CRPS = (1/k) sum |x_j - y| - (1/(2 k^2)) sum_i sum_j |x_i - x_j|, the double sum = 2 sum_i (2 i - k - 1) x_(i)
    // (i from 1), taken on centred values: the weights sum to zero
    if (a.crps) a.crps[c] = has_y && !isnan(yf) ? __dsub_rn(__ddiv_rn(absdev, kd), __ddiv_rn(spread, __dmul_rn(kd, kd)))
                                                : (double)NAN;
    if (a.rank) a.rank[c] = below;
  }
  if (a.quant && lane < a.nq) {
    double r = (double)NAN;
    if (!nan) {
      const double last = (double)(k - 1);
      const double vi = __dmul_rn(last, a.q[lane]);
      int64_t prev, next;
      double base;                            // numpy's previous index as used in gamma (-1 past the last element)
      if (vi >= last) {
        prev = next = k - 1;
        base = -1.0;
      } else {
        base = floor(vi);
        prev = (int64_t)base;
        next = prev + 1;
      }
      const double g = __dsub_rn(vi, base);
      const float lo = key2f(col[prev]), hi = key2f(col[next]);
      const double diff = (double)__fsub_rn(hi, lo);
      r = g >= 0.5 ? __dsub_rn((double)hi, __dmul_rn(diff, __dsub_rn(1.0, g)))
                   : __dadd_rn((double)lo, __dmul_rn(diff, g));
    }
    a.quant[(int64_t)lane * a.q_stride + c] = r;
  }
}

}  // namespace

extern "C" int rnvp_draw_summary(const float* d_draws, int64_t k, int64_t cells, const double* q, int nq,
                                 const float* d_y, double* d_mean, double* d_std, double* d_quant, int64_t q_stride,
                                 double* d_crps, int32_t* d_rank, void* stream) {
  if (k < 1 || k > RNVP_SUMMARY_MAX_DRAWS) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: k must be in [1, 8192]");
  if (cells < 0) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: cells must be >= 0");
  if (nq < 0 || nq > RNVP_SUMMARY_MAX_QUANTILES || (nq > 0 && !q))
    return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: nq must be in [0, 32] with a host array q");
  for (int i = 0; i < nq; ++i)
    if (!(q[i] >= 0.0 && q[i] <= 1.0)) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: quantiles must be in [0, 1]");
  if (d_quant && nq > 0 && q_stride < cells) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: q_stride < cells");
  if ((d_crps || d_rank) && !d_y) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: d_crps / d_rank need d_y");
  if (cells == 0) return 0;
  if (!d_draws) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: null d_draws");

  SummaryArgs a{};
  a.draws = d_draws;
  a.y = d_y;
  a.mean = d_mean;
  a.std = d_std;
  a.quant = nq > 0 ? d_quant : nullptr;
  a.crps = d_crps;
  a.rank = d_rank;
  a.k = k;
  a.cells = cells;
  a.q_stride = q_stride;
  a.nq = nq;
  for (int i = 0; i < nq; ++i) a.q[i] = q[i];
  int k_pad = 1;
  while (k_pad < k) k_pad <<= 1;
  a.k_pad = k_pad;
  a.stride = k_pad + S_PAD;
  const int64_t col_bytes = (int64_t)a.stride * 4;
  a.G = (int)(S_SMEM_MAX / col_bytes < S_MAX_G ? S_SMEM_MAX / col_bytes : S_MAX_G);   // 7 at k_pad = 8192
  const int smem = (int)(a.G * col_bytes);
  cudaError_t e = cudaFuncSetAttribute(draw_summary_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_draw_summary: cudaFuncSetAttribute");
  const int64_t blocks = (cells + a.G - 1) / a.G;
  if (blocks > 0x7fffffff) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_summary: too many cells");
  draw_summary_kernel<<<(unsigned)blocks, 32 * a.G, smem, (cudaStream_t)stream>>>(a);
  e = cudaGetLastError();
  if (e != cudaSuccess) return rnvp_fail((int)e, "draw_summary_kernel");
  return 0;
}

// Joint scores of k draws per row (probaforms_b200/predictive.py predictive_joint): the row mean, the covariance, the
// energy score and the variogram score of an observation y.  The draws arrive as a row block laid out
// d_draws[(j * rows + r) * D + d] (draw j, row r, feature d).  Three kernels:
//
//   joint_moments_kernel   one CTA per row.  Pass 1: the fp64 mean per feature; thread (s, d) sums draws s, s + S, ...
//                          (S = 256 / D slices) and thread d adds the S partials in slice order.  Pass 2 (cov): the
//                          draws in chunks of J_CHUNK, centred in fp64 and rounded to fp32 in shared memory; each thread
//                          owns pairs d <= e and adds the fp32 chain of a chunk's J_CHUNK products into an fp64 sum.
//   joint_pairs_kernel     grid (tile pair, row).  A row's draws are cut into tiles of J_TILE; CTA (ta <= tb) stages
//                          both tiles centred and transposed in 32-feature chunks and each thread takes an 8 x 8 register
//                          tile of pairs: fp32 squared distance, IEEE sqrt, an fp32 chain of its 64 distances into fp64,
//                          then a fixed-order CTA sum.  One partial per CTA (doubled off the diagonal) goes to the
//                          workspace [rows, tile pairs]; padding draws are masked.
//   joint_finish_kernel    one CTA per row: the partials summed in tile-pair order, sum_j ||x_j - y|| in fp64 (one warp
//                          per draw), and the variogram's pair sums (the same chunked pass as the covariance on the raw
//                          draws), then energy and variogram.
//
// Every sum has a fixed order and a row's arithmetic does not depend on its position in the block, so repeated calls
// and any split into row blocks give the same bits.  Nothing of size k^2 is stored.  A row with a non-finite draw (a
// non-finite fp64 mean: k finite floats cannot overflow it) gives NaN cov, energy and variogram; a NaN in y gives NaN
// energy and variogram.
namespace {

constexpr int J_THREADS = 256;
constexpr int J_CHUNK = 32;                 // draws per staged chunk of the row passes: the length of an fp32 chain
constexpr int J_TILE = 128;                 // draws per tile of the energy pair pass
constexpr int J_FEAT = 32;                  // features per staged chunk of the pair pass
constexpr int J_REG = J_TILE / 16;          // 16 x 16 threads, each an J_REG x J_REG register tile of pairs

struct JointArgs {
  const float* draws;
  const float* y;
  double* mean;
  double* cov;
  double* energy;
  double* variogram;
  double* ws;
  int64_t k, rows;
  int D, P, pmode;                          // P tile pairs; pmode 0: p = 0.5, 1: p = 1, 2: p = 2, 3: any other p
  float pf;
  double p;
};

// p < N (N + 1) / 2 -> (lo, hi) with lo <= hi < N, hi-major: (0,0) (0,1) (1,1) (0,2) (1,2) (2,2) ...
__device__ __forceinline__ void tri_index(int p, int& lo, int& hi) {
  int i = (int)((sqrtf(8.0f * (float)p + 1.0f) - 1.0f) * 0.5f);
  while (i * (i + 1) / 2 > p) --i;
  while ((i + 1) * (i + 2) / 2 <= p) ++i;
  hi = i;
  lo = p - i * (i + 1) / 2;
}

__device__ __forceinline__ const float* row_draw(const JointArgs& a, int64_t j, int64_t r) {
  return a.draws + (j * a.rows + r) * a.D;
}

// |v|^p in fp32 for the draws: sqrtf / fabsf / square for p = 0.5, 1, 2, else the accurate powf
__device__ __forceinline__ float vpow(float v, int mode, float p) {
  const float u = fabsf(v);
  return mode == 0 ? __fsqrt_rn(u) : mode == 1 ? u : mode == 2 ? __fmul_rn(u, u) : powf(u, p);
}
__device__ __forceinline__ double vpow(double v, int mode, double p) {
  const double u = fabs(v);
  return mode == 0 ? sqrt(u) : mode == 1 ? u : mode == 2 ? __dmul_rn(u, u) : pow(u, p);
}

// fixed-order CTA sum of one double per thread; the result is valid on thread 0
__device__ __forceinline__ double cta_sum(double v, double* s_red) {
  v = warp_sum(v);
  const int t = threadIdx.x;
  __syncthreads();
  if ((t & 31) == 0) s_red[t >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (t == 0)
    for (int w = 0; w < J_THREADS / 32; ++w) s = __dadd_rn(s, s_red[w]);
  return s;
}

// The chunked pass over one row's draws shared by the covariance and the variogram: pair q < np is (lo, hi + off) with
// (lo, hi) = tri_index(q); s_acc[q] += the fp32 chain term(x_lo, x_hi, f) over a chunk's draws.  With centre the staged
// values are (float)(x - centre[d]) computed in fp64.
template <class Term>
__device__ void row_pair_pass(const JointArgs& a, int64_t r, const double* centre, int np, int off, double* s_acc,
                              float* s_c, Term term) {
  const int D = a.D, t = threadIdx.x;
  for (int q = t; q < np; q += J_THREADS) s_acc[q] = 0.0;
  for (int64_t j0 = 0; j0 < a.k; j0 += J_CHUNK) {
    const int nj = (int)min((int64_t)J_CHUNK, a.k - j0);
    __syncthreads();
    for (int i = t; i < nj * D; i += J_THREADS) {
      const int jj = i / D, d = i - jj * D;
      const float x = row_draw(a, j0 + jj, r)[d];
      s_c[i] = centre ? (float)__dsub_rn((double)x, centre[d]) : x;
    }
    __syncthreads();
    for (int q = t; q < np; q += J_THREADS) {
      int lo, hi;
      tri_index(q, lo, hi);
      hi += off;
      float f = 0.0f;
      for (int jj = 0; jj < nj; ++jj) f = term(s_c[jj * D + lo], s_c[jj * D + hi], f);
      s_acc[q] = __dadd_rn(s_acc[q], (double)f);
    }
  }
  __syncthreads();
}

// dynamic shared memory: s_acc [np] doubles, s_mean [D] doubles, s_part [J_THREADS] doubles, s_c [J_CHUNK * D] floats
__global__ void __launch_bounds__(J_THREADS) joint_moments_kernel(const JointArgs a) {
  extern __shared__ double s_dyn[];
  const int D = a.D, t = threadIdx.x;
  const int np = a.cov ? D * (D + 1) / 2 : 0;
  double* s_acc = s_dyn;
  double* s_mean = s_acc + np;
  double* s_part = s_mean + D;
  float* s_c = (float*)(s_part + J_THREADS);
  const int64_t r = blockIdx.x;

  const int S = J_THREADS / D;
  double sum = 0.0;
  bool bad = false;
  if (t < S * D) {
    const int s = t / D, d = t - s * D;
    for (int64_t j = s; j < a.k; j += S) {
      const float x = row_draw(a, j, r)[d];
      bad |= !isfinite(x);
      sum = __dadd_rn(sum, (double)x);
    }
  }
  s_part[t] = sum;
  bad = __syncthreads_or(bad);
  if (t < D) {
    double tot = 0.0;
    for (int s = 0; s < S; ++s) tot = __dadd_rn(tot, s_part[s * D + t]);
    const double m = __ddiv_rn(tot, (double)a.k);
    s_mean[t] = m;
    a.mean[r * D + t] = m;
  }
  if (!a.cov) return;
  double* cov = a.cov + r * D * D;
  if (bad) {
    for (int i = t; i < D * D; i += J_THREADS) cov[i] = (double)NAN;
    return;
  }
  __syncthreads();
  row_pair_pass(a, r, s_mean, np, 0, s_acc, s_c, [](float u, float v, float f) { return fmaf(u, v, f); });
  for (int q = t; q < np; q += J_THREADS) {
    int lo, hi;
    tri_index(q, lo, hi);
    const double c = __ddiv_rn(s_acc[q], (double)a.k);
    cov[lo * D + hi] = c;
    cov[hi * D + lo] = c;
  }
}

__global__ void __launch_bounds__(J_THREADS) joint_pairs_kernel(const JointArgs a, int64_t row0) {
  __shared__ float sA[J_FEAT][J_TILE + 1], sB[J_FEAT][J_TILE + 1];
  __shared__ double s_mean[RNVP_JOINT_MAX_D];
  __shared__ double s_red[J_THREADS / 32];
  const int D = a.D, t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t r = row0 + blockIdx.y;
  int ta, tb;
  tri_index((int)blockIdx.x, ta, tb);
  bool bad = false;
  for (int d = t; d < D; d += J_THREADS) {
    s_mean[d] = a.mean[r * D + d];
    bad |= !isfinite(s_mean[d]);
  }
  if (__syncthreads_or(bad)) {
    if (t == 0) a.ws[r * a.P + blockIdx.x] = 0.0;
    return;
  }
  const int64_t iA = (int64_t)ta * J_TILE, iB = (int64_t)tb * J_TILE;

  float acc[J_REG][J_REG];
#pragma unroll
  for (int u = 0; u < J_REG; ++u)
#pragma unroll
    for (int v = 0; v < J_REG; ++v) acc[u][v] = 0.0f;

  for (int c0 = 0; c0 < D; c0 += J_FEAT) {
    const int nf = min(J_FEAT, D - c0), nf4 = (nf + 3) & ~3;   // zero features beyond nf add nothing
    __syncthreads();
    for (int i = t; i < J_FEAT * J_TILE; i += J_THREADS) {
      const int f = i & (J_FEAT - 1), jj = i / J_FEAT;
      float va = 0.0f, vb = 0.0f;
      if (f < nf) {
        const double m = s_mean[c0 + f];
        if (iA + jj < a.k) va = (float)__dsub_rn((double)row_draw(a, iA + jj, r)[c0 + f], m);
        if (iB + jj < a.k) vb = (float)__dsub_rn((double)row_draw(a, iB + jj, r)[c0 + f], m);
      }
      sA[f][jj] = va;
      sB[f][jj] = vb;
    }
    __syncthreads();
#pragma unroll 4
    for (int f = 0; f < nf4; ++f) {
      float xa[J_REG], xb[J_REG];
#pragma unroll
      for (int u = 0; u < J_REG; ++u) {
        xa[u] = sA[f][tx + 16 * u];
        xb[u] = sB[f][ty + 16 * u];
      }
#pragma unroll
      for (int u = 0; u < J_REG; ++u)
#pragma unroll
        for (int v = 0; v < J_REG; ++v) {
          const float df = __fsub_rn(xa[u], xb[v]);
          acc[u][v] = __fmaf_rn(df, df, acc[u][v]);
        }
    }
  }

  float s = 0.0f;
#pragma unroll
  for (int u = 0; u < J_REG; ++u)
#pragma unroll
    for (int v = 0; v < J_REG; ++v)
      if (iA + tx + 16 * u < a.k && iB + ty + 16 * v < a.k) s = __fadd_rn(s, __fsqrt_rn(acc[u][v]));
  const double tot = cta_sum((double)s, s_red);
  if (t == 0) a.ws[r * a.P + blockIdx.x] = ta == tb ? tot : __dmul_rn(2.0, tot);
}

// dynamic shared memory: s_acc [D (D - 1) / 2] doubles, s_c [J_CHUNK * D] floats
__global__ void __launch_bounds__(J_THREADS) joint_finish_kernel(const JointArgs a) {
  extern __shared__ double s_dyn[];
  __shared__ double s_red[J_THREADS / 32];
  const int D = a.D, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int np = a.variogram ? D * (D - 1) / 2 : 0;
  double* s_acc = s_dyn;
  float* s_c = (float*)(s_acc + np);
  const int64_t r = blockIdx.x;
  const float* y = a.y + r * D;

  bool bad = false;
  for (int d = t; d < D; d += J_THREADS) bad |= !isfinite(a.mean[r * D + d]) || isnan(y[d]);
  if (__syncthreads_or(bad)) {
    if (t == 0) {
      if (a.energy) a.energy[r] = (double)NAN;
      if (a.variogram) a.variogram[r] = (double)NAN;
    }
    return;
  }
  const double kd = (double)a.k;

  if (a.energy) {
    // sum_j ||x_j - y||: one warp per draw, warps take draws w, w + 8, ...; then the warps' sums in warp order
    double first = 0.0;
    for (int64_t j = warp; j < a.k; j += J_THREADS / 32) {
      const float* x = row_draw(a, j, r);
      double ss = 0.0;
      for (int d = lane; d < D; d += 32) {
        const double dv = __dsub_rn((double)x[d], (double)y[d]);
        ss = __fma_rn(dv, dv, ss);
      }
      first = __dadd_rn(first, sqrt(warp_sum(ss)));
    }
    // the pair partials in tile-pair order (warp 0 only contributes)
    double pairs = 0.0;
    if (warp == 0)
      for (int i = lane; i < a.P; i += 32) pairs = __dadd_rn(pairs, a.ws[r * a.P + i]);
    pairs = warp_sum(pairs);
    first = cta_sum(lane == 0 ? first : 0.0, s_red);
    if (t == 0) a.energy[r] = __dsub_rn(__ddiv_rn(first, kd), __ddiv_rn(pairs, __dmul_rn(2.0 * kd, kd)));
  }

  if (a.variogram) {
    const int mode = a.pmode;
    const float pf = a.pf;
    row_pair_pass(a, r, nullptr, np, 1, s_acc, s_c,
                  [mode, pf](float u, float v, float f) { return __fadd_rn(f, vpow(__fsub_rn(u, v), mode, pf)); });
    double vs = 0.0;
    for (int q = t; q < np; q += J_THREADS) {
      int lo, hi;
      tri_index(q, lo, hi);
      ++hi;
      const double yv = vpow(__dsub_rn((double)y[lo], (double)y[hi]), mode, a.p);
      const double dv = __dsub_rn(yv, __ddiv_rn(s_acc[q], kd));
      vs = __fma_rn(dv, dv, vs);
    }
    vs = cta_sum(vs, s_red);
    if (t == 0) a.variogram[r] = vs;
  }
}

int64_t joint_tile_pairs(int64_t k) {
  const int64_t nt = (k + J_TILE - 1) / J_TILE;
  return nt * (nt + 1) / 2;
}

}  // namespace

extern "C" int64_t rnvp_draw_joint_workspace_bytes(int64_t k, int64_t rows, int D) {
  if (k < 1 || k > RNVP_SUMMARY_MAX_DRAWS || rows < 0 || D < 1 || D > RNVP_JOINT_MAX_D) return -1;
  return rows * joint_tile_pairs(k) * (int64_t)sizeof(double);
}

extern "C" int rnvp_draw_joint(const float* d_draws, int64_t k, int64_t rows, int D, const float* d_y, double p,
                               double* d_mean, double* d_cov, double* d_energy, double* d_variogram, void* d_workspace,
                               int64_t workspace_bytes, void* stream) {
  if (k < 1 || k > RNVP_SUMMARY_MAX_DRAWS) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: k must be in [1, 8192]");
  if (rows < 0) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: rows must be >= 0");
  if (D < 1 || D > RNVP_JOINT_MAX_D) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: D must be in [1, 128]");
  if (!(p > 0.0) || !isfinite(p)) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: p must be finite and > 0");
  if ((d_energy || d_variogram) && !d_y)
    return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: d_energy / d_variogram need d_y");
  if (rows == 0) return 0;
  if (!d_draws || !d_mean) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: null d_draws or d_mean");
  if (d_energy && (!d_workspace || workspace_bytes < rnvp_draw_joint_workspace_bytes(k, rows, D)))
    return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: workspace smaller than rnvp_draw_joint_workspace_bytes");
  if (rows > 0x7fffffff) return rnvp_fail(RNVP_EINVAL, "rnvp_draw_joint: too many rows");

  JointArgs a{};
  a.draws = d_draws;
  a.y = d_y;
  a.mean = d_mean;
  a.cov = d_cov;
  a.energy = d_energy;
  a.variogram = d_variogram;
  a.ws = (double*)d_workspace;
  a.k = k;
  a.rows = rows;
  a.D = D;
  a.P = (int)joint_tile_pairs(k);
  a.p = p;
  a.pf = (float)p;
  a.pmode = p == 0.5 ? 0 : p == 1.0 ? 1 : p == 2.0 ? 2 : 3;
  cudaStream_t st = (cudaStream_t)stream;

  const int chunk_bytes = J_CHUNK * D * (int)sizeof(float);
  const int smem_mom = (d_cov ? D * (D + 1) / 2 : 0) * 8 + (D + J_THREADS) * 8 + chunk_bytes;
  cudaError_t e = cudaFuncSetAttribute(joint_moments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_mom);
  if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_draw_joint: cudaFuncSetAttribute");
  joint_moments_kernel<<<(unsigned)rows, J_THREADS, smem_mom, st>>>(a);
  e = cudaGetLastError();
  if (e != cudaSuccess) return rnvp_fail((int)e, "joint_moments_kernel");

  if (d_energy) {
    for (int64_t r0 = 0; r0 < rows; r0 += 65535) {             // gridDim.y <= 65535
      const unsigned m = (unsigned)(rows - r0 < 65535 ? rows - r0 : 65535);
      joint_pairs_kernel<<<dim3((unsigned)a.P, m), J_THREADS, 0, st>>>(a, r0);
      e = cudaGetLastError();
      if (e != cudaSuccess) return rnvp_fail((int)e, "joint_pairs_kernel");
    }
  }
  if (d_energy || d_variogram) {
    const int smem_fin = (d_variogram ? D * (D - 1) / 2 : 0) * 8 + chunk_bytes;
    e = cudaFuncSetAttribute(joint_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_fin);
    if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_draw_joint: cudaFuncSetAttribute");
    joint_finish_kernel<<<(unsigned)rows, J_THREADS, smem_fin, st>>>(a);
    e = cudaGetLastError();
    if (e != cudaSuccess) return rnvp_fail((int)e, "joint_finish_kernel");
  }
  return 0;
}
