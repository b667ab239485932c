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
