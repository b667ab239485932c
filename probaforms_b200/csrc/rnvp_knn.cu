// k-nearest-neighbour precision, recall, density and coverage (probaforms_b200/metrics/knn.py
// precision_recall_density_coverage).  Real rows R [n, D], fake rows F [m, D], fp64, k <= RNVP_KNN_MAX_K.
//
// Every squared distance is d2(a, b) = (((0 + t_0 t_0) + t_1 t_1) + ...) with t_c = a_c - b_c, each operation rounded on
// its own (__dsub_rn / __dmul_rn / __dadd_rn: no FMA contraction), columns in order.  That is the value a numpy loop over
// the columns gives, and it does not depend on which row is the query.  From it:
//   radius pass   r2[i] = the (k+1)-th smallest d2(A_i, A_j) over all j (self included), run on R and then on F;
//   cross pass    count[j] = #{i : d2(R_i, F_j) < r2[i]}, flags[i] bit 0 = some j has d2(R_i, F_j) < s2[j] (recall),
//                 bit 1 = some j has d2(R_i, F_j) < r2[i] (coverage);
//   tally         { #{j : count[j] > 0}, sum_j count[j], #recall flags, #coverage flags } as uint64.
//
// Both passes walk 64 x 64 pair tiles: query and candidate rows are staged in 16-column chunks, transposed, in shared
// memory, and each of the 256 threads keeps a 4 x 4 register tile of d2.  In the radius pass the tile is written to
// shared memory and warp w scans rows 8w .. 8w + 7: each row keeps its k+1 smallest values as a set spread over the
// lanes (slot l on lane l, slot 32 on lane 0), and the largest of the set, the running threshold, rejects a candidate
// with one compare; a candidate below it replaces the largest slot.  The (k+1)-th smallest value of a multiset does not
// depend on the order the values arrive in, so the radius is exact whatever the schedule.  When the row blocks alone
// cannot fill the GPU, the candidate tiles are split into slices; every slice writes its set of k+1 values per row and
// a merge kernel takes the (k+1)-th smallest of their union.  The cross pass sums per-fake counts in shared memory and
// adds them to the global counts once per CTA and candidate tile; the per-real flags are OR-ed per CTA and written with
// atomicOr.  All results are integers or selected values, so neither the slicing nor the scheduling changes any bit.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <algorithm>

#include "../../include/rnvp.h"

int rnvp_fail(int code, const char* msg);

namespace {

constexpr int QB = 64;                      // query rows per CTA
constexpr int CB = 64;                      // candidate rows per pair tile
constexpr int KC = 16;                      // feature columns staged per chunk
constexpr int LDS = QB + 1;                 // stride of the transposed staging buffers (doubles)
constexpr int LDD = CB;                     // row stride of the d2 tile of the radius pass
constexpr int THREADS = 256;                // 16 x 16 threads, 4 x 4 pairs each
constexpr int RPW = QB / (THREADS / 32);    // query rows scanned per warp
constexpr int TARGET_CTAS = 296;            // two CTAs on each of the 148 SMs of a B200
constexpr int64_t WS_BUDGET = int64_t(1) << 30;   // bytes of slice lists at most
constexpr unsigned FULL = 0xffffffffu;

constexpr size_t STAGE_BYTES = 2 * KC * LDS * sizeof(double);
constexpr size_t RADIUS_SMEM = STAGE_BYTES + QB * LDD * sizeof(double);

__device__ inline int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }

// d2[r][s] = d2(A[ty + 16 r], B[tx + 16 s]) for the 4 x 4 pairs of this thread; rows at or past va / vb read as zeros
__device__ inline void pair_tile(const double* __restrict__ A, int va, const double* __restrict__ B, int vb, int D,
                                 double* sA, double* sB, double (&d2)[4][4]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int s = 0; s < 4; ++s) d2[r][s] = 0.0;
  for (int k0 = 0; k0 < D; k0 += KC) {
    const int kc = min(KC, D - k0);
    __syncthreads();
    for (int e = tid; e < QB * kc; e += THREADS) {
      const int r = e / kc, kk = e - r * kc;
      sA[kk * LDS + r] = r < va ? __ldg(A + (int64_t)r * D + k0 + kk) : 0.0;
      sB[kk * LDS + r] = r < vb ? __ldg(B + (int64_t)r * D + k0 + kk) : 0.0;
    }
    __syncthreads();
    for (int kk = 0; kk < kc; ++kk) {
      double a[4], b[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = sA[kk * LDS + ty + 16 * r];
#pragma unroll
      for (int s = 0; s < 4; ++s) b[s] = sB[kk * LDS + tx + 16 * s];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          const double t = __dsub_rn(a[r], b[s]);
          d2[r][s] = __dadd_rn(d2[r][s], __dmul_rn(t, t));
        }
    }
  }
}

__device__ inline double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
  return v;
}

// The k+1 smallest values seen by one warp for one row: slot l on lane l (v0) and slot 32 on lane 0 (v1); unused slots
// hold -inf so that they are never the largest.  thr is the largest slot, +inf until k+1 values have arrived.
__device__ inline void set_init(int K1, double& v0, double& v1, double& thr) {
  const int lane = threadIdx.x & 31;
  v0 = lane < K1 ? INFINITY : -INFINITY;
  v1 = lane + 32 < K1 ? INFINITY : -INFINITY;
  thr = INFINITY;
}

// Offer the 64 values x0 (lane l: value l) and x1 (value 32 + l) to the set.  Warp-uniform control flow throughout.
__device__ inline void set_offer(double& v0, double& v1, double& thr, double x0, double x1) {
  const int lane = threadIdx.x & 31;
  unsigned m0 = __ballot_sync(FULL, x0 < thr), m1 = __ballot_sync(FULL, x1 < thr);
  while (m0 | m1) {
    double x;
    if (m0) {
      const int src = __ffs(m0) - 1;
      m0 &= m0 - 1;
      x = __shfl_sync(FULL, x0, src);
    } else {
      const int src = __ffs(m1) - 1;
      m1 &= m1 - 1;
      x = __shfl_sync(FULL, x1, src);
    }
    if (x < thr) {
      const unsigned b0 = __ballot_sync(FULL, v0 == thr);
      if (b0) {
        if (lane == __ffs(b0) - 1) v0 = x;
      } else {
        const unsigned b1 = __ballot_sync(FULL, v1 == thr);
        if (lane == __ffs(b1) - 1) v1 = x;
      }
      thr = warp_max(fmax(v0, v1));
      m0 &= __ballot_sync(FULL, x0 < thr);
      m1 &= __ballot_sync(FULL, x1 < thr);
    }
  }
}

// Write the set: its threshold to r2 (one slice) or its k+1 slots to the slice list of the row
__device__ inline void set_store(int K1, double v0, double v1, double thr, double* out, double* list) {
  const int lane = threadIdx.x & 31;
  if (list) {
    if (lane < K1) list[lane] = v0;
    if (lane == 0 && K1 > 32) list[32] = v1;
  } else if (lane == 0) {
    *out = thr;
  }
}

// grid (row blocks of A, slices).  Slice s walks candidate tiles [tiles s / slices, tiles (s + 1) / slices).
// slices == 1: r2[i] directly; otherwise part[(i * slices + s) * K1 + slot].
__global__ void __launch_bounds__(THREADS, 2)
    knn_radius_kernel(const double* __restrict__ A, int64_t n, int D, int K1, int64_t tiles, int slices,
                      double* __restrict__ r2, double* __restrict__ part) {
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;
  double* sB = sA + KC * LDS;
  double* sD = sB + KC * LDS;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
  const int64_t q0 = (int64_t)blockIdx.x * QB;
  const int vq = (int)min64(QB, n - q0);
  const int s = blockIdx.y;
  const int64_t t0 = tiles * s / slices, t1 = tiles * (s + 1) / slices;

  double v0[RPW], v1[RPW], thr[RPW];
#pragma unroll
  for (int r = 0; r < RPW; ++r) set_init(K1, v0[r], v1[r], thr[r]);

  double d2[4][4];
  for (int64_t t = t0; t < t1; ++t) {
    const int64_t c0 = t * CB;
    const int vc = (int)min64(CB, n - c0);
    pair_tile(A + q0 * D, vq, A + c0 * D, vc, D, sA, sB, d2);   // starts with __syncthreads: the last scan is done
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) sD[(ty + 16 * r) * LDD + tx + 16 * c] = tx + 16 * c < vc ? d2[r][c] : INFINITY;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
      const int row = warp * RPW + r;
      if (row < vq) set_offer(v0[r], v1[r], thr[r], sD[row * LDD + lane], sD[row * LDD + 32 + lane]);
    }
  }
#pragma unroll
  for (int r = 0; r < RPW; ++r) {
    const int64_t i = q0 + warp * RPW + r;
    if (i < n)
      set_store(K1, v0[r], v1[r], thr[r], r2 + i, slices > 1 ? part + (i * slices + s) * K1 : nullptr);
  }
}

// one warp per row: r2[i] = the K1-th smallest of the row's slices * K1 listed values
__global__ void __launch_bounds__(THREADS)
    knn_merge_kernel(const double* __restrict__ part, int64_t n, int K1, int slices, double* __restrict__ r2) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5);
  if (i >= n) return;
  const int total = slices * K1;
  const double* p = part + i * total;
  double v0, v1, thr;
  set_init(K1, v0, v1, thr);
  for (int c = 0; c < total; c += 64) {
    const double x0 = c + lane < total ? p[c + lane] : INFINITY;
    const double x1 = c + 32 + lane < total ? p[c + 32 + lane] : INFINITY;
    set_offer(v0, v1, thr, x0, x1);
  }
  set_store(K1, v0, v1, thr, r2 + i, nullptr);
}

// grid (row blocks of R, slices over the tiles of F)
__global__ void __launch_bounds__(THREADS, 2)
    knn_cross_kernel(const double* __restrict__ R, int64_t n, const double* __restrict__ F, int64_t m, int D,
                     const double* __restrict__ r2, const double* __restrict__ s2, int64_t tiles, int slices,
                     uint32_t* __restrict__ count, uint32_t* __restrict__ flags) {
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;
  double* sB = sA + KC * LDS;
  __shared__ double s_r[QB], s_s[CB];
  __shared__ uint32_t s_cnt[CB], s_flag[QB];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t i0 = (int64_t)blockIdx.x * QB;
  const int vq = (int)min64(QB, n - i0);
  const int s = blockIdx.y;
  const int64_t t0 = tiles * s / slices, t1 = tiles * (s + 1) / slices;
  if (tid < QB) {
    s_r[tid] = tid < vq ? r2[i0 + tid] : -INFINITY;      // padded rows are in no ball
    s_flag[tid] = 0u;
  }
  uint32_t cov = 0u, rec = 0u;                           // bit r: row ty + 16 r
  double d2[4][4];
  for (int64_t t = t0; t < t1; ++t) {
    const int64_t j0 = t * CB;
    const int vc = (int)min64(CB, m - j0);
    if (tid < CB) {
      s_s[tid] = tid < vc ? s2[j0 + tid] : -INFINITY;
      s_cnt[tid] = 0u;
    }
    pair_tile(R + i0 * D, vq, F + j0 * D, vc, D, sA, sB, d2);   // its first __syncthreads publishes s_s, s_cnt
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int col = tx + 16 * c;
      if (col < vc) {
        const double sj = s_s[col];
        uint32_t k = 0u;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const bool in_r = d2[r][c] < s_r[ty + 16 * r];
          k += in_r;
          cov |= (uint32_t)in_r << r;
          rec |= (uint32_t)(d2[r][c] < sj) << r;
        }
        if (k) atomicAdd(&s_cnt[col], k);
      }
    }
    __syncthreads();
    if (tid < vc && s_cnt[tid]) atomicAdd(&count[j0 + tid], s_cnt[tid]);
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const uint32_t f = ((rec >> r) & 1u) | (((cov >> r) & 1u) << 1);
    if (f) atomicOr(&s_flag[ty + 16 * r], f);
  }
  __syncthreads();
  if (tid < vq && s_flag[tid]) atomicOr(&flags[i0 + tid], s_flag[tid]);
}

// tallies[0] += #{j : count[j] > 0}, [1] += sum count[j], [2] += #recall flags, [3] += #coverage flags
__global__ void __launch_bounds__(THREADS)
    knn_tally_kernel(const uint32_t* __restrict__ count, int64_t m, const uint32_t* __restrict__ flags, int64_t n,
                     unsigned long long* __restrict__ tallies) {
  unsigned long long t[4] = {0ull, 0ull, 0ull, 0ull};
  const int64_t stride = (int64_t)gridDim.x * THREADS;
  for (int64_t j = (int64_t)blockIdx.x * THREADS + threadIdx.x; j < m; j += stride) {
    const uint32_t c = count[j];
    t[0] += c > 0u;
    t[1] += c;
  }
  for (int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x; i < n; i += stride) {
    const uint32_t f = flags[i];
    t[2] += f & 1u;
    t[3] += (f >> 1) & 1u;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t[q] += __shfl_xor_sync(FULL, t[q], o);
    if ((threadIdx.x & 31) == 0 && t[q]) atomicAdd(&tallies[q], t[q]);
  }
}

int64_t blocks_of(int64_t rows) { return (rows + QB - 1) / QB; }

// candidate slices for a pass with `rows` query rows over `cand` candidate rows
int slices_for(int64_t rows, int64_t cand) {
  const int64_t b = blocks_of(rows), tiles = (cand + CB - 1) / CB;
  int64_t s = b >= TARGET_CTAS ? 1 : (TARGET_CTAS + b - 1) / b;
  return (int)(s < tiles ? s : tiles);
}

// slices of the radius pass over `rows` rows, capped so that the slice lists fit WS_BUDGET
int radius_slices(int64_t rows, int K1) {
  int64_t s = slices_for(rows, rows);
  const int64_t cap = WS_BUDGET / (rows * K1 * (int64_t)sizeof(double));
  if (s > cap) s = cap;
  return (int)(s < 1 ? 1 : s);
}

int64_t radius_ws_bytes(int64_t rows, int K1) {
  const int s = radius_slices(rows, K1);
  return s > 1 ? rows * s * K1 * (int64_t)sizeof(double) : 0;
}

bool bad_rows(int64_t rows, int k) { return rows < 1 || rows > 0x7fffffff || (int64_t)k >= rows; }
bool bad_k(int k) { return k < 1 || k > RNVP_KNN_MAX_K; }

int launch_fail(const char* what) {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : rnvp_fail((int)e, what);
}

int radii(const double* d_A, int64_t n, int D, int k, double* d_r2, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int K1 = k + 1;
  const int slices = radius_slices(n, K1);
  if (slices > 1 && (!ws || ws_bytes < radius_ws_bytes(n, K1)))
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_radii: workspace too small (see rnvp_knn_workspace_bytes)");
  cudaError_t e = cudaFuncSetAttribute(knn_radius_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RADIUS_SMEM);
  if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_knn_radii: cudaFuncSetAttribute");
  double* part = slices > 1 ? (double*)ws : nullptr;
  knn_radius_kernel<<<dim3((unsigned)blocks_of(n), slices), THREADS, RADIUS_SMEM, st>>>(
      d_A, n, D, K1, (n + CB - 1) / CB, slices, d_r2, part);
  if (int rc = launch_fail("knn_radius_kernel")) return rc;
  if (slices == 1) return 0;
  const int64_t per = THREADS / 32;
  knn_merge_kernel<<<(unsigned)((n + per - 1) / per), THREADS, 0, st>>>(part, n, K1, slices, d_r2);
  return launch_fail("knn_merge_kernel");
}

int cross(const double* d_R, int64_t n, const double* d_F, int64_t m, int D, const double* d_r2, const double* d_s2,
          uint32_t* d_count, uint32_t* d_flags, uint64_t* d_tallies, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(d_count, 0, sizeof(uint32_t) * m, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_flags, 0, sizeof(uint32_t) * n, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_tallies, 0, 4 * sizeof(uint64_t), st);
  if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_knn_cross: memset");
  const int slices = slices_for(n, m);
  knn_cross_kernel<<<dim3((unsigned)blocks_of(n), slices), THREADS, STAGE_BYTES, st>>>(
      d_R, n, d_F, m, D, d_r2, d_s2, (m + CB - 1) / CB, slices, d_count, d_flags);
  if (int rc = launch_fail("knn_cross_kernel")) return rc;
  const int64_t most = n > m ? n : m;
  const int64_t grid = std::min<int64_t>((most + THREADS - 1) / THREADS, TARGET_CTAS);
  knn_tally_kernel<<<(unsigned)grid, THREADS, 0, st>>>(d_count, m, d_flags, n, (unsigned long long*)d_tallies);
  return launch_fail("knn_tally_kernel");
}

}  // namespace

extern "C" int64_t rnvp_knn_workspace_bytes(int64_t n, int64_t m, int D, int k) {
  if (D < 1 || bad_k(k) || bad_rows(n, k) || bad_rows(m, k))
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_workspace_bytes: need D >= 1, 1 <= k <= 32 and k < n, m < 2^31");
  const int64_t a = radius_ws_bytes(n, k + 1), b = radius_ws_bytes(m, k + 1);
  return a > b ? a : b;
}

extern "C" int rnvp_knn_radii(const double* d_A, int64_t n, int D, int k, double* d_radius2, void* d_workspace,
                              int64_t workspace_bytes, void* stream) {
  if (D < 1 || bad_k(k) || bad_rows(n, k))
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_radii: need D >= 1, 1 <= k <= 32 and k < n < 2^31");
  if (!d_A || !d_radius2) return rnvp_fail(RNVP_EINVAL, "rnvp_knn_radii: null buffer");
  return radii(d_A, n, D, k, d_radius2, d_workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int rnvp_knn_cross(const double* d_R, int64_t n, const double* d_F, int64_t m, int D, const double* d_r2,
                              const double* d_s2, uint32_t* d_count, uint32_t* d_flags, uint64_t* d_tallies,
                              void* stream) {
  if (D < 1 || n < 1 || m < 1 || n > 0x7fffffff || m > 0x7fffffff)
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_cross: need D >= 1 and 1 <= n, m < 2^31");
  if (!d_R || !d_F || !d_r2 || !d_s2 || !d_count || !d_flags || !d_tallies)
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_cross: null buffer");
  return cross(d_R, n, d_F, m, D, d_r2, d_s2, d_count, d_flags, d_tallies, (cudaStream_t)stream);
}

extern "C" int rnvp_knn_prdc(const double* d_R, int64_t n, const double* d_F, int64_t m, int D, int k, double* d_r2,
                             double* d_s2, uint32_t* d_count, uint32_t* d_flags, uint64_t* d_tallies, void* d_workspace,
                             int64_t workspace_bytes, void* stream) {
  if (D < 1 || bad_k(k) || bad_rows(n, k) || bad_rows(m, k))
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_prdc: need D >= 1, 1 <= k <= 32 and k < n, m < 2^31");
  if (!d_R || !d_F || !d_r2 || !d_s2 || !d_count || !d_flags || !d_tallies)
    return rnvp_fail(RNVP_EINVAL, "rnvp_knn_prdc: null buffer");
  const cudaStream_t st = (cudaStream_t)stream;
  if (int rc = radii(d_R, n, D, k, d_r2, d_workspace, workspace_bytes, st)) return rc;
  if (int rc = radii(d_F, m, D, k, d_s2, d_workspace, workspace_bytes, st)) return rc;
  return cross(d_R, n, d_F, m, D, d_r2, d_s2, d_count, d_flags, d_tallies, st);
}
