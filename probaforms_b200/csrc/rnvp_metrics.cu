// Bootstrap MMD and the moments of the bootstrap Frechet distance (probaforms/metrics/mmd.py, fd.py).
//
// Every bootstrap draw is a per-row count vector c (bincount of the resampled indices), so one draw of the reference's
// mmd_calc (mmd.py:8-21) over the concatenated rows Z = [X; Y] is
//   median = weighted median of d_ij over all ordered pairs (i, j), pair weight c_i c_j   (np.median of the (n+m)^2
//            distance matrix: a row drawn twice appears as two rows at distance 0 from each other, which is the pair
//            (i, i) with weight c_i^2, the same as the diagonal)
//   gamma  = 1 / (2 median^2)
//   mmd    = S_XX / n^2 + S_YY / m^2 - 2 S_XY / (n m),   S = sum c_i c_j exp(-gamma d_ij^2) over the pairs of a block.
// The distances are shared by all draws; only the weights and gamma differ.  The kernels never hold more than a 128 x 128
// tile of them: X and Y are cut separately into 128-row tiles (the last one of each padded with count-0 rows), the
// upper-triangular tile pairs are walked, and d^2 = sum (x - y)^2 is recomputed with FP32 FMA in every pass.
//
// The median is selected exactly on the bit pattern of d^2 (monotone for d^2 >= 0, sign bit always 0) in three radix
// passes over bits 30..20, 19..9 and 8..0.  Each pass builds count-weighted histograms in shared memory (uint32, flushed to
// uint64 before they can overflow) for a group of draws.  When (n+m)^2 is even, np.median averages the ranks k and k+1; if
// they fall in different buckets, rank k+1 is the smallest d^2 of its bucket, found by an atomicMin in the next pass (or
// given exactly by the bucket in the last pass).  The sum pass evaluates exp(-gamma d^2) with ex2.approx and keeps fp32
// partial sums over 64 terms per thread, combined in fp64 in a fixed order (per-warp slots, per-CTA partials summed by
// the finishing kernel), so a call's result does not depend on the order in which CTAs finish.
//
// Sharding (the staged entry points): shard s of N runs the CTAs [s hx, (s+1) hx) of a virtual radix grid N hx wide, and
// the CTA block [s sx / N, (s+1) sx / N) of every draw group of the sum pass.  Between stages the host adds the shards'
// histograms (exact integers), takes the minimum of their pending-bucket minima, and finally adds their per-CTA sum
// partials (each row is written by one shard only, the others hold +0.0), so every shard count gives the single-device bits.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <algorithm>

#include "../../include/rnvp.h"

int rnvp_fail(int code, const char* msg);

namespace {

constexpr int TILE = 128;                  // rows of a pair tile
constexpr int KC = 32;                     // feature columns staged per chunk
constexpr int LDS = TILE + 1;              // transposed tile stride (bank-conflict-free stores)
constexpr uint32_t LIST_CAP = 2 * KC * LDS * sizeof(float) / 8;   // pair-list entries that fit the staging buffers
constexpr int NB = 2048;                   // histogram buckets (11 bits)
constexpr int HG = 8;                      // draws per CTA in radix pass 0 (two CTAs per SM)
constexpr int HG1 = 16;                    // ... in passes 1 and 2 (one CTA per SM: the pair list needs the registers)
constexpr int SG = 32;                     // draws per CTA in the sum pass
constexpr int THREADS = 256;               // 16 x 16 threads, 8 x 8 pairs each
constexpr uint32_t MAX_TILE_COUNT = 46340; // 2 * 46340^2 < 2^32: one doubled tile pair fits a uint32 bucket
constexpr uint32_t NO_MIN = 0x7fffffffu;   // "no pending minimum": above every d^2 bit pattern (sign bit clear), and
                                           // still the largest value under a signed int32 MIN reduction

__host__ __device__ constexpr int pass_shift(int p) { return p == 0 ? 20 : (p == 1 ? 9 : 0); }
__host__ __device__ constexpr int pass_width(int p) { return p == 2 ? 9 : 11; }

struct MmdState {
  unsigned long long lo_rank;   // rank k (0-based) within the current prefix
  unsigned long long n_x, n_y;  // count totals of the draw
  uint32_t lo_prefix;           // bits of d^2 selected so far for rank k
  uint32_t two;                 // (n+m)^2 even: also rank k+1
  uint32_t hi_mode;             // 0: rank k+1 in the same bucket as k; 1: min of bucket hi_prefix pending; 2: hi_bits final
  uint32_t hi_prefix, hi_shift, hi_bits;
  float ng2;                    // -gamma * log2(e)
};

struct MmdWs {
  MmdState* st;
  unsigned long long* hist;     // [n_draws][NB]
  double* part;                 // [sum_ctas][n_draws][3]: per-CTA S_XX, S_YY, 2 S_XY of the sum pass
  uint32_t* minval;             // [n_draws]: smallest d^2 bits of the pending bucket (hi_mode 1), or NO_MIN
  uint32_t* smax;               // largest count sum of one tile over all draws
};

inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

constexpr int SUM_CTAS = 2048;             // CTAs of the sum pass, over all draw groups

int sum_groups(int n_draws) { return (n_draws + SG - 1) / SG; }
int64_t sum_ctas_per_group(int64_t ntp, int n_draws) {
  return std::max<int64_t>(1, std::min<int64_t>(ntp, SUM_CTAS / sum_groups(n_draws)));
}

MmdWs carve(void* ws, int n_draws, int64_t sum_ctas, size_t* bytes) {
  char* p = (char*)ws;
  size_t o = 0;
  MmdWs w;
  w.st = (MmdState*)(p + o);            o += align256(sizeof(MmdState) * n_draws);
  w.hist = (unsigned long long*)(p + o); o += align256(sizeof(unsigned long long) * NB * (size_t)n_draws);
  w.part = (double*)(p + o);            o += align256(sizeof(double) * 3 * (size_t)n_draws * sum_ctas);
  w.minval = (uint32_t*)(p + o);        o += align256(sizeof(uint32_t) * (size_t)n_draws);
  w.smax = (uint32_t*)(p + o);          o += align256(sizeof(uint32_t));
  *bytes = o;
  return w;
}

struct Geo {
  const float* X;
  const float* Y;
  int64_t n, m;
  int D;
  int64_t tx, ty;               // tiles of X and of Y
  const uint16_t* counts;       // [n_draws][n+m]
  int n_draws;
};

__device__ inline int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }

// rows of tile t: base pointer, valid rows, offset of its counts within a draw's row of counts
__device__ inline void tile_rows(const Geo& g, int64_t t, const float** base, int* valid, int64_t* cofs) {
  if (t < g.tx) {
    int64_t r0 = t * TILE;
    *base = g.X + r0 * g.D;
    *valid = (int)min64(TILE, g.n - r0);
    *cofs = r0;
  } else {
    int64_t r0 = (t - g.tx) * TILE;
    *base = g.Y + r0 * g.D;
    *valid = (int)min64(TILE, g.m - r0);
    *cofs = g.n + r0;
  }
}

// pair tile q of the upper triangle, ordered by column tile: q = tb (tb + 1) / 2 + ta, ta <= tb
__device__ inline void tile_pair(int64_t q, int64_t* ta, int64_t* tb) {
  int64_t b = (int64_t)((sqrt(8.0 * (double)q + 1.0) - 1.0) * 0.5);
  while (b * (b + 1) / 2 > q) --b;
  while ((b + 1) * (b + 2) / 2 <= q) ++b;
  *tb = b;
  *ta = q - b * (b + 1) / 2;
}

__device__ inline float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// d2[r][s] = |z_a(ty + 16 r) - z_b(tx + 16 s)|^2 for the 8 x 8 pairs of this thread, FP32 FMA over KC-column chunks
__device__ inline void tile_d2(const Geo& g, const float* A, int va, const float* B, int vb, float* sA, float* sB,
                               float (&d2)[8][8]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int s = 0; s < 8; ++s) d2[r][s] = 0.f;
  for (int k0 = 0; k0 < g.D; k0 += KC) {
    const int kc = min(KC, g.D - k0);
    __syncthreads();
    // only the kc staged columns: at small D the loads of a tile are a few per thread, all issued before the stores
#pragma unroll 4
    for (int e = tid; e < TILE * kc; e += THREADS) {
      const int r = e / kc, kk = e - r * kc;
      const float va_ = r < va ? __ldg(A + (int64_t)r * g.D + k0 + kk) : 0.f;
      const float vb_ = r < vb ? __ldg(B + (int64_t)r * g.D + k0 + kk) : 0.f;
      sA[kk * LDS + r] = va_;
      sB[kk * LDS + r] = vb_;
    }
    __syncthreads();
    for (int kk = 0; kk < kc; ++kk) {
      float a[8], b[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) a[r] = sA[kk * LDS + ty + 16 * r];
#pragma unroll
      for (int s = 0; s < 8; ++s) b[s] = sB[kk * LDS + tx + 16 * s];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int s = 0; s < 8; ++s) {
          const float d = a[r] - b[s];
          d2[r][s] = fmaf(d, d, d2[r][s]);
        }
    }
  }
}

__global__ void mmd_prep_kernel(Geo g, MmdWs w) {
  // grid (tiles, n_draws), 128 threads: count sum of one tile of one draw
  const int64_t t = blockIdx.x;
  const int b = blockIdx.y;
  const float* base;
  int valid;
  int64_t cofs;
  tile_rows(g, t, &base, &valid, &cofs);
  uint32_t c = threadIdx.x < valid ? g.counts[(int64_t)b * (g.n + g.m) + cofs + threadIdx.x] : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  __shared__ uint32_t part[TILE / 32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t s = 0;
    for (int q = 0; q < TILE / 32; ++q) s += part[q];
    atomicMax(w.smax, s);
    atomicAdd(t < g.tx ? &w.st[b].n_x : &w.st[b].n_y, (unsigned long long)s);
  }
}

__global__ void mmd_init_kernel(MmdWs w, int n_draws) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_draws) return;
  MmdState& s = w.st[b];
  const unsigned long long N = s.n_x + s.n_y, W = N * N;
  s.lo_rank = W ? (W - 1) / 2 : 0;
  s.two = (W & 1ull) == 0 ? 1u : 0u;
  s.lo_prefix = 0;
  s.hi_mode = 0;
  w.minval[b] = NO_MIN;
}

// Radix pass PASS (MODE 0) or the exponential-sum pass (MODE 1) for draws [group*blockIdx.y, +group).  CTA blockIdx.x is
// CTA cta0 + blockIdx.x of a virtual grid `ctas` wide striding over the pair tiles (a shard's part of the grid; cta0 = 0,
// ctas = gridDim.x on one device).  In passes 1 and 2 only pairs inside the bucket ranges still open for some draw of the
// group (at most a few buckets of the previous pass) reach the per-draw loop.
template <int MODE, int PASS>
__global__ void __launch_bounds__(THREADS, (MODE == 0 && PASS > 0) ? 1 : 2)
    mmd_pass_kernel(Geo g, MmdWs w, int group, int64_t cta0, int64_t ctas) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sA = (float*)smem_raw;
  float* sB = sA + KC * LDS;
  uint32_t* sCA = (uint32_t*)(sB + KC * LDS);                    // [group][TILE] counts (as float in MODE 1)
  uint32_t* sCB = sCA + group * TILE;
  uint32_t* shist = sCB + group * TILE;                           // MODE 0: [group][NB]; MODE 1: double [warp][group][3]
  __shared__ uint32_t s_pfx[SG], s_hpfx[SG], s_hshift[SG], s_hmode[SG], s_min[SG];   // SG >= HG1 >= HG
  __shared__ float s_ng2[SG];
  __shared__ uint32_t s_rlo, s_rhi;       // [s_rlo, s_rhi]: d^2 bit patterns some draw of the group still selects in
  __shared__ uint32_t s_cnt;              // entries of the pair list

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31;
  const int b0 = blockIdx.y * group;
  const int nb = min(group, g.n_draws - b0);
  const int64_t T = g.tx + g.ty;
  const int64_t ntp = T * (T + 1) / 2;
  constexpr int pshift = pass_shift(PASS), pw = pass_width(PASS), lshift = pshift + pw;
  double* ssum = (double*)shist;

  if (MODE == 0) {
    for (int e = tid; e < group * NB; e += THREADS) shist[e] = 0u;
  } else {
    for (int e = tid; e < (THREADS / 32) * group * 3; e += THREADS) ssum[e] = 0.0;
  }
  if (tid < nb) {
    const MmdState& s = w.st[b0 + tid];
    s_pfx[tid] = s.lo_prefix;
    s_hmode[tid] = s.hi_mode;
    s_hpfx[tid] = s.hi_prefix;
    s_hshift[tid] = s.hi_shift;
    s_min[tid] = NO_MIN;
    if (MODE == 1) s_ng2[tid] = s.ng2;
  }
  if (tid == 0) {
    uint32_t lo = 0xffffffffu, hi = 0u;
    for (int gi = 0; gi < nb; ++gi) {
      const MmdState& s = w.st[b0 + gi];
      const uint64_t l = (uint64_t)s.lo_prefix << lshift;
      lo = min(lo, (uint32_t)l);
      hi = max(hi, (uint32_t)(l + (1ull << lshift) - 1));   // < 2^31: the sign bit is never set
      if (s.hi_mode == 1) {
        const uint64_t h = (uint64_t)s.hi_prefix << s.hi_shift;
        lo = min(lo, (uint32_t)h);
        hi = max(hi, (uint32_t)(h + (1ull << s.hi_shift) - 1));
      }
    }
    s_rlo = lo;
    s_rhi = hi;
    s_cnt = 0;
  }
  // tile pairs between flushes of the uint32 histograms: each adds at most 2 * smax^2 to a bucket
  const unsigned long long sm = *w.smax;
  const unsigned long long per = 2ull * sm * sm;
  const int64_t flush_every = per ? (int64_t)(0xffffffffull / per) : INT64_MAX;
  int64_t since_flush = 0;
  __syncthreads();

  float d2[8][8];
  for (int64_t q = cta0 + blockIdx.x; q < ntp; q += ctas) {
    int64_t ta, tb;
    tile_pair(q, &ta, &tb);
    const float *A, *B;
    int va, vb;
    int64_t ca0, cb0;
    tile_rows(g, ta, &A, &va, &ca0);
    tile_rows(g, tb, &B, &vb, &cb0);
    const uint32_t mult = ta == tb ? 1u : 2u;          // off-diagonal tiles stand for (i, j) and (j, i)
    const int blk = tb < g.tx ? 0 : (ta >= g.tx ? 1 : 2);
    tile_d2(g, A, va, B, vb, sA, sB, d2);               // begins and ends with __syncthreads on the staging buffers
#pragma unroll 4
    for (int e = tid; e < nb * TILE; e += THREADS) {
      const int gi = e / TILE, r = e % TILE;
      const uint16_t* cr = g.counts + (int64_t)(b0 + gi) * (g.n + g.m);
      const uint32_t a = r < va ? cr[ca0 + r] : 0u, b = r < vb ? cr[cb0 + r] : 0u;
      if (MODE == 0) {
        sCA[e] = a;
        sCB[e] = b;
      } else {
        ((float*)sCA)[e] = (float)a;
        ((float*)sCB)[e] = (float)b;
      }
    }
    __syncthreads();

    if (MODE == 0 && PASS == 0) {
      for (int gi = 0; gi < nb; ++gi) {
        uint32_t* h = shist + gi * NB;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const uint32_t ca = sCA[gi * TILE + ty + 16 * r] * mult;
          if (ca == 0) continue;
#pragma unroll
          for (int s = 0; s < 8; ++s) {
            const uint32_t wgt = ca * sCB[gi * TILE + tx + 16 * s];
            if (wgt) atomicAdd(h + ((__float_as_uint(d2[r][s]) >> pshift) & (NB - 1)), wgt);
          }
        }
      }
    } else if (MODE == 0) {
      // Passes 1 and 2: a few percent of the pairs at most fall into a bucket still open for some draw of the group.
      // Compact those into a list on the staging buffers (free until the next tile) and run the per-draw loop over the
      // list.  A tile with more than LIST_CAP such pairs recomputes its d^2 and takes the per-draw loop over all pairs instead.
      uint2* list = (uint2*)sA;                        // (d^2 bits, row_a << 8 | row_b)
      const uint32_t rlo = s_rlo, rw = s_rhi - s_rlo;
      uint32_t mine = 0;
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int s = 0; s < 8; ++s) mine += __float_as_uint(d2[r][s]) - rlo <= rw;
      uint32_t at = mine ? atomicAdd(&s_cnt, mine) : 0u;
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int s = 0; s < 8; ++s) {
          const uint32_t bits = __float_as_uint(d2[r][s]);
          if (bits - rlo <= rw) {
            if (at < LIST_CAP) list[at] = make_uint2(bits, ((ty + 16 * r) << 8) | (tx + 16 * s));
            ++at;
          }
        }
      __syncthreads();
      const uint32_t cnt = s_cnt;
      if (cnt <= LIST_CAP) {
        for (uint32_t e = tid; e < cnt; e += THREADS) {
          const uint2 it = list[e];
          const uint32_t bits = it.x, ia = it.y >> 8, ib = it.y & 255;
          for (int gi = 0; gi < nb; ++gi) {
            const uint32_t wgt = sCA[gi * TILE + ia] * sCB[gi * TILE + ib] * mult;
            if (wgt == 0) continue;
            if ((bits >> lshift) == s_pfx[gi]) atomicAdd(shist + gi * NB + ((bits >> pshift) & (NB - 1)), wgt);
            if (s_hmode[gi] == 1 && (bits >> s_hshift[gi]) == s_hpfx[gi]) atomicMin(&s_min[gi], bits);
          }
        }
      } else {
        tile_d2(g, A, va, B, vb, sA, sB, d2);         // the list overwrote the staged rows
        for (int gi = 0; gi < nb; ++gi) {
          const uint32_t pfx = s_pfx[gi], hm = s_hmode[gi], hp = s_hpfx[gi], hs = s_hshift[gi];
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const uint32_t ca = sCA[gi * TILE + ty + 16 * r] * mult;
            if (ca == 0) continue;
#pragma unroll
            for (int s = 0; s < 8; ++s) {
              const uint32_t wgt = ca * sCB[gi * TILE + tx + 16 * s];
              const uint32_t bits = __float_as_uint(d2[r][s]);
              if (wgt == 0) continue;
              if ((bits >> lshift) == pfx) atomicAdd(shist + gi * NB + ((bits >> pshift) & (NB - 1)), wgt);
              if (hm == 1 && (bits >> hs) == hp) atomicMin(&s_min[gi], bits);
            }
          }
        }
      }
      __syncthreads();
      if (tid == 0) s_cnt = 0;                         // next written after the barriers of the next tile's staging
    } else {
      const float* fa = (const float*)sCA;
      const float* fb = (const float*)sCB;
      for (int gi = 0; gi < nb; ++gi) {
        const float ng2 = s_ng2[gi];
        float acc = 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          float t = 0.f;
#pragma unroll
          for (int s = 0; s < 8; ++s) t = fmaf(fb[gi * TILE + tx + 16 * s], ex2_approx(ng2 * d2[r][s]), t);
          acc = fmaf(fa[gi * TILE + ty + 16 * r], t, acc);
        }
        double v = (double)acc * (double)mult;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) ssum[((tid >> 5) * group + gi) * 3 + blk] += v;   // this warp's own slot
      }
    }
    if (MODE == 0 && ++since_flush >= flush_every) {
      __syncthreads();
      for (int e = tid; e < nb * NB; e += THREADS)
        if (shist[e]) {
          atomicAdd(&w.hist[(int64_t)b0 * NB + e], (unsigned long long)shist[e]);
          shist[e] = 0u;
        }
      since_flush = 0;
    }
  }
  __syncthreads();
  if (MODE == 0) {
    for (int e = tid; e < nb * NB; e += THREADS)
      if (shist[e]) atomicAdd(&w.hist[(int64_t)b0 * NB + e], (unsigned long long)shist[e]);
    if (tid < nb && s_hmode[tid] == 1 && s_min[tid] != NO_MIN) atomicMin(&w.minval[b0 + tid], s_min[tid]);
  } else {
    for (int e = tid; e < nb * 3; e += THREADS) {
      double t = 0.0;
      for (int wp = 0; wp < THREADS / 32; ++wp) t += ssum[wp * group * 3 + e];
      w.part[((cta0 + blockIdx.x) * g.n_draws + b0) * 3 + e] = t;
    }
  }
}

// After radix pass `pass`: pick the buckets of ranks k (and k+1) per draw, zero the histogram for the next pass.
// After the last pass: the median and gamma.  One CTA per draw.
__global__ void mmd_select_kernel(MmdWs w, int pass, double* d_median) {
  const int b = blockIdx.x;
  unsigned long long* H = w.hist + (int64_t)b * NB;
  if (threadIdx.x == 0) {
    MmdState& s = w.st[b];
    const int shift = pass_shift(pass), width = pass_width(pass);
    if (s.hi_mode == 1) {                     // its minimum was taken during this pass
      s.hi_bits = w.minval[b];
      s.hi_mode = 2;
    }
    unsigned long long cum = 0;
    int bl = 0;
    for (; bl < NB - 1; ++bl) {
      if (cum + H[bl] > s.lo_rank) break;
      cum += H[bl];
    }
    const unsigned long long rel = s.lo_rank - cum;
    if (s.two && s.hi_mode == 0 && rel + 1 >= H[bl]) {   // rank k is the last of its bucket: k+1 opens the next one
      int bh = bl + 1;
      while (bh < NB - 1 && H[bh] == 0) ++bh;
      const uint32_t hp = (s.lo_prefix << width) | (uint32_t)bh;
      if (pass == 2) {
        s.hi_bits = hp;
        s.hi_mode = 2;
      } else {
        s.hi_prefix = hp;
        s.hi_shift = shift;
        s.hi_mode = 1;
        w.minval[b] = NO_MIN;
      }
    }
    s.lo_prefix = (s.lo_prefix << width) | (uint32_t)bl;
    s.lo_rank = rel;
    if (pass == 2) {
      const uint32_t lo = s.lo_prefix, hi = (s.two && s.hi_mode == 2) ? s.hi_bits : lo;
      const double med = 0.5 * (sqrt((double)__uint_as_float(lo)) + sqrt((double)__uint_as_float(hi)));
      const double gamma = 1.0 / (2.0 * med * med);
      s.ng2 = (float)(-gamma * 1.4426950408889634);
      d_median[b] = *w.smax > MAX_TILE_COUNT ? nan("") : med;
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < NB; e += blockDim.x) H[e] = 0ull;
}

__global__ void mmd_finish_kernel(MmdWs w, int n_draws, int sum_ctas, double* d_mmd) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_draws) return;
  const MmdState& s = w.st[b];
  const double nx = (double)s.n_x, ny = (double)s.n_y;
  double S[3] = {0.0, 0.0, 0.0};
  for (int c = 0; c < sum_ctas; ++c)
    for (int k = 0; k < 3; ++k) S[k] += w.part[((int64_t)c * n_draws + b) * 3 + k];
  d_mmd[b] = *w.smax > MAX_TILE_COUNT ? nan("") : S[0] / (nx * nx) + S[1] / (ny * ny) - S[2] / (nx * ny);
}

// ---------------------------------------------------------------------------------------------------------------------
// Bootstrap moments: sum_i c_bi x_i and sum_i c_bi x_i x_i^T for every draw b.  A CTA owns a 32 x 32 tile of the outer
// product and MG draws over all rows; fp32 partials over 128-row chunks are added to fp64 registers in row order, so
// every output is written once, by one thread, in a fixed order.
constexpr int MG = 1;
constexpr int MR = 128;

__global__ void __launch_bounds__(THREADS) boot_moments_kernel(const float* X, int64_t n, int D, const uint16_t* counts,
                                                              int n_draws, int kt_tiles, double* d_sum, double* d_outer) {
  __shared__ float xj[MR][33], xk[MR][33], sc[MG][MR];
  const int tid = threadIdx.x;
  const int jt = blockIdx.y / kt_tiles, kt = blockIdx.y % kt_tiles;
  const int b0 = blockIdx.z * MG, nb = min(MG, n_draws - b0);
  const bool do_sum = kt == 0 && tid < 32;
  double acc[MG][4], sacc[MG];
#pragma unroll
  for (int g = 0; g < MG; ++g) {
    sacc[g] = 0.0;
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[g][q] = 0.0;
  }
  for (int64_t c0 = 0; c0 < n; c0 += MR) {
    const int rows = (int)min64(MR, n - c0);
    __syncthreads();
    for (int e = tid; e < MR * 32; e += THREADS) {
      const int r = e >> 5, c = e & 31;
      const int j = jt * 32 + c, k = kt * 32 + c;
      xj[r][c] = (r < rows && j < D) ? X[(c0 + r) * D + j] : 0.f;
      xk[r][c] = (r < rows && k < D) ? X[(c0 + r) * D + k] : 0.f;
    }
    for (int e = tid; e < MG * MR; e += THREADS) {
      const int g = e / MR, r = e % MR;
      sc[g][r] = (g < nb && r < rows) ? (float)counts[(int64_t)(b0 + g) * n + c0 + r] : 0.f;
    }
    __syncthreads();
    float p32[MG][4], s32[MG];
#pragma unroll
    for (int g = 0; g < MG; ++g) {
      s32[g] = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) p32[g][q] = 0.f;
    }
    const int k = tid & 31;
    for (int r = 0; r < rows; ++r) {
      const float xkv = xk[r][k];
      float pr[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) pr[q] = xj[r][(tid >> 5) + 8 * q] * xkv;
#pragma unroll
      for (int g = 0; g < MG; ++g) {
        const float c = sc[g][r];
#pragma unroll
        for (int q = 0; q < 4; ++q) p32[g][q] = fmaf(c, pr[q], p32[g][q]);
        if (do_sum) s32[g] = fmaf(c, xj[r][tid], s32[g]);
      }
    }
#pragma unroll
    for (int g = 0; g < MG; ++g) {
      sacc[g] += (double)s32[g];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[g][q] += (double)p32[g][q];
    }
  }
  const int kk = kt * 32 + (tid & 31);
  for (int g = 0; g < nb; ++g) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = jt * 32 + (tid >> 5) + 8 * q;
      if (j < D && kk < D) d_outer[((int64_t)(b0 + g) * D + j) * D + kk] = acc[g][q];
    }
    if (do_sum && jt * 32 + tid < D) d_sum[(int64_t)(b0 + g) * D + jt * 32 + tid] = sacc[g];
  }
}

int num_sms() {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}

size_t pass_smem(int mode, int group) {
  const size_t tiles = 2 * KC * LDS * sizeof(float) + 2 * (size_t)group * TILE * sizeof(uint32_t);
  return tiles + (mode == 0 ? (size_t)group * NB * sizeof(uint32_t) : (size_t)(THREADS / 32) * group * 3 * sizeof(double));
}

template <int MODE, int PASS>
void launch_pass(const Geo& g, const MmdWs& w, dim3 grid, int group, int64_t cta0, int64_t ctas, cudaStream_t st) {
  const size_t smem = pass_smem(MODE, group);
  // per device, so set on every call (no synchronisation)
  cudaFuncSetAttribute(mmd_pass_kernel<MODE, PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)pass_smem(MODE, MODE == 1 ? SG : (PASS == 0 ? HG : HG1)));
  mmd_pass_kernel<MODE, PASS><<<grid, THREADS, smem, st>>>(g, w, group, cta0, ctas);
}

int launch_fail(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return 0;
  return rnvp_fail((int)e, what);
}

// One call's geometry and workspace, shared by the stages of rnvp_mmd_draws and the staged entry points.
struct MmdCall {
  Geo g;
  MmdWs w;
  int64_t ntp;                  // upper-triangular pair tiles
  size_t need;                  // workspace bytes
  int hgroups, hg, h1groups, hg1, sgroups, sg;
  int64_t sx;                   // sum-pass CTAs per draw group: a function of the problem only
};

int mmd_setup(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
              void* d_workspace, int64_t workspace_bytes, MmdCall* c) {
  if (n < 1 || m < 1 || D < 1 || n_draws < 1) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd: bad sizes");
  if (!d_X || !d_Y || !d_counts || !d_workspace) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd: null buffer");
  c->g = Geo{d_X, d_Y, n, m, D, (n + TILE - 1) / TILE, (m + TILE - 1) / TILE, d_counts, n_draws};
  const int64_t T = c->g.tx + c->g.ty;
  c->ntp = T * (T + 1) / 2;
  c->sx = sum_ctas_per_group(c->ntp, n_draws);
  c->w = carve(d_workspace, n_draws, c->sx, &c->need);
  if (workspace_bytes < (int64_t)c->need)
    return rnvp_fail(RNVP_EINVAL, "rnvp_mmd: workspace too small (see rnvp_mmd_workspace_bytes)");
  if (T > 0x7fffffff || n_draws > 65535) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd: too many tiles or draws");
  // draws split evenly over the fewest groups of at most HG (HG1, SG) draws
  c->hgroups = (n_draws + HG - 1) / HG;
  c->hg = (n_draws + c->hgroups - 1) / c->hgroups;
  c->h1groups = (n_draws + HG1 - 1) / HG1;
  c->hg1 = (n_draws + c->h1groups - 1) / c->h1groups;
  c->sgroups = sum_groups(n_draws);
  c->sg = (n_draws + c->sgroups - 1) / c->sgroups;
  return 0;
}

int mmd_begin(const MmdCall& c, void* d_workspace, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(d_workspace, 0, c.need, st);
  if (e != cudaSuccess) return rnvp_fail((int)e, "rnvp_mmd: workspace memset");
  const int64_t T = c.g.tx + c.g.ty;
  mmd_prep_kernel<<<dim3((unsigned)T, (unsigned)c.g.n_draws), TILE, 0, st>>>(c.g, c.w);
  mmd_init_kernel<<<(c.g.n_draws + 127) / 128, 128, 0, st>>>(c.w, c.g.n_draws);
  return launch_fail("mmd_prep_kernel");
}

// Radix pass `pass` of shard `shard` of n_shards: this device's grid (as on one device) at CTA offset shard * grid.
// Every shard must see the same SM count, so that the shards' grids tile one virtual grid.
int mmd_hist_pass(const MmdCall& c, int pass, int shard, int n_shards, cudaStream_t st) {
  const int sms = num_sms();
  if (pass == 0) {
    const int64_t hx = std::max<int64_t>(1, std::min<int64_t>(c.ntp, (int64_t)8 * sms / c.hgroups));
    launch_pass<0, 0>(c.g, c.w, dim3((unsigned)hx, c.hgroups), c.hg, shard * hx, n_shards * hx, st);
  } else {
    const int64_t h1x = std::max<int64_t>(1, std::min<int64_t>(c.ntp, (int64_t)4 * sms / c.h1groups));
    const dim3 grid1((unsigned)h1x, c.h1groups);
    if (pass == 1) launch_pass<0, 1>(c.g, c.w, grid1, c.hg1, shard * h1x, n_shards * h1x, st);
    else launch_pass<0, 2>(c.g, c.w, grid1, c.hg1, shard * h1x, n_shards * h1x, st);
  }
  return launch_fail("mmd_pass_kernel<hist>");
}

int mmd_select(const MmdCall& c, int pass, double* d_median, cudaStream_t st) {
  mmd_select_kernel<<<c.g.n_draws, 256, 0, st>>>(c.w, pass, d_median);
  return launch_fail("mmd_select_kernel");
}

// Sum pass of shard `shard`: CTAs [shard sx / n_shards, (shard+1) sx / n_shards) of every draw group (none: no launch).
int mmd_sum_pass(const MmdCall& c, int shard, int n_shards, cudaStream_t st) {
  const int64_t c0 = c.sx * shard / n_shards, c1 = c.sx * (shard + 1) / n_shards;
  if (c1 == c0) return 0;
  launch_pass<1, 0>(c.g, c.w, dim3((unsigned)(c1 - c0), c.sgroups), c.sg, c0, c.sx, st);
  return launch_fail("mmd_pass_kernel<sum>");
}

int mmd_finish(const MmdCall& c, double* d_mmd, cudaStream_t st) {
  mmd_finish_kernel<<<(c.g.n_draws + 127) / 128, 128, 0, st>>>(c.w, c.g.n_draws, (int)c.sx, d_mmd);
  return launch_fail("mmd_finish_kernel");
}

int check_shard(const char* who, int shard, int n_shards) {
  if (n_shards < 1 || shard < 0 || shard >= n_shards) return rnvp_fail(RNVP_EINVAL, who);
  return 0;
}

}  // namespace

extern "C" {

int64_t rnvp_mmd_workspace_bytes(int64_t n, int64_t m, int D, int n_draws) {
  if (n < 1 || m < 1 || D < 1 || n_draws < 1) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_workspace_bytes: bad sizes");
  size_t bytes;
  const int64_t T = (n + TILE - 1) / TILE + (m + TILE - 1) / TILE;
  carve(nullptr, n_draws, sum_ctas_per_group(T * (T + 1) / 2, n_draws), &bytes);
  return (int64_t)bytes;
}

int rnvp_mmd_draws(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                   double* d_median, double* d_mmd, void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (!d_median || !d_mmd) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_draws: null buffer");
  MmdCall c;
  if (int rc = mmd_setup(d_X, n, d_Y, m, D, d_counts, n_draws, d_workspace, workspace_bytes, &c)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = mmd_begin(c, d_workspace, st)) return rc;
  for (int p = 0; p < 3; ++p) {
    if (int rc = mmd_hist_pass(c, p, 0, 1, st)) return rc;
    if (int rc = mmd_select(c, p, d_median, st)) return rc;
  }
  if (int rc = mmd_sum_pass(c, 0, 1, st)) return rc;
  return mmd_finish(c, d_mmd, st);
}

int rnvp_mmd_layout(int64_t n, int64_t m, int n_draws, int64_t* offsets) {
  if (n < 1 || m < 1 || n_draws < 1 || n_draws > 65535 || !offsets)
    return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_layout: bad sizes or null buffer");
  const int64_t T = (n + TILE - 1) / TILE + (m + TILE - 1) / TILE;
  const int64_t sx = sum_ctas_per_group(T * (T + 1) / 2, n_draws);
  size_t bytes;
  const MmdWs w = carve(nullptr, n_draws, sx, &bytes);
  offsets[0] = (int64_t)(uintptr_t)w.hist;
  offsets[1] = (int64_t)(sizeof(unsigned long long) * NB * (size_t)n_draws);
  offsets[2] = (int64_t)(uintptr_t)w.minval;
  offsets[3] = (int64_t)(sizeof(uint32_t) * (size_t)n_draws);
  offsets[4] = (int64_t)(uintptr_t)w.part;
  offsets[5] = (int64_t)(sizeof(double) * 3 * (size_t)n_draws * sx);
  return 0;
}

// the common arguments of every stage: validated as rnvp_mmd_draws validates them
#define MMD_STAGE_SETUP                                                                                           \
  MmdCall c;                                                                                                      \
  if (int rc = mmd_setup(d_X, n, d_Y, m, D, d_counts, n_draws, d_workspace, workspace_bytes, &c)) return rc;      \
  cudaStream_t st = (cudaStream_t)stream;

int rnvp_mmd_begin(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                   void* d_workspace, int64_t workspace_bytes, void* stream) {
  MMD_STAGE_SETUP
  return mmd_begin(c, d_workspace, st);
}

int rnvp_mmd_hist_pass(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts,
                       int n_draws, void* d_workspace, int64_t workspace_bytes, int pass, int shard, int n_shards,
                       void* stream) {
  if (pass < 0 || pass > 2) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_hist_pass: pass must be 0, 1 or 2");
  if (int rc = check_shard("rnvp_mmd_hist_pass: need 0 <= shard < n_shards", shard, n_shards)) return rc;
  MMD_STAGE_SETUP
  return mmd_hist_pass(c, pass, shard, n_shards, st);
}

int rnvp_mmd_select(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                    void* d_workspace, int64_t workspace_bytes, int pass, double* d_median, void* stream) {
  if (pass < 0 || pass > 2) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_select: pass must be 0, 1 or 2");
  if (!d_median) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_select: null buffer");
  MMD_STAGE_SETUP
  return mmd_select(c, pass, d_median, st);
}

int rnvp_mmd_sum_pass(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts,
                      int n_draws, void* d_workspace, int64_t workspace_bytes, int shard, int n_shards, void* stream) {
  if (int rc = check_shard("rnvp_mmd_sum_pass: need 0 <= shard < n_shards", shard, n_shards)) return rc;
  MMD_STAGE_SETUP
  return mmd_sum_pass(c, shard, n_shards, st);
}

int rnvp_mmd_finish(const float* d_X, int64_t n, const float* d_Y, int64_t m, int D, const uint16_t* d_counts, int n_draws,
                    void* d_workspace, int64_t workspace_bytes, double* d_mmd, void* stream) {
  if (!d_mmd) return rnvp_fail(RNVP_EINVAL, "rnvp_mmd_finish: null buffer");
  MMD_STAGE_SETUP
  return mmd_finish(c, d_mmd, st);
}

#undef MMD_STAGE_SETUP

int rnvp_boot_moments(const float* d_X, int64_t n, int D, const uint16_t* d_counts, int n_draws, double* d_sum,
                      double* d_outer, void* stream) {
  if (n < 1 || D < 1 || n_draws < 1) return rnvp_fail(RNVP_EINVAL, "rnvp_boot_moments: bad sizes");
  if (!d_X || !d_counts || !d_sum || !d_outer) return rnvp_fail(RNVP_EINVAL, "rnvp_boot_moments: null buffer");
  cudaStream_t st = (cudaStream_t)stream;
  const int kt = (D + 31) / 32;
  const int groups = (n_draws + MG - 1) / MG;
  if ((int64_t)kt * kt > 65535 || groups > 65535) return rnvp_fail(RNVP_EINVAL, "rnvp_boot_moments: too many features or draws");
  boot_moments_kernel<<<dim3(1, kt * kt, groups), THREADS, 0, st>>>(d_X, n, D, d_counts, n_draws, kt, d_sum, d_outer);
  return launch_fail("boot_moments_kernel");
}

}  // extern "C"
