// tcgen05 primitive self-test (rnvp_mma_selftest): D[128 x N] = A[128 x K] * B[N x K]^T with A
// staged in TMEM (tcgen05.st, one thread per row), B in shared memory in the no-swizzle K-major
// core-matrix layout, kind::tf32 MMAs issued by one thread, completion through tcgen05.commit on an
// mbarrier, and the accumulator read back with tcgen05.ld.  passes = 1: plain TF32;
// passes = 3: error-compensated split (A_hi*B_hi + A_lo*B_hi + A_hi*B_lo), fp32-grade accuracy.
// The fused coupling-layer kernels are built from exactly these pieces.
#include <cuda_runtime.h>
#include <stdint.h>
#include "tc05.cuh"

namespace {
using namespace tc05;

// float offset of element (n, k) of an [N x K] K-major operand in the core-matrix tiled layout
__host__ __device__ inline int tiled_off(int n, int k, int K) { return (n >> 3) * (K >> 2) * 32 + (k >> 2) * 32 + (n & 7) * 4 + (k & 3); }

__global__ void __launch_bounds__(128, 1) mma_selftest_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                              float* __restrict__ D, int N, int K, int passes) {
  extern __shared__ __align__(128) float sm[];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x, warp = tid >> 5;
  float* Bhi = sm;
  float* Blo = sm + N * K;

  if (warp == 0) tmem_alloc(&tmem_base_s, 512);
  if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  for (int e = tid; e < N * K; e += 128) {
    const int n = e / K, k = e - n * K;
    uint32_t hi, lo;
    split_tf32(B[e], hi, lo);
    // passes 4 / 5: B stored MN-major (4 consecutive n contiguous, 8 k at 16 B stride, n-groups 128 B apart, k-groups after)
    const int off = passes >= 4 ? (n & 3) + (k & 7) * 4 + (n >> 2) * 32 + (k >> 3) * (N >> 2) * 32 : tiled_off(n, k, K);
    Bhi[off] = __uint_as_float(hi);
    Blo[off] = __uint_as_float(lo);
  }
  // generic-proxy smem writes must be visible to the tensor core (async proxy)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = tmem_base_s;
  const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
  const uint32_t colA_hi = 0, colA_lo = 64, colD = 128;

  // A: thread r owns row r
  for (int k0 = 0; k0 < K; k0 += 8) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) split_tf32(A[tid * K + k0 + j], hi[j], lo[j]);
    tmem_st_x8(tbase + lane_base + colA_hi + k0, hi);
    tmem_st_x8(tbase + lane_base + colA_lo + k0, lo);
  }
  tmem_wait_st();
  fence_before_sync();
  __syncthreads();

  if (tid == 0) {
    fence_after_sync();
    const uint32_t idesc = idesc_tf32(128, N);
    const uint32_t sbo = (uint32_t)(K >> 2) * 128u, lbo = 128u;
    uint32_t acc = 0;
    if (passes >= 4) {
      // MN-major B: passes 4 = (LBO = k-group stride, SBO = n-group stride) as in the CUTLASS canonical form, 5 = swapped
      const uint32_t kg = (uint32_t)(N >> 2) * 128u, ng = 128u;
      for (int j = 0; j < K / 8; ++j) {
        const uint64_t bdesc = smem_desc_kmajor_nosw(smem_u32(Bhi) + (uint32_t)j * kg, passes == 4 ? kg : ng, passes == 4 ? ng : kg);
        mma_tf32_ts(tbase + colD, tbase + colA_hi + 8 * j, bdesc, idesc | (1u << 16), acc);
        acc = 1;
      }
    }
    for (int p = 0; p < (passes >= 4 ? 0 : passes); ++p) {
      const uint32_t a_col = (p == 1) ? colA_lo : colA_hi;
      const float* Bp = (p == 2) ? Blo : Bhi;
      for (int j = 0; j < K / 8; ++j) {
        const uint64_t bdesc = smem_desc_kmajor_nosw(smem_u32(Bp) + (uint32_t)j * 256u, lbo, sbo);
        mma_tf32_ts(tbase + colD, tbase + a_col + 8 * j, bdesc, idesc, acc);
        acc = 1;
      }
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  fence_after_sync();
  for (int n0 = 0; n0 < N; n0 += 16) {
    uint32_t r[16];
    tmem_ld_x16(tbase + lane_base + colD + n0, r);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 16; ++j) D[tid * N + n0 + j] = __uint_as_float(r[j]);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, 512);
}

}  // namespace

cudaError_t rnvp_launch_mma_selftest(const float* A, const float* B, float* D, int N, int K, int passes, cudaStream_t st) {
  const size_t smem = (size_t)2 * N * K * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(mma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  mma_selftest_kernel<<<1, 128, smem, st>>>(A, B, D, N, K, passes);
  return cudaGetLastError();
}
