// Row-tile MLP pieces shared by the FP32 model sweeps (rnvp_cnormal.cu, rnvp_cvae.cu, rnvp_wgan.cu): activations, a
// dense layer over the rows of a shared-memory tile, a whole MLP forward pass, weight and input gradients, a deterministic
// block sum and torch.optim.Adam's per-step coefficients.  Every helper is a whole-block loop over the calling CTA's threads; the caller synchronises.
// It also holds the three models' shared limits, training noise, ordered reduction of per-CTA partials and host-side
// descriptor set-up.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <initializer_list>
#include <string>

#include "../../include/rnvp.h"
#include "rnvp_adam.cuh"
#include "rnvp_philox.cuh"

int rnvp_fail(int code, const char* msg);   // rnvp_api.cu: sets rnvp_last_error()

namespace {

constexpr int MLP_MAX_D = 128, MLP_MAX_CD = 256, MLP_MAX_LAT = 128, MLP_MAX_HIDDEN = 4, MLP_MAX_WIDTH = 512;
constexpr int MLP_MAX_ROWS = 64;                      // rows per CTA tile
constexpr int MLP_SMEM_BUDGET = 96 * 1024;            // per sweep CTA: two CTAs of 256 threads per SM
constexpr int MLP_THREADS = 256, MLP_TAIL_THREADS = 512;

__host__ __device__ inline int odd_ld(int n) { return n | 1; }

__device__ __forceinline__ float act_f(int act, float x) {
  if (act == RNVP_ACT_TANH) return tanhf(x);
  if (act == RNVP_ACT_SIGMOID) return 1.0f / (1.0f + expf(-x));
  return fmaxf(x, 0.0f);
}
// derivative from the activation's OUTPUT y
__device__ __forceinline__ float act_d(int act, float y) {
  if (act == RNVP_ACT_TANH) return fmaf(-y, y, 1.0f);
  if (act == RNVP_ACT_SIGMOID) return y * (1.0f - y);
  return y > 0.0f ? 1.0f : 0.0f;
}

// out[r][i] = act?(b[i] + sum_j in[r][j] W[i][j]) for r < nr, i < no; consecutive threads walk rows (W is warp-uniform)
__device__ __forceinline__ void dense_rows(const float* __restrict__ in, int ldi, int ni, const float* __restrict__ W,
                                  const float* __restrict__ bias, float* out, int ldo, int no, int nr, int act) {
  for (int t = threadIdx.x; t < nr * no; t += blockDim.x) {
    const int i = t / nr, r = t - i * nr;
    const float* x = in + r * ldi;
    const float* w = W + (size_t)i * ni;
    float acc = bias[i];
    for (int j = 0; j < ni; ++j) acc = fmaf(x[j], __ldg(w + j), acc);
    out[r * ldo + i] = act ? act_f(act, acc) : acc;
  }
}

// gW[i][j] = sum_r dA[r][i] in[r][j], gb[i] = sum_r dA[r][i] (rows in order: the sums are deterministic).  ACC adds the
// tile's sums to gW / gb instead (each element is read and written by the same thread as in the call it follows).
template <bool ACC = false>
__device__ __forceinline__ void wgrad(const float* dA, int lda, int no, const float* in, int ldi, int ni, int nr,
                             float* __restrict__ gW, float* __restrict__ gb) {
  for (int t = threadIdx.x; t < no * ni; t += blockDim.x) {
    const int i = t / ni, j = t - i * ni;
    float acc = 0.0f;
    for (int r = 0; r < nr; ++r) acc = fmaf(dA[r * lda + i], in[r * ldi + j], acc);
    gW[t] = ACC ? gW[t] + acc : acc;
  }
  if (gb)
    for (int i = threadIdx.x; i < no; i += blockDim.x) {
      float acc = 0.0f;
      for (int r = 0; r < nr; ++r) acc += dA[r * lda + i];
      gb[i] = ACC ? gb[i] + acc : acc;
    }
}

// dIn[r][j] = (sum_i dA[r][i] W[i][j]) * act'(In[r][j]), written over In (each element reads only itself)
__device__ __forceinline__ void back_rows(const float* dA, int lda, int no, const float* __restrict__ W, float* io, int ldi,
                                 int ni, int nr, int act) {
  for (int t = threadIdx.x; t < nr * ni; t += blockDim.x) {
    const int j = t / nr, r = t - j * nr;
    const float* g = dA + r * lda;
    float acc = 0.0f;
    for (int i = 0; i < no; ++i) acc = fmaf(g[i], __ldg(W + (size_t)i * ni + j), acc);
    io[r * ldi + j] = acc * act_d(act, io[r * ldi + j]);
  }
}

// hidden layers (act) from `in`, then an affine layer or two heads; out2 may be NULL.  Net has nh, h[] and act.
template <class Net>
__device__ __forceinline__ void mlp_forward(const Net& s, const float* __restrict__ params, const float* in, int ldi,
                                            int ni, float* const* hid, const int* ldh, const int* w, const int* b,
                                            int w1, int b1, float* out1, int w2, int b2, float* out2, int ldo, int no,
                                            int nr) {
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {          // unrolled: the per-layer arrays are indexed statically
    if (k >= s.nh) break;
    dense_rows(in, ldi, ni, params + w[k], params + b[k], hid[k], ldh[k], s.h[k], nr, s.act);
    __syncthreads();
    in = hid[k]; ldi = ldh[k]; ni = s.h[k];
  }
  dense_rows(in, ldi, ni, params + w1, params + b1, out1, ldo, no, nr, 0);
  if (out2) dense_rows(in, ldi, ni, params + w2, params + b2, out2, ldo, no, nr, 0);
  __syncthreads();
}

// deterministic block sum of one value per thread (fixed tree); result valid in every thread
__device__ __forceinline__ float block_sum(float v, float* scratch) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[w] = v;
  __syncthreads();
  float s = 0.0f;
  for (int k = 0; k < nw; ++k) s += scratch[k];
  __syncthreads();
  return s;
}

// s[k] = sum of p[k n .. k n + n) for k < K: strided per-thread sums in order (the K sums in one loop, so their loads
// overlap), then the fixed tree of block_sum; valid in every thread
template <int K>
__device__ __forceinline__ void block_sums_strided(const float* __restrict__ p, int64_t n, float* scratch, float* s) {
  float acc[K] = {};
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x)
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] += p[k * n + i];
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = block_sum(acc[k], scratch);
}

// training noise of batch position p, column j of an L-wide row: buf[p * L + j] if given, else Philox keyed on
// (seed, row0 + p, j)
struct MlpNoise {
  const float* buf;
  unsigned long long seed;
  long long row0;
};

__device__ __forceinline__ float noise_at(const MlpNoise& nz, int L, int64_t p, int j) {
  return nz.buf ? nz.buf[p * L + j] : rnvp_rng::normal1(nz.seed, nz.row0 + p, j);
}

// g[c] = sum of the n_ctas partial records (stride floats apart) in CTA order, for the gradient entries c in lo .. hi
// and the n_sums loss or score sums P .. P + n_sums - 1 after them; nothing when *status is set
__global__ void mlp_reduce_kernel(const float* __restrict__ partials, int n_ctas, int stride, int P, int lo, int hi,
                                  int n_sums, float* __restrict__ g, const int* status) {
  if (status && *status) return;
  const int t = blockIdx.x * blockDim.x + threadIdx.x, m = hi - lo;
  if (t >= m + n_sums) return;
  const int c = t < m ? lo + t : P + (t - m);
  float acc = 0.0f;
  for (int b = 0; b < n_ctas; ++b) acc += partials[(size_t)b * stride + c];
  g[c] = acc;
}

void launch_reduce(const float* partials, int n_ctas, int stride, int P, int lo, int hi, int n_sums, float* g,
                   const int* status, cudaStream_t stream) {
  const int n = hi - lo + n_sums;
  mlp_reduce_kernel<<<(n + 255) / 256, 256, 0, stream>>>(partials, n_ctas, stride, P, lo, hi, n_sums, g, status);
}

RnvpAdamCoef adam_coef(double lr, double b1, double b2, double eps, double wd, int64_t step) {
  const double bc1 = 1.0 - pow(b1, (double)step), bc2 = 1.0 - pow(b2, (double)step);
  return RnvpAdamCoef{(float)wd, (float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)(lr / bc1), (float)sqrt(bc2),
                      (float)eps};
}

int64_t n_tiles(int R, int64_t n) { return (n + R - 1) / R; }

// more tiles than a grid's x dimension can hold
bool bad_rows(int R, int64_t n) { return n_tiles(R, n) > 0x7fffffffLL; }

// rows per sweep tile: MLP_MAX_ROWS, halved until tile_floats(s, R) (the model's own) fits MLP_SMEM_BUDGET
template <class Shape>
int rows_per_tile(const Shape& s) {
  int R = MLP_MAX_ROWS;
  while (R > 1 && tile_floats(s, R) * 4 > MLP_SMEM_BUDGET) R >>= 1;
  return R;
}

// the hidden layers of one MLP with nin inputs, in torch's parameters() order: checks each width, then appends its
// weight and bias offsets (h[k], w[k], b[k]) at off
int hidden_layout(int nh, const int* hidden, int nin, int* h, int* w, int* b, int64_t& off, const char* model,
                  const char* fn) {
  for (int k = 0; k < nh; ++k) {
    if (hidden[k] < 1) return rnvp_fail(RNVP_EINVAL, (std::string(fn) + ": hidden widths must be >= 1").c_str());
    if (hidden[k] > MLP_MAX_WIDTH)
      return rnvp_fail(RNVP_ESHAPE, (std::string(model) + ": hidden widths must be <= 512").c_str());
    h[k] = hidden[k];
    w[k] = (int)off; off += (int64_t)hidden[k] * nin;
    b[k] = (int)off; off += hidden[k];
    nin = hidden[k];
  }
  return 0;
}

// one linear layer, nin to nout: its weight and bias offsets at off
void linear_layout(int& w, int& b, int nin, int nout, int64_t& off) {
  w = (int)off; off += (int64_t)nout * nin;
  b = (int)off; off += nout;
}

// Lets each kernel take `need` bytes of dynamic shared memory.  The limit is a property of the kernel on this device,
// shared by every descriptor: set it to the device's opt-in maximum less the kernel's static shared memory
// (idempotent), never to this shape's need, which would lower it under a larger model created earlier.
int opt_in_smem(std::initializer_list<const void*> kernels, int need, const char* model, const char* fn) {
  int dev = 0, max_optin = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (e != cudaSuccess) return rnvp_fail(RNVP_ENODEVICE, (std::string(fn) + ": no CUDA device").c_str());
  const std::string too_big = std::string(model) + ": shape exceeds the shared memory of one CTA";
  if (need > max_optin) return rnvp_fail(RNVP_ESHAPE, too_big.c_str());
  for (const void* k : kernels) {
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, k);
    const int dyn_max = max_optin - (int)fa.sharedSizeBytes;
    if (e == cudaSuccess && need > dyn_max) return rnvp_fail(RNVP_ESHAPE, too_big.c_str());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_max);
    if (e != cudaSuccess) {
      cudaGetLastError();                             // do not leave the error for the caller's next call
      return rnvp_fail((int)e, (std::string(fn) + ": cudaFuncSetAttribute").c_str());
    }
  }
  return 0;
}

// 0 if the kernels just enqueued launched, else their error, reported as `what`
int launched(const char* what) {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : rnvp_fail((int)e, what);
}

}  // namespace
