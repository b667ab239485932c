// Row-tile MLP pieces shared by the FP32 model sweeps (rnvp_cnormal.cu, rnvp_cvae.cu, rnvp_wgan.cu): activations, a
// dense layer over the rows of a shared-memory tile, a whole MLP forward pass, weight and input gradients, a deterministic
// block sum and torch.optim.Adam's per-step coefficients.  Every helper is a whole-block loop over the calling CTA's threads; the caller synchronises.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/rnvp.h"
#include "rnvp_adam.cuh"

namespace {

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

constexpr int MLP_MAX_HIDDEN = 4;

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

RnvpAdamCoef adam_coef(double lr, double b1, double b2, double eps, double wd, int64_t step) {
  const double bc1 = 1.0 - pow(b1, (double)step), bc2 = 1.0 - pow(b2, (double)step);
  return RnvpAdamCoef{(float)wd, (float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)(lr / bc1), (float)sqrt(bc2),
                      (float)eps};
}

}  // namespace
