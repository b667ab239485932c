// CVAE (reference probaforms/models/cvae.py): an encoder MLP from [x|c] to the heads mu and log_sigma of a Gaussian
// posterior over the latent z, z = mu + exp(log_sigma / 2) eps, and a decoder MLP from [z|c] back to x, trained on
// mean((x - x_rec)^2) + KL_weight * mean_rows(-1/2 sum_j (1 + log_sigma - mu^2 - exp(log_sigma))).  FP32 FMA throughout.
//
// A CTA owns a tile of up to R rows of a step's batch and keeps every activation of the tile in shared memory (row-major
// with an odd row stride, as in rnvp_cnormal.cu): [x|c], the encoder's hidden layers, mu, log_sigma, exp(ls/2) eps,
// [z|c], the decoder's hidden layers and x_rec.  The fit sweep runs the encoder, the reparameterisation, the decoder,
// the loss, the decoder's backward pass down to dz (no gradient for the c columns, no activation derivative on the
// linear input), dmu / dls, and the encoder's backward pass, and writes per-CTA partial sums of every weight gradient
// plus the loss.  mlp_reduce_kernel adds the partials in CTA order and cv_tail_kernel runs Adam, so repeated fits are
// bitwise identical.  A batch of at most R rows is one launch (cv_step_kernel).  The same sweep without the backward
// pass gives the loss alone (per-CTA partials, then cv_loss_reduce_kernel in a fixed order).
//
// eps is either a caller buffer indexed by batch position, or Philox keyed on (seed, row base + batch position, j).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "../../include/rnvp.h"
#include "rnvp_adam.cuh"
#include "rnvp_mlp.cuh"

namespace {

struct CvShape {
  int D, Cd, L, nh, act, R;
  int h[MLP_MAX_HIDDEN];
  int ew[MLP_MAX_HIDDEN], eb[MLP_MAX_HIDDEN];         // float offsets of encoder.model.{2k}.weight / .bias
  int mu_w, mu_b, ls_w, ls_b;                         // encoder.mu, encoder.log_sigma
  int dw[MLP_MAX_HIDDEN], db[MLP_MAX_HIDDEN];         // decoder.model.{2k}.weight / .bias
  int out_w, out_b, P;                                // decoder.model.{2 nh}
  int stride;                                         // floats of one CTA's partial record (P gradients + loss)
  int smem;
};

// shared-memory layout of one tile: XC | EH_0 .. EH_{nh-1} | MU | LS | EP | ZC | DH_0 .. DH_{nh-1} | XR, each
// [R][odd stride]; EP holds exp(ls / 2) eps once the latent is drawn
struct CvTile {
  float *xc, *eh[MLP_MAX_HIDDEN], *mu, *ls, *ep, *zc, *dh[MLP_MAX_HIDDEN], *xr;
  int ldxc, ldh[MLP_MAX_HIDDEN], ldl, ldz, ldx;
};

__host__ __device__ inline int tile_floats(const CvShape& s, int R) {
  int f = R * (odd_ld(s.D + s.Cd) + 3 * odd_ld(s.L) + odd_ld(s.L + s.Cd) + odd_ld(s.D));
  for (int k = 0; k < s.nh; ++k) f += 2 * R * odd_ld(s.h[k]);
  return f + 64;                                      // + the block reduction scratch
}

__device__ __forceinline__ CvTile carve(const CvShape& s, float* sm) {
  CvTile t;
  const int R = s.R;
  t.ldxc = odd_ld(s.D + s.Cd);
  t.xc = sm; sm += R * t.ldxc;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {
    t.ldh[k] = k < s.nh ? odd_ld(s.h[k]) : 0;
    t.eh[k] = sm;
    sm += R * t.ldh[k];
  }
  t.ldl = odd_ld(s.L);
  t.mu = sm; sm += R * t.ldl;
  t.ls = sm; sm += R * t.ldl;
  t.ep = sm; sm += R * t.ldl;
  t.ldz = odd_ld(s.L + s.Cd);
  t.zc = sm; sm += R * t.ldz;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {
    t.dh[k] = sm;
    sm += R * t.ldh[k];
  }
  t.ldx = odd_ld(s.D);
  t.xr = sm;
  return t;
}

// [x|c] rows X[idx[r]], C[idx[r]] into XC (and c into the tail of ZC)
__device__ __forceinline__ void load_xc(const CvShape& s, const CvTile& t, const float* __restrict__ X,
                                        const float* __restrict__ C, const int64_t* __restrict__ idx, int64_t row0,
                                        int nr) {
  const int D = s.D, Cd = s.Cd, W = D + Cd;
  for (int e = threadIdx.x; e < nr * W; e += blockDim.x) {
    const int r = e / W, j = e - r * W;
    const int64_t row = idx ? idx[row0 + r] : row0 + r;
    float v;
    if (j < D) {
      v = X[row * D + j];
    } else {
      v = C[row * Cd + (j - D)];
      t.zc[r * t.ldz + s.L + (j - D)] = v;
    }
    t.xc[r * t.ldxc + j] = v;
  }
}

// forward, loss and (with g) backward of one tile of batch positions row0 .. row0 + nr; the tile's loss sum goes to
// *loss_dst and, with g, its gradient partials to g[0..P)
__device__ __forceinline__ void sweep_tile(const CvShape& s, float* sm, const float* __restrict__ params,
                                           const float* __restrict__ X, const float* __restrict__ C,
                                           const int64_t* __restrict__ idx, int64_t row0, int nr, const MlpNoise& nz,
                                           float inv_bd, float kl_b, float* __restrict__ g, float* loss_dst) {
  const CvTile t = carve(s, sm);
  float* scratch = t.xr + s.R * t.ldx;                 // the 64 floats after the tile (tile_floats)
  const int D = s.D, Cd = s.Cd, L = s.L;
  load_xc(s, t, X, C, idx, row0, nr);
  for (int e = threadIdx.x; e < nr * L; e += blockDim.x) {
    const int r = e / L, j = e - r * L;
    t.ep[r * t.ldl + j] = noise_at(nz, L, row0 + r, j);
  }
  __syncthreads();
  mlp_forward(s, params, t.xc, t.ldxc, D + Cd, t.eh, t.ldh, s.ew, s.eb, s.mu_w, s.mu_b, t.mu, s.ls_w, s.ls_b, t.ls,
              t.ldl, L, nr);
  for (int e = threadIdx.x; e < nr * L; e += blockDim.x) {   // z = mu + exp(ls / 2) eps (sample_z)
    const int r = e / L, j = e - r * L, o = r * t.ldl + j;
    const float se = expf(0.5f * t.ls[o]) * t.ep[o];
    t.ep[o] = se;
    t.zc[r * t.ldz + j] = t.mu[o] + se;
  }
  __syncthreads();
  mlp_forward(s, params, t.zc, t.ldz, L + Cd, t.dh, t.ldh, s.dw, s.db, s.out_w, s.out_b, t.xr, 0, 0, nullptr, t.ldx, D,
              nr);
  float rec = 0.0f, kl = 0.0f;
  for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
    const int r = e / D, j = e - r * D, o = r * t.ldx + j;
    const float d = t.xr[o] - t.xc[r * t.ldxc + j];
    rec = fmaf(d, d, rec);
    if (g) t.xr[o] = 2.0f * d * inv_bd;                // d loss / d x_rec
  }
  for (int e = threadIdx.x; e < nr * L; e += blockDim.x) {
    const int r = e / L, j = e - r * L, o = r * t.ldl + j;
    const float mu = t.mu[o], ls = t.ls[o];
    kl += 1.0f + ls - mu * mu - expf(ls);
  }
  const float tot = block_sum(fmaf(rec, inv_bd, -0.5f * kl_b * kl), scratch);
  if (threadIdx.x == 0) *loss_dst = tot;
  if (!g) return;

  // decoder: output layer, hidden layers, then dz (the c columns of [z|c] need no gradient)
  int hl = 0, ldl = 0;
  float *DHl = nullptr, *EHl = nullptr;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k)
    if (k == s.nh - 1) { hl = s.h[k]; DHl = t.dh[k]; EHl = t.eh[k]; ldl = t.ldh[k]; }
  wgrad(t.xr, t.ldx, D, DHl, ldl, hl, nr, g + s.out_w, g + s.out_b);
  __syncthreads();
  back_rows(t.xr, t.ldx, D, params + s.out_w, DHl, ldl, hl, nr, s.act);
  __syncthreads();
#pragma unroll
  for (int k = MLP_MAX_HIDDEN - 1; k >= 0; --k) {
    if (k >= s.nh) continue;
    const float* in = k ? t.dh[k - 1] : t.zc;
    const int ldi = k ? t.ldh[k - 1] : t.ldz, ni = k ? s.h[k - 1] : L + Cd;
    wgrad(t.dh[k], t.ldh[k], s.h[k], in, ldi, ni, nr, g + s.dw[k], g + s.db[k]);
    __syncthreads();
    if (k) {
      back_rows(t.dh[k], t.ldh[k], s.h[k], params + s.dw[k], t.dh[k - 1], t.ldh[k - 1], ni, nr, s.act);
      __syncthreads();
    }
  }
  // dz, then dmu = dz + KLw mu / nb and dls = dz exp(ls / 2) eps / 2 + KLw (exp(ls) - 1) / (2 nb), over MU and LS
  {
    const int h0 = s.h[0], ld0 = t.ldh[0], nz_in = L + Cd;
    const float* W0 = params + s.dw[0];
    for (int e = threadIdx.x; e < nr * L; e += blockDim.x) {
      const int j = e / nr, r = e - j * nr;
      const float* gr = t.dh[0] + r * ld0;
      float acc = 0.0f;
      for (int i = 0; i < h0; ++i) acc = fmaf(gr[i], __ldg(W0 + (size_t)i * nz_in + j), acc);
      const int o = r * t.ldl + j;
      const float mu = t.mu[o], ls = t.ls[o];
      t.mu[o] = fmaf(kl_b, mu, acc);
      t.ls[o] = 0.5f * fmaf(acc, t.ep[o], kl_b * (expf(ls) - 1.0f));
    }
  }
  __syncthreads();
  // encoder: both heads, then the hidden layers (no gradient for [x|c])
  wgrad(t.mu, t.ldl, L, EHl, ldl, hl, nr, g + s.mu_w, g + s.mu_b);
  wgrad(t.ls, t.ldl, L, EHl, ldl, hl, nr, g + s.ls_w, g + s.ls_b);
  __syncthreads();
  for (int e = threadIdx.x; e < nr * hl; e += blockDim.x) {
    const int j = e / nr, r = e - j * nr;
    const float *gm = t.mu + r * t.ldl, *gl = t.ls + r * t.ldl;
    float acc = 0.0f;
    for (int i = 0; i < L; ++i)
      acc = fmaf(gm[i], __ldg(params + s.mu_w + (size_t)i * hl + j), fmaf(gl[i], __ldg(params + s.ls_w + (size_t)i * hl + j), acc));
    EHl[r * ldl + j] = acc * act_d(s.act, EHl[r * ldl + j]);
  }
  __syncthreads();
#pragma unroll
  for (int k = MLP_MAX_HIDDEN - 1; k >= 0; --k) {
    if (k >= s.nh) continue;
    const float* in = k ? t.eh[k - 1] : t.xc;
    const int ldi = k ? t.ldh[k - 1] : t.ldxc, ni = k ? s.h[k - 1] : D + Cd;
    wgrad(t.eh[k], t.ldh[k], s.h[k], in, ldi, ni, nr, g + s.ew[k], g + s.eb[k]);
    __syncthreads();
    if (k) {
      back_rows(t.eh[k], t.ldh[k], s.h[k], params + s.ew[k], t.eh[k - 1], t.ldh[k - 1], ni, nr, s.act);
      __syncthreads();
    }
  }
}

struct CvStep {
  RnvpAdamCoef k;
  float inv_bd, kl_b;                                 // 1 / (nb D), KL_weight / nb
  int adam;                                           // 0: gradient only (rnvp_cv_grad)
};

// the whole batch's gradient g (reduced, P + 1 floats): loss hand-off, then Adam or a copy to gflat
__device__ __forceinline__ void cv_tail(const CvShape& s, float* __restrict__ params, float* __restrict__ m,
                                        float* __restrict__ v, const float* g, float* __restrict__ gflat,
                                        float* loss_dst, const CvStep& st) {
  if (threadIdx.x == 0 && loss_dst) *loss_dst = g[s.P];
  if (!st.adam) {
    for (int i = threadIdx.x; i < s.P; i += blockDim.x) gflat[i] = g[i];
    return;
  }
  for (int i = threadIdx.x; i < s.P; i += blockDim.x) {
    float mi = m[i], vi = v[i];
    params[i] = rnvp_adam_update(g[i], params[i], mi, vi, st.k);
    m[i] = mi; v[i] = vi;
  }
}

// with bwd: gradient partials + loss per CTA at partials + b * stride; without: the loss sum alone at partials[b]
__global__ void __launch_bounds__(MLP_THREADS) cv_sweep_kernel(CvShape s, const float* __restrict__ params,
    const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx, int64_t nb, MlpNoise nz,
    float inv_bd, float kl_b, float* __restrict__ partials, int bwd) {
  extern __shared__ __align__(16) float smem[];
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(nb - row0 < s.R ? nb - row0 : s.R);
  float* g = bwd ? partials + (size_t)blockIdx.x * s.stride : nullptr;
  sweep_tile(s, smem, params, X, C, idx, row0, nr, nz, inv_bd, kl_b, g, bwd ? g + s.P : partials + blockIdx.x);
}

// *dst = sum of n loss partials: strided per-thread sums in order, then the fixed block tree
__global__ void __launch_bounds__(MLP_THREADS) cv_loss_reduce_kernel(const float* __restrict__ partials, int64_t n,
                                                                    float* dst) {
  __shared__ float scratch[32];
  float tot;
  block_sums_strided<1>(partials, n, scratch, &tot);
  if (threadIdx.x == 0) *dst = tot;
}

__global__ void __launch_bounds__(MLP_TAIL_THREADS) cv_tail_kernel(CvShape s, float* params, float* m, float* v,
                                                                 const float* g, float* gflat, float* loss_dst,
                                                                 CvStep st) {
  cv_tail(s, params, m, v, g, gflat, loss_dst, st);
}

// a whole step of a batch that fits one tile
__global__ void __launch_bounds__(MLP_TAIL_THREADS) cv_step_kernel(CvShape s, float* params, float* m, float* v,
    const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx, int nb, MlpNoise nz,
    float* g, float* gflat, float* loss_dst, CvStep st) {
  extern __shared__ __align__(16) float smem[];
  sweep_tile(s, smem, params, X, C, idx, 0, nb, nz, st.inv_bd, st.kl_b, g, g + s.P);
  __syncthreads();                                     // g (global) is read back by other threads of this CTA
  cv_tail(s, params, m, v, g, gflat, loss_dst, st);
}

// Encoder.forward for inference: mu, log_sigma of rows [X|C]
__global__ void __launch_bounds__(MLP_THREADS) cv_encode_kernel(CvShape s, const float* __restrict__ params,
    const float* __restrict__ X, const float* __restrict__ C, int64_t N, float* mu_o, float* ls_o) {
  extern __shared__ __align__(16) float smem[];
  const CvTile t = carve(s, smem);
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(N - row0 < s.R ? N - row0 : s.R);
  load_xc(s, t, X, C, nullptr, row0, nr);
  __syncthreads();
  mlp_forward(s, params, t.xc, t.ldxc, s.D + s.Cd, t.eh, t.ldh, s.ew, s.eb, s.mu_w, s.mu_b, t.mu, s.ls_w, s.ls_b, t.ls,
              t.ldl, s.L, nr);
  const int L = s.L;
  for (int e = threadIdx.x; e < nr * L; e += blockDim.x) {
    const int r = e / L, j = e - r * L, o = r * t.ldl + j;
    mu_o[(row0 + r) * L + j] = t.mu[o];
    ls_o[(row0 + r) * L + j] = t.ls[o];
  }
}

// Decoder.forward for inference: x of rows [z|C], z from Z or from Philox keyed on (seed, row_offset + row, j)
__global__ void __launch_bounds__(MLP_THREADS) cv_decode_kernel(CvShape s, const float* __restrict__ params,
    const float* __restrict__ Z, const float* __restrict__ C, int64_t N, unsigned long long seed, long long row_offset,
    float* x_o) {
  extern __shared__ __align__(16) float smem[];
  const CvTile t = carve(s, smem);
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(N - row0 < s.R ? N - row0 : s.R);
  const int L = s.L, Cd = s.Cd, W = L + Cd;
  const MlpNoise nz{Z, seed, row_offset};
  for (int e = threadIdx.x; e < nr * W; e += blockDim.x) {
    const int r = e / W, j = e - r * W;
    const int64_t row = row0 + r;
    t.zc[r * t.ldz + j] = j < L ? noise_at(nz, L, row, j) : C[row * Cd + (j - L)];
  }
  __syncthreads();
  mlp_forward(s, params, t.zc, t.ldz, W, t.dh, t.ldh, s.dw, s.db, s.out_w, s.out_b, t.xr, 0, 0, nullptr, t.ldx, s.D,
              nr);
  const int D = s.D;
  for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
    const int r = e / D, j = e - r * D;
    x_o[(row0 + r) * D + j] = t.xr[r * t.ldx + j];
  }
}

}  // namespace

struct rnvp_cv_desc {
  CvShape s;
};

namespace {

int check_cv(const rnvp_cv_desc* d) { return d ? 0 : rnvp_fail(RNVP_EINVAL, "null CVAE descriptor"); }

// the gradient (gflat, with m == NULL) or the Adam step of one batch of nb positions of idx
void launch_step(const CvShape& s, float* params, float* m, float* v, const float* X, const float* C,
                 const int64_t* idx, int64_t nb, const MlpNoise& nz, float* gflat, float* loss_dst, const CvStep& st,
                 float* ws, cudaStream_t stream) {
  const int64_t nt = n_tiles(s.R, nb);
  float* g = ws;                                       // reduced gradient + loss (stride floats), then the partials
  if (nt == 1) {
    cv_step_kernel<<<1, MLP_TAIL_THREADS, s.smem, stream>>>(s, params, m, v, X, C, idx, (int)nb, nz, g, gflat, loss_dst,
                                                           st);
    return;
  }
  float* partials = ws + s.stride;
  cv_sweep_kernel<<<(unsigned)nt, MLP_THREADS, s.smem, stream>>>(s, params, X, C, idx, nb, nz, st.inv_bd, st.kl_b,
                                                                partials, 1);
  launch_reduce(partials, (int)nt, s.stride, s.P, 0, s.P, 1, g, nullptr, stream);
  cv_tail_kernel<<<1, MLP_TAIL_THREADS, 0, stream>>>(s, params, m, v, g, gflat, loss_dst, st);
}

// the loss alone over N positions of idx into *loss_dst
void launch_loss(const CvShape& s, const float* params, const float* X, const float* C, const int64_t* idx, int64_t N,
                 const MlpNoise& nz, float kl_weight, float* loss_dst, float* ws, cudaStream_t stream) {
  const int64_t nt = n_tiles(s.R, N);
  const float inv_bd = (float)(1.0 / ((double)N * s.D)), kl_b = (float)((double)kl_weight / (double)N);
  cv_sweep_kernel<<<(unsigned)nt, MLP_THREADS, s.smem, stream>>>(s, params, X, C, idx, N, nz, inv_bd, kl_b,
                                                                nt == 1 ? loss_dst : ws, 0);
  if (nt > 1) cv_loss_reduce_kernel<<<1, MLP_THREADS, 0, stream>>>(ws, nt, loss_dst);
}

}  // namespace

extern "C" {

int rnvp_cv_desc_create(int D, int Cd, int latent, int n_hidden, const int* hidden, int act, rnvp_cv_desc** out) {
  if (!out) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_desc_create: out is null");
  *out = nullptr;
  if (!hidden || D < 1 || Cd < 0 || latent < 1 || n_hidden < 1)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_desc_create: bad shape");
  if (act != RNVP_ACT_TANH && act != RNVP_ACT_RELU)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_desc_create: act must be RNVP_ACT_TANH or _RELU");
  if (D > MLP_MAX_D) return rnvp_fail(RNVP_ESHAPE, "CVAE: var_size D must be <= 128");
  if (Cd > MLP_MAX_CD) return rnvp_fail(RNVP_ESHAPE, "CVAE: cond_size must be <= 256");
  if (latent > MLP_MAX_LAT) return rnvp_fail(RNVP_ESHAPE, "CVAE: latent_dim must be <= 128");
  if (n_hidden > MLP_MAX_HIDDEN) return rnvp_fail(RNVP_ESHAPE, "CVAE: at most 4 hidden layers");
  CvShape s{};
  s.D = D; s.Cd = Cd; s.L = latent; s.nh = n_hidden; s.act = act;
  int64_t off = 0;
  const int hl = hidden[n_hidden - 1];
  // encoder.parameters(), then decoder.parameters()
  if (int rc = hidden_layout(n_hidden, hidden, D + Cd, s.h, s.ew, s.eb, off, "CVAE", "rnvp_cv_desc_create")) return rc;
  linear_layout(s.mu_w, s.mu_b, hl, latent, off);
  linear_layout(s.ls_w, s.ls_b, hl, latent, off);
  hidden_layout(n_hidden, hidden, latent + Cd, s.h, s.dw, s.db, off, "CVAE", "rnvp_cv_desc_create");   // checked above
  linear_layout(s.out_w, s.out_b, hl, D, off);
  s.P = (int)off;
  s.stride = (s.P + 1 + 3) & ~3;
  s.R = rows_per_tile(s);
  s.smem = tile_floats(s, s.R) * 4;
  if (int rc = opt_in_smem({(const void*)cv_sweep_kernel, (const void*)cv_step_kernel, (const void*)cv_encode_kernel,
                            (const void*)cv_decode_kernel},
                           s.smem, "CVAE", "rnvp_cv_desc_create"))
    return rc;
  *out = new rnvp_cv_desc{s};
  return 0;
}

void rnvp_cv_desc_destroy(rnvp_cv_desc* d) { delete d; }

int64_t rnvp_cv_param_count(const rnvp_cv_desc* d) { return d ? d->s.P : -1; }

int64_t rnvp_cv_workspace_bytes(const rnvp_cv_desc* d, int64_t batch_rows, int64_t loss_rows) {
  if (!d || batch_rows < 0 || loss_rows < 0) return -1;
  const int64_t nt = n_tiles(d->s.R, batch_rows);
  return 4 * std::max((int64_t)d->s.stride * (1 + (nt > 1 ? nt : 0)), n_tiles(d->s.R, loss_rows));
}

int rnvp_cv_encode(const rnvp_cv_desc* d, const float* d_params, const float* d_X, const float* d_C, int64_t N,
                   float* d_mu, float* d_log_sigma, void* stream) {
  if (check_cv(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || (d->s.Cd && !d_C) || !d_mu || !d_log_sigma || N < 0)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_encode: bad argument");
  if (N == 0) return 0;
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_encode: too many rows");
  cv_encode_kernel<<<(unsigned)n_tiles(d->s.R, N), MLP_THREADS, d->s.smem, (cudaStream_t)stream>>>(
      d->s, d_params, d_X, d_C, N, d_mu, d_log_sigma);
  return launched("cv_encode_kernel launch");
}

int rnvp_cv_decode(const rnvp_cv_desc* d, const float* d_params, const float* d_Z, const float* d_C, int64_t N,
                   uint64_t seed, int64_t row_offset, float* d_x, void* stream) {
  if (check_cv(d)) return RNVP_EINVAL;
  if (!d_params || (d->s.Cd && !d_C) || !d_x || N < 0) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_decode: bad argument");
  if (N == 0) return 0;
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_decode: too many rows");
  cv_decode_kernel<<<(unsigned)n_tiles(d->s.R, N), MLP_THREADS, d->s.smem, (cudaStream_t)stream>>>(
      d->s, d_params, d_Z, d_C, N, seed, row_offset, d_x);
  return launched("cv_decode_kernel launch");
}

int rnvp_cv_grad(const rnvp_cv_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_eps, int64_t N, double kl_weight, float* d_gflat, float* d_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_cv(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || (d->s.Cd && !d_C) || !d_eps || !d_gflat || N < 1)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_grad: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_cv_workspace_bytes(d, N, 0))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_grad: workspace smaller than rnvp_cv_workspace_bytes(N, 0)");
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_grad: too many rows");
  CvStep st{};
  st.inv_bd = (float)(1.0 / ((double)N * d->s.D));
  st.kl_b = (float)(kl_weight / (double)N);
  st.adam = 0;
  launch_step(d->s, const_cast<float*>(d_params), nullptr, nullptr, d_X, d_C, d_idx, N, MlpNoise{d_eps, 0, 0}, d_gflat,
              d_loss, st, (float*)d_workspace, (cudaStream_t)stream);
  return launched("CVAE gradient launch");
}

int rnvp_cv_loss(const rnvp_cv_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_eps, int64_t N, double kl_weight, float* d_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_cv(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || (d->s.Cd && !d_C) || !d_eps || !d_loss || N < 1)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_loss: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_cv_workspace_bytes(d, 0, N))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_loss: workspace smaller than rnvp_cv_workspace_bytes(0, N)");
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_loss: too many rows");
  launch_loss(d->s, d_params, d_X, d_C, d_idx, N, MlpNoise{d_eps, 0, 0}, (float)kl_weight, d_loss, (float*)d_workspace,
              (cudaStream_t)stream);
  return launched("CVAE loss launch");
}

int rnvp_cv_fit_epoch(const rnvp_cv_desc* d, float* d_params, float* d_exp_avg, float* d_exp_avg_sq, const float* d_X,
                      const float* d_C, const int64_t* d_perm, int64_t n, int64_t batch_size, double lr, double beta1,
                      double beta2, double eps, double weight_decay, double kl_weight, int64_t step0,
                      const float* d_noise, uint64_t seed, float* d_loss, void* d_workspace, int64_t workspace_bytes,
                      void* stream) {
  if (check_cv(d)) return RNVP_EINVAL;
  if (!d_params || !d_exp_avg || !d_exp_avg_sq || !d_X || (d->s.Cd && !d_C) || !d_perm || !d_loss || n < 1 ||
      batch_size < 1 || step0 < 0)
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_fit_epoch: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_cv_workspace_bytes(d, std::min(n, batch_size), n))
    return rnvp_fail(RNVP_EINVAL, "rnvp_cv_fit_epoch: workspace smaller than rnvp_cv_workspace_bytes(batch_size, n)");
  if (bad_rows(d->s.R, n)) return rnvp_fail(RNVP_EINVAL, "rnvp_cv_fit_epoch: too many rows");
  const CvShape& s = d->s;
  const cudaStream_t st_ = (cudaStream_t)stream;
  int64_t k = 0;
  for (int64_t b0 = 0; b0 < n; b0 += batch_size, ++k) {
    const int64_t nb = std::min(batch_size, n - b0);
    CvStep st{};
    st.k = adam_coef(lr, beta1, beta2, eps, weight_decay, step0 + k + 1);
    st.inv_bd = (float)(1.0 / ((double)nb * s.D));
    st.kl_b = (float)(kl_weight / (double)nb);
    st.adam = 1;
    const MlpNoise nz{d_noise ? d_noise + b0 * s.L : nullptr, seed, (long long)b0};
    launch_step(s, d_params, d_exp_avg, d_exp_avg_sq, d_X, d_C, d_perm + b0, nb, nz, nullptr, nullptr, st,
                (float*)d_workspace, st_);
    if (int rc = launched("CVAE fit step launch")) return rc;
  }
  // compute_loss(X_real, C): every row in dataset order, with its own noise (rows n .. 2n - 1 of the Philox stream)
  const MlpNoise nz{d_noise ? d_noise + n * s.L : nullptr, seed, (long long)n};
  launch_loss(s, d_params, d_X, d_C, nullptr, n, nz, (float)kl_weight, d_loss, (float*)d_workspace, st_);
  return launched("CVAE epoch loss launch");
}

}  // extern "C"
