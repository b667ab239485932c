// ConditionalWGAN (reference probaforms/models/wgan.py): a generator MLP from [z|c] to x and a critic MLP from [x|c] to
// one score, trained alternately: generator steps on -mean(D([G([z|c])|c])) and critic steps on
// -mean(D([x|c])) + mean(D([G([z|c])|c])), each followed by torch.optim.RMSprop on its own net, and the critic's
// parameters clamped to [-clip, clip] after its steps.  FP32 FMA throughout.
//
// A CTA owns a tile of up to R rows of a step's batch and keeps every activation of the tile in shared memory
// (row-major with an odd row stride, as in rnvp_cvae.cu): [z|c], the generator's hidden layers, the fake rows
// [G(z|c)|c], the real rows [x|c], the critic's hidden layers and its scores.  A critic step runs the generator forward,
// then the critic forward and backward on the real rows and writes their weight-gradient sums, then the same on the fake
// rows, adding their sums (wgrad<true>).  Real and fake rows are summed separately, in the same row order, so the
// critic's output-bias gradient sum_real(-1/nb) + sum_fake(+1/nb) is exactly 0 for every nb, as in the reference; an
// interleaved sum would leave rounding noise there that RMSprop turns into steps of up to ~lr.  A generator step runs
// the critic backward down to the x columns of the fake rows (no weight gradients, nothing into c) and then the
// generator backward.  Per-CTA partial records hold the stepped net's gradient and the tile's two score sums;
// mlp_reduce_kernel adds them in CTA order and wg_tail_kernel runs RMSprop (and the clamp), so repeated fits are
// bitwise identical.  A batch of at most R rows is one launch (wg_step_kernel).  The loss pass (the epoch losses) runs
// both forward passes and writes per-CTA score sums, added by wg_loss_reduce_kernel in a fixed order.
//
// z is either a caller buffer indexed by batch position, or Philox keyed on (seed, row base + batch position, j).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "../../include/rnvp.h"
#include "rnvp_mlp.cuh"
#include "rnvp_rmsprop.cuh"

namespace {

// one MLP: hidden layers (act), then a linear output layer of nout columns
struct WgNet {
  int nh, act, nin, nout;
  int h[MLP_MAX_HIDDEN];
  int w[MLP_MAX_HIDDEN], b[MLP_MAX_HIDDEN];           // float offsets of model.{2k}.weight / .bias in the flat buffer
  int ow, ob;                                         // model.{2 nh}
};

struct WgShape {
  int D, Cd, L, R;
  WgNet g, d;                                         // generator (flat offsets 0 .. PG), critic (PG .. P)
  int PG, P;
  int stride;                                         // floats of one CTA's partial record (P gradients + 2 score sums)
  int smem;
};

// shared-memory layout of one tile: ZC | GH_0 .. | XF | XR | DH_0 .. | O, each [R][odd stride] (O: [R])
struct WgTile {
  float *zc, *gh[MLP_MAX_HIDDEN], *xf, *xr, *dh[MLP_MAX_HIDDEN], *o;
  int ldz, ldg[MLP_MAX_HIDDEN], ldx, ldd[MLP_MAX_HIDDEN];
};

__host__ __device__ inline int tile_floats(const WgShape& s, int R) {
  int f = R * (odd_ld(s.L + s.Cd) + 2 * odd_ld(s.D + s.Cd) + 1);
  for (int k = 0; k < s.g.nh; ++k) f += R * odd_ld(s.g.h[k]);
  for (int k = 0; k < s.d.nh; ++k) f += R * odd_ld(s.d.h[k]);
  return f + 64;                                      // + the block reduction scratch
}

__device__ __forceinline__ WgTile carve(const WgShape& s, float* sm) {
  WgTile t;
  const int R = s.R;
  t.ldz = odd_ld(s.L + s.Cd);
  t.zc = sm; sm += R * t.ldz;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {
    t.ldg[k] = k < s.g.nh ? odd_ld(s.g.h[k]) : 0;
    t.gh[k] = sm;
    sm += R * t.ldg[k];
  }
  t.ldx = odd_ld(s.D + s.Cd);
  t.xf = sm; sm += R * t.ldx;
  t.xr = sm; sm += R * t.ldx;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k) {
    t.ldd[k] = k < s.d.nh ? odd_ld(s.d.h[k]) : 0;
    t.dh[k] = sm;
    sm += R * t.ldd[k];
  }
  t.o = sm;
  return t;
}

// ZC = [z|c] of the tile's rows; with real, XR = [x|c]; the c columns of XF too
__device__ __forceinline__ void load_tile(const WgShape& s, const WgTile& t, const float* __restrict__ X,
                                          const float* __restrict__ C, const int64_t* __restrict__ idx, int64_t row0,
                                          int nr, const MlpNoise& nz, bool real) {
  const int D = s.D, Cd = s.Cd, L = s.L;
  for (int e = threadIdx.x; e < nr * L; e += blockDim.x) {
    const int r = e / L, j = e - r * L;
    t.zc[r * t.ldz + j] = noise_at(nz, L, row0 + r, j);
  }
  for (int e = threadIdx.x; e < nr * Cd; e += blockDim.x) {
    const int r = e / Cd, j = e - r * Cd;
    const int64_t row = idx ? idx[row0 + r] : row0 + r;
    const float v = C[row * Cd + j];
    t.zc[r * t.ldz + L + j] = v;
    t.xf[r * t.ldx + D + j] = v;
    t.xr[r * t.ldx + D + j] = v;
  }
  if (real)
    for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
      const int r = e / D, j = e - r * D;
      const int64_t row = idx ? idx[row0 + r] : row0 + r;
      t.xr[r * t.ldx + j] = X[row * D + j];
    }
}

__device__ __forceinline__ void gen_forward(const WgShape& s, const WgTile& t, const float* __restrict__ params, int nr) {
  mlp_forward(s.g, params, t.zc, t.ldz, s.L + s.Cd, t.gh, t.ldg, s.g.w, s.g.b, s.g.ow, s.g.ob, t.xf, 0, 0, nullptr,
              t.ldx, s.D, nr);
}

// the critic's scores of the rows `in` into O; returns (in every thread) their sum over the tile, in row order
__device__ __forceinline__ float critic_forward(const WgShape& s, const WgTile& t, const float* __restrict__ params,
                                                const float* in, int nr, float* scratch) {
  mlp_forward(s.d, params, in, t.ldx, s.D + s.Cd, t.dh, t.ldd, s.d.w, s.d.b, s.d.ow, s.d.ob, t.o, 0, 0, nullptr, 1, 1,
              nr);
  float v = 0.0f;
  if (threadIdx.x == 0)
    for (int r = 0; r < nr; ++r) v += t.o[r];
  return block_sum(v, scratch);
}

// the critic's backward pass from d score = dout on every row, down to its first hidden layer; with g (ACC: added to
// it) the weight gradients of the rows `in`
template <bool ACC>
__device__ __forceinline__ void critic_backward(const WgShape& s, const WgTile& t, const float* __restrict__ params,
                                                const float* in, int nr, float dout, float* __restrict__ g) {
  const WgNet& n = s.d;
  for (int r = threadIdx.x; r < nr; r += blockDim.x) t.o[r] = dout;
  __syncthreads();
  int hl = 0, ldl = 0;
  float* Hl = nullptr;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k)
    if (k == n.nh - 1) { hl = n.h[k]; Hl = t.dh[k]; ldl = t.ldd[k]; }
  if (g) {
    wgrad<ACC>(t.o, 1, 1, Hl, ldl, hl, nr, g + n.ow, g + n.ob);
    __syncthreads();
  }
  back_rows(t.o, 1, 1, params + n.ow, Hl, ldl, hl, nr, n.act);
  __syncthreads();
#pragma unroll
  for (int k = MLP_MAX_HIDDEN - 1; k >= 0; --k) {
    if (k >= n.nh) continue;
    const float* x = k ? t.dh[k - 1] : in;
    const int ldi = k ? t.ldd[k - 1] : t.ldx, ni = k ? n.h[k - 1] : s.D + s.Cd;
    if (g) {
      wgrad<ACC>(t.dh[k], t.ldd[k], n.h[k], x, ldi, ni, nr, g + n.w[k], g + n.b[k]);
      __syncthreads();
    }
    if (k) {
      back_rows(t.dh[k], t.ldd[k], n.h[k], params + n.w[k], t.dh[k - 1], t.ldd[k - 1], ni, nr, n.act);
      __syncthreads();
    }
  }
}

enum { WG_LOSS = 0, WG_CRITIC = 1, WG_GENERATOR = 2 };

// one tile of batch positions row0 .. row0 + nr: forward passes and, for a step, the backward pass of its net into
// g[0..P) (the other net's entries are not written); the tile's fake and real score sums go to sums[0], sums[1]
__device__ __forceinline__ void sweep_tile(const WgShape& s, float* sm, const float* __restrict__ params,
                                           const float* __restrict__ X, const float* __restrict__ C,
                                           const int64_t* __restrict__ idx, int64_t row0, int nr, const MlpNoise& nz,
                                           float inv_nb, int kind, float* __restrict__ g, float* sums) {
  const WgTile t = carve(s, sm);
  float* scratch = t.o + s.R;                          // the 64 floats after the tile (tile_floats)
  load_tile(s, t, X, C, idx, row0, nr, nz, kind != WG_GENERATOR);
  __syncthreads();
  gen_forward(s, t, params, nr);
  float sr = 0.0f, sf;
  if (kind != WG_GENERATOR) {
    sr = critic_forward(s, t, params, t.xr, nr, scratch);
    if (kind == WG_CRITIC) critic_backward<false>(s, t, params, t.xr, nr, -inv_nb, g);
  }
  sf = critic_forward(s, t, params, t.xf, nr, scratch);
  if (threadIdx.x == 0) { sums[0] = sf; sums[1] = sr; }
  if (kind == WG_CRITIC) critic_backward<true>(s, t, params, t.xf, nr, inv_nb, g);
  if (kind != WG_GENERATOR) return;

  critic_backward<false>(s, t, params, t.xf, nr, -inv_nb, nullptr);
  // d x_fake: the x columns of the critic's first layer (no gradient for c; the generator's output is linear)
  {
    const int h0 = s.d.h[0], ld0 = t.ldd[0], ni = s.D + s.Cd;
    const float* W0 = params + s.d.w[0];
    for (int e = threadIdx.x; e < nr * s.D; e += blockDim.x) {
      const int j = e / nr, r = e - j * nr;
      const float* gr = t.dh[0] + r * ld0;
      float acc = 0.0f;
      for (int i = 0; i < h0; ++i) acc = fmaf(gr[i], __ldg(W0 + (size_t)i * ni + j), acc);
      t.xf[r * t.ldx + j] = acc;
    }
  }
  __syncthreads();
  const WgNet& n = s.g;
  int hl = 0, ldl = 0;
  float* Hl = nullptr;
#pragma unroll
  for (int k = 0; k < MLP_MAX_HIDDEN; ++k)
    if (k == n.nh - 1) { hl = n.h[k]; Hl = t.gh[k]; ldl = t.ldg[k]; }
  wgrad(t.xf, t.ldx, s.D, Hl, ldl, hl, nr, g + n.ow, g + n.ob);
  __syncthreads();
  back_rows(t.xf, t.ldx, s.D, params + n.ow, Hl, ldl, hl, nr, n.act);
  __syncthreads();
#pragma unroll
  for (int k = MLP_MAX_HIDDEN - 1; k >= 0; --k) {
    if (k >= n.nh) continue;
    const float* x = k ? t.gh[k - 1] : t.zc;
    const int ldi = k ? t.ldg[k - 1] : t.ldz, ni = k ? n.h[k - 1] : s.L + s.Cd;
    wgrad(t.gh[k], t.ldg[k], n.h[k], x, ldi, ni, nr, g + n.w[k], g + n.b[k]);
    __syncthreads();
    if (k) {
      back_rows(t.gh[k], t.ldg[k], n.h[k], params + n.w[k], t.gh[k - 1], t.ldg[k - 1], ni, nr, n.act);
      __syncthreads();
    }
  }
}

struct WgStep {
  RnvpRmspropCoef k;
  float nb, inv_nb, clip;                             // clip > 0: clamp the stepped net to [-clip, clip]
  int kind, lo, hi;                                   // stepped net: flat entries lo .. hi
  int update;                                         // 0: gradient only (rnvp_wg_grad)
};

// the whole batch's record g (reduced: P gradients, fake and real score sums): the step's loss, then RMSprop (and the
// clamp) on lo .. hi, or the gradient to gflat (zero outside lo .. hi)
__device__ __forceinline__ void wg_tail(const WgShape& s, float* __restrict__ params, float* __restrict__ sq,
                                        const float* g, float* __restrict__ gflat, float* loss_dst, const WgStep& st) {
  if (threadIdx.x == 0 && loss_dst) {
    const float mf = g[s.P] / st.nb;
    *loss_dst = st.kind == WG_CRITIC ? -(g[s.P + 1] / st.nb) + mf : -mf;
  }
  if (!st.update) {
    for (int i = threadIdx.x; i < s.P; i += blockDim.x) gflat[i] = i >= st.lo && i < st.hi ? g[i] : 0.0f;
    return;
  }
  for (int i = st.lo + threadIdx.x; i < st.hi; i += blockDim.x) {
    float v = sq[i];
    float p = rnvp_rmsprop_update(g[i], params[i], v, st.k);
    if (st.clip > 0.0f) p = fminf(fmaxf(p, -st.clip), st.clip);
    params[i] = p;
    sq[i] = v;
  }
}

// gradient partials + score sums per CTA at partials + b * stride (steps), or the score sums alone at partials[b],
// partials[n_ctas + b] (loss)
__global__ void __launch_bounds__(MLP_THREADS) wg_sweep_kernel(WgShape s, const float* __restrict__ params,
    const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx, int64_t nb, MlpNoise nz,
    float inv_nb, int kind, float* __restrict__ partials) {
  extern __shared__ __align__(16) float smem[];
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(nb - row0 < s.R ? nb - row0 : s.R);
  if (kind == WG_LOSS) {
    float sums[2];
    sweep_tile(s, smem, params, X, C, idx, row0, nr, nz, inv_nb, kind, nullptr, sums);
    if (threadIdx.x == 0) {
      partials[blockIdx.x] = sums[0];
      partials[gridDim.x + blockIdx.x] = sums[1];
    }
    return;
  }
  float* g = partials + (size_t)blockIdx.x * s.stride;
  sweep_tile(s, smem, params, X, C, idx, row0, nr, nz, inv_nb, kind, g, g + s.P);
}

// the epoch losses from n_ctas per-CTA fake and real score sums: gen = -mean(D(fake)), disc = mean(D(real)) + gen
__global__ void __launch_bounds__(MLP_THREADS) wg_loss_reduce_kernel(const float* __restrict__ partials, int64_t n_ctas,
                                                                    int64_t N, float* gen_dst, float* disc_dst) {
  __shared__ float scratch[32];
  float s[2];                                         // fake, real
  block_sums_strided<2>(partials, n_ctas, scratch, s);
  if (threadIdx.x == 0) {
    const float gen = -(s[0] / (float)N);
    *gen_dst = gen;
    *disc_dst = s[1] / (float)N + gen;
  }
}

__global__ void __launch_bounds__(MLP_TAIL_THREADS) wg_tail_kernel(WgShape s, float* params, float* sq, const float* g,
                                                                 float* gflat, float* loss_dst, WgStep st) {
  wg_tail(s, params, sq, g, gflat, loss_dst, st);
}

// a whole step of a batch that fits one tile
__global__ void __launch_bounds__(MLP_TAIL_THREADS) wg_step_kernel(WgShape s, float* params, float* sq,
    const float* __restrict__ X, const float* __restrict__ C, const int64_t* __restrict__ idx, int nb, MlpNoise nz,
    float* g, float* gflat, float* loss_dst, WgStep st) {
  extern __shared__ __align__(16) float smem[];
  sweep_tile(s, smem, params, X, C, idx, 0, nb, nz, st.inv_nb, st.kind, g, g + s.P);
  __syncthreads();                                     // g (global) is read back by other threads of this CTA
  wg_tail(s, params, sq, g, gflat, loss_dst, st);
}

// Generator.forward for inference: x of rows [z|C], z from Z or from Philox keyed on (seed, row_offset + row, j)
__global__ void __launch_bounds__(MLP_THREADS) wg_generate_kernel(WgShape s, const float* __restrict__ params,
    const float* __restrict__ Z, const float* __restrict__ C, int64_t N, unsigned long long seed, long long row_offset,
    float* x_o) {
  extern __shared__ __align__(16) float smem[];
  const WgTile t = carve(s, smem);
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(N - row0 < s.R ? N - row0 : s.R);
  load_tile(s, t, nullptr, C, nullptr, row0, nr, MlpNoise{Z, seed, row_offset}, false);
  __syncthreads();
  gen_forward(s, t, params, nr);
  const int D = s.D;
  for (int e = threadIdx.x; e < nr * D; e += blockDim.x) {
    const int r = e / D, j = e - r * D;
    x_o[(row0 + r) * D + j] = t.xf[r * t.ldx + j];
  }
}

// Discriminator.forward for inference: the scores [N] of rows [X|C]
__global__ void __launch_bounds__(MLP_THREADS) wg_critic_kernel(WgShape s, const float* __restrict__ params,
    const float* __restrict__ X, const float* __restrict__ C, int64_t N, float* score_o) {
  extern __shared__ __align__(16) float smem[];
  const WgTile t = carve(s, smem);
  const int64_t row0 = (int64_t)blockIdx.x * s.R;
  const int nr = (int)(N - row0 < s.R ? N - row0 : s.R);
  const int D = s.D, Cd = s.Cd, W = D + Cd;
  for (int e = threadIdx.x; e < nr * W; e += blockDim.x) {
    const int r = e / W, j = e - r * W;
    const int64_t row = row0 + r;
    t.xr[r * t.ldx + j] = j < D ? X[row * D + j] : C[row * Cd + (j - D)];
  }
  __syncthreads();
  mlp_forward(s.d, params, t.xr, t.ldx, W, t.dh, t.ldd, s.d.w, s.d.b, s.d.ow, s.d.ob, t.o, 0, 0, nullptr, 1, 1, nr);
  for (int r = threadIdx.x; r < nr; r += blockDim.x) score_o[row0 + r] = t.o[r];
}

}  // namespace

struct rnvp_wg_desc {
  WgShape s;
};

namespace {

int check_wg(const rnvp_wg_desc* d) { return d ? 0 : rnvp_fail(RNVP_EINVAL, "null ConditionalWGAN descriptor"); }

// the gradient (gflat, update 0) or the RMSprop step of one batch of nb positions of idx
void launch_step(const WgShape& s, float* params, float* sq, const float* X, const float* C, const int64_t* idx,
                 int64_t nb, const MlpNoise& nz, float* gflat, float* loss_dst, const WgStep& st, float* ws,
                 cudaStream_t stream) {
  const int64_t nt = n_tiles(s.R, nb);
  float* g = ws;                                       // reduced record (stride floats), then the partials
  if (nt == 1) {
    wg_step_kernel<<<1, MLP_TAIL_THREADS, s.smem, stream>>>(s, params, sq, X, C, idx, (int)nb, nz, g, gflat, loss_dst,
                                                           st);
    return;
  }
  float* partials = ws + s.stride;
  wg_sweep_kernel<<<(unsigned)nt, MLP_THREADS, s.smem, stream>>>(s, params, X, C, idx, nb, nz, st.inv_nb, st.kind,
                                                                partials);
  launch_reduce(partials, (int)nt, s.stride, s.P, st.lo, st.hi, 2, g, nullptr, stream);   // + fake and real score sums
  wg_tail_kernel<<<1, MLP_TAIL_THREADS, 0, stream>>>(s, params, sq, g, gflat, loss_dst, st);
}

// the epoch losses over N positions of idx into *gen_dst, *disc_dst
void launch_loss(const WgShape& s, const float* params, const float* X, const float* C, const int64_t* idx, int64_t N,
                 const MlpNoise& nz, float* gen_dst, float* disc_dst, float* ws, cudaStream_t stream) {
  const int64_t nt = n_tiles(s.R, N);
  wg_sweep_kernel<<<(unsigned)nt, MLP_THREADS, s.smem, stream>>>(s, params, X, C, idx, N, nz, 0.0f, WG_LOSS, ws);
  wg_loss_reduce_kernel<<<1, MLP_THREADS, 0, stream>>>(ws, nt, N, gen_dst, disc_dst);
}

WgStep make_step(const WgShape& s, int generator, int64_t nb, int update) {
  WgStep st{};
  st.kind = generator ? WG_GENERATOR : WG_CRITIC;
  st.lo = generator ? 0 : s.PG;
  st.hi = generator ? s.PG : s.P;
  st.nb = (float)nb;
  st.inv_nb = (float)(1.0 / (double)nb);
  st.update = update;
  return st;
}

}  // namespace

extern "C" {

int rnvp_wg_desc_create(int D, int Cd, int latent, int g_hidden_n, const int* g_hidden, int g_act, int d_hidden_n,
                        const int* d_hidden, int d_act, rnvp_wg_desc** out) {
  if (!out) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_desc_create: out is null");
  *out = nullptr;
  if (!g_hidden || !d_hidden || D < 1 || Cd < 0 || latent < 1 || g_hidden_n < 1 || d_hidden_n < 1)
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_desc_create: bad shape");
  for (int a : {g_act, d_act})
    if (a != RNVP_ACT_TANH && a != RNVP_ACT_RELU)
      return rnvp_fail(RNVP_EINVAL, "rnvp_wg_desc_create: act must be RNVP_ACT_TANH or _RELU");
  if (D > MLP_MAX_D) return rnvp_fail(RNVP_ESHAPE, "ConditionalWGAN: var_size D must be <= 128");
  if (Cd > MLP_MAX_CD) return rnvp_fail(RNVP_ESHAPE, "ConditionalWGAN: cond_size must be <= 256");
  if (latent > MLP_MAX_LAT) return rnvp_fail(RNVP_ESHAPE, "ConditionalWGAN: latent_dim must be <= 128");
  if (g_hidden_n > MLP_MAX_HIDDEN || d_hidden_n > MLP_MAX_HIDDEN)
    return rnvp_fail(RNVP_ESHAPE, "ConditionalWGAN: at most 4 hidden layers per net");
  WgShape s{};
  s.D = D; s.Cd = Cd; s.L = latent;
  s.g = WgNet{g_hidden_n, g_act, latent + Cd, D};
  s.d = WgNet{d_hidden_n, d_act, D + Cd, 1};
  const char *model = "ConditionalWGAN", *fn = "rnvp_wg_desc_create";
  int64_t off = 0;
  if (int rc = hidden_layout(g_hidden_n, g_hidden, latent + Cd, s.g.h, s.g.w, s.g.b, off, model, fn)) return rc;
  linear_layout(s.g.ow, s.g.ob, g_hidden[g_hidden_n - 1], D, off);
  s.PG = (int)off;
  if (int rc = hidden_layout(d_hidden_n, d_hidden, D + Cd, s.d.h, s.d.w, s.d.b, off, model, fn)) return rc;
  linear_layout(s.d.ow, s.d.ob, d_hidden[d_hidden_n - 1], 1, off);
  s.P = (int)off;
  s.stride = (s.P + 2 + 3) & ~3;
  s.R = rows_per_tile(s);
  s.smem = tile_floats(s, s.R) * 4;
  if (int rc = opt_in_smem({(const void*)wg_sweep_kernel, (const void*)wg_step_kernel, (const void*)wg_generate_kernel,
                            (const void*)wg_critic_kernel},
                           s.smem, model, fn))
    return rc;
  *out = new rnvp_wg_desc{s};
  return 0;
}

void rnvp_wg_desc_destroy(rnvp_wg_desc* d) { delete d; }

int64_t rnvp_wg_param_count(const rnvp_wg_desc* d, int net) {
  if (!d) return -1;
  if (net == 0) return d->s.PG;
  if (net == 1) return d->s.P - d->s.PG;
  return d->s.P;
}

int64_t rnvp_wg_workspace_bytes(const rnvp_wg_desc* d, int64_t batch_rows, int64_t loss_rows) {
  if (!d || batch_rows < 0 || loss_rows < 0) return -1;
  const int64_t nt = n_tiles(d->s.R, batch_rows);
  return 4 * std::max((int64_t)d->s.stride * (1 + (nt > 1 ? nt : 0)), 2 * n_tiles(d->s.R, loss_rows));
}

int rnvp_wg_generate(const rnvp_wg_desc* d, const float* d_params, const float* d_Z, const float* d_C, int64_t N,
                     uint64_t seed, int64_t row_offset, float* d_x, void* stream) {
  if (check_wg(d)) return RNVP_EINVAL;
  if (!d_params || (d->s.Cd && !d_C) || !d_x || N < 0) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_generate: bad argument");
  if (N == 0) return 0;
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_generate: too many rows");
  wg_generate_kernel<<<(unsigned)n_tiles(d->s.R, N), MLP_THREADS, d->s.smem, (cudaStream_t)stream>>>(
      d->s, d_params, d_Z, d_C, N, seed, row_offset, d_x);
  return launched("wg_generate_kernel launch");
}

int rnvp_wg_critic(const rnvp_wg_desc* d, const float* d_params, const float* d_X, const float* d_C, int64_t N,
                   float* d_score, void* stream) {
  if (check_wg(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || (d->s.Cd && !d_C) || !d_score || N < 0)
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_critic: bad argument");
  if (N == 0) return 0;
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_critic: too many rows");
  wg_critic_kernel<<<(unsigned)n_tiles(d->s.R, N), MLP_THREADS, d->s.smem, (cudaStream_t)stream>>>(
      d->s, d_params, d_X, d_C, N, d_score);
  return launched("wg_critic_kernel launch");
}

int rnvp_wg_grad(const rnvp_wg_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_z, int64_t N, int generator_step, float* d_gflat, float* d_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_wg(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || (d->s.Cd && !d_C) || !d_z || !d_gflat || N < 1)
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_grad: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_wg_workspace_bytes(d, N, 0))
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_grad: workspace smaller than rnvp_wg_workspace_bytes(N, 0)");
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_grad: too many rows");
  const WgStep st = make_step(d->s, generator_step, N, 0);
  launch_step(d->s, const_cast<float*>(d_params), nullptr, d_X, d_C, d_idx, N, MlpNoise{d_z, 0, 0}, d_gflat, d_loss, st,
              (float*)d_workspace, (cudaStream_t)stream);
  return launched("ConditionalWGAN gradient launch");
}

int rnvp_wg_loss(const rnvp_wg_desc* d, const float* d_params, const float* d_X, const float* d_C,
                 const int64_t* d_idx, const float* d_z, int64_t N, float* d_gen_loss, float* d_disc_loss,
                 void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_wg(d)) return RNVP_EINVAL;
  if (!d_params || !d_X || (d->s.Cd && !d_C) || !d_z || !d_gen_loss || !d_disc_loss || N < 1)
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_loss: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_wg_workspace_bytes(d, 0, N))
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_loss: workspace smaller than rnvp_wg_workspace_bytes(0, N)");
  if (bad_rows(d->s.R, N)) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_loss: too many rows");
  launch_loss(d->s, d_params, d_X, d_C, d_idx, N, MlpNoise{d_z, 0, 0}, d_gen_loss, d_disc_loss, (float*)d_workspace,
              (cudaStream_t)stream);
  return launched("ConditionalWGAN loss launch");
}

int rnvp_wg_fit_epoch(const rnvp_wg_desc* d, float* d_params, float* d_square_avg, const float* d_X, const float* d_C,
                      const int64_t* d_perm, int64_t n, int64_t batch_size, int64_t n_critic, int64_t step0, double lr,
                      double alpha, double eps, double weight_decay, double clip, const float* d_noise, uint64_t seed,
                      float* d_gen_loss, float* d_disc_loss, void* d_workspace, int64_t workspace_bytes,
                      void* stream) {
  if (check_wg(d)) return RNVP_EINVAL;
  if (!d_params || !d_square_avg || !d_X || (d->s.Cd && !d_C) || !d_perm || !d_gen_loss || !d_disc_loss || n < 1 ||
      batch_size < 1 || n_critic < 1 || step0 < 0)
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_fit_epoch: bad argument");
  if (!d_workspace || workspace_bytes < rnvp_wg_workspace_bytes(d, std::min(n, batch_size), n))
    return rnvp_fail(RNVP_EINVAL, "rnvp_wg_fit_epoch: workspace smaller than rnvp_wg_workspace_bytes(batch_size, n)");
  if (bad_rows(d->s.R, n)) return rnvp_fail(RNVP_EINVAL, "rnvp_wg_fit_epoch: too many rows");
  const WgShape& s = d->s;
  const cudaStream_t st_ = (cudaStream_t)stream;
  const RnvpRmspropCoef k{(float)lr, (float)alpha, (float)(1.0 - alpha), (float)eps, (float)weight_decay};
  int64_t i = step0;
  for (int64_t b0 = 0; b0 < n; b0 += batch_size, ++i) {
    const int64_t nb = std::min(batch_size, n - b0);
    const int generator = i % n_critic == 0;          // wgan.py: iter_i % n_critic != 0 is a critic step
    WgStep st = make_step(s, generator, nb, 1);
    st.k = k;
    st.clip = generator ? 0.0f : (float)clip;
    const MlpNoise nz{d_noise ? d_noise + b0 * s.L : nullptr, seed, (long long)b0};
    launch_step(s, d_params, d_square_avg, d_X, d_C, d_perm + b0, nb, nz, nullptr, nullptr, st, (float*)d_workspace,
                st_);
    if (int rc = launched("ConditionalWGAN fit step launch")) return rc;
  }
  // the epoch losses: every row in dataset order, with its own noise (rows n .. 2n - 1 of the Philox stream)
  const MlpNoise nz{d_noise ? d_noise + n * s.L : nullptr, seed, (long long)n};
  launch_loss(s, d_params, d_X, d_C, nullptr, n, nz, d_gen_loss, d_disc_loss, (float*)d_workspace, st_);
  return launched("ConditionalWGAN epoch loss launch");
}

}  // extern "C"
