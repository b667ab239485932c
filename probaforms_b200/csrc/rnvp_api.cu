// Host side of librnvp_b200.so: flow descriptor, packed-layout maps, per-tile program planner,
// pack / unpack / fused-Adam kernels and the extern "C" entry points declared in include/rnvp.h.
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/rnvp.h"
#include "rnvp_plan.h"
#include <cstdlib>
#include "rnvp_planner.h"
#include "rnvp_small.h"
#include "rnvp_wide.h"
#include "rnvp_wgrad.h"

cudaError_t rnvp_launch_tile(int mode, int TR, const RnvpKArgs& a, int grid, size_t smem_bytes, cudaStream_t stream);
int rnvp_tile_occupancy(int mode, int TR, size_t smem_bytes);
cudaError_t rnvp_launch_small(int NE, int NC, int act, int mode, const RnvpSmallArgs& a, int grid, size_t smem,
                              cudaStream_t st);
int rnvp_small_rows_per_block();
int rnvp_small_fit_rows_per_block();
int rnvp_small_fit_max_layers();
cudaError_t rnvp_launch_wgrad_tc(int NU, int TP, const RnvpWgradTcArgs& a, int grid, cudaStream_t st);
cudaError_t rnvp_launch_wide(int DH, int act, int mode, const RnvpWideArgs& a, int grid, cudaStream_t st);
int rnvp_wide_ctas_per_sm(int DH);
cudaError_t rnvp_launch_mma_selftest(const float* A, const float* B, float* D, int N, int K, int passes, cudaStream_t st);

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return (int)e;
}

struct Program {
  RnvpOp* d_ops = nullptr;
  RnvpChunk* d_chunks = nullptr;
  int n_ops = 0, n_chunks = 0;
  RnvpSmem sm{};
  int TR = 0;
  size_t smem_bytes = 0;
  int stash_per_cta = 0;
  int occupancy = 1;
};

}  // namespace

struct rnvp_desc : rnvp_planner::FlowGeom {
  int device = 0, num_sms = 1;
  int* d_p2f = nullptr;   // packed index -> flat index or -1
  int* d_f2p = nullptr;   // flat index -> packed index or -1
  int* d_s2g = nullptr;   // small-flow layout index -> index in the packed gradient accumulator or -1 (fit step of small flows)
  int* d_f2p2 = nullptr;  // flat index -> index in the small-flow layout or -1 (nullptr if unused)
  int* d_m2f = nullptr;   // tcgen05 region: 4*flat + code (0 hi, 1 lo, 2 full) or -1
  int* d_f2m = nullptr;   // [4*P]: positions of each parameter's TF32 hi / lo images (plain, transposed) in the tcgen05 region, or -1
  RnvpWgradLayer* d_wg = nullptr;   // per-layer gradient offsets for the weight-gradient sweep
  int path = 0;           // 0 auto, 1 FP32 tile/small kernels only, 2 tcgen05 where eligible
  // FP32 tile programs by (mode, layer range), built on first use: a cache, so entry points that take the descriptor
  // const may fill it
  mutable std::map<std::tuple<int, int, int>, Program> programs;
  mutable std::mutex mu;
};

namespace {
using namespace rnvp_planner;

int get_program(const rnvp_desc* d, int mode, int l0, int l1, Program** out) {
  std::lock_guard<std::mutex> lock(d->mu);
  auto key = std::make_tuple(mode, l0, l1);
  auto it = d->programs.find(key);
  if (it != d->programs.end()) { *out = &it->second; return 0; }
  Builder b;
  b.d = d; b.mode = mode; b.l0 = l0; b.l1 = l1;
  const char* force = getenv("RNVP_FORCE_TR");     // development knob: force the row-tile size
  const bool ok = b.plan_best(force ? atoi(force) : 0);
  if (!ok) {
    char msg[256];
    snprintf(msg, sizeof(msg), "flow does not fit the shared-memory plan (D=%d Cd=%d H0=%d mode=%d needs %d B > %d B)",
             d->D, d->Cd, d->hidden[0], mode, b.sm.total_floats * 4, d->max_smem);
    return fail(RNVP_ESHAPE, msg);
  }
  b.build();
  Program p;
  p.n_ops = (int)b.ops.size();
  p.n_chunks = (int)b.chunks.size();
  p.sm = b.sm;
  p.TR = b.TR;
  p.smem_bytes = (size_t)b.sm.total_floats * 4;
  p.stash_per_cta = b.stash_per_cta;
  cudaError_t e = cudaMalloc(&p.d_ops, sizeof(RnvpOp) * std::max(p.n_ops, 1));
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(ops)");
  e = cudaMalloc(&p.d_chunks, sizeof(RnvpChunk) * std::max(p.n_chunks, 1));
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(chunks)");
  e = cudaMemcpy(p.d_ops, b.ops.data(), sizeof(RnvpOp) * p.n_ops, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(ops)");
  if (p.n_chunks) {
    e = cudaMemcpy(p.d_chunks, b.chunks.data(), sizeof(RnvpChunk) * p.n_chunks, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(chunks)");
  }
  p.occupancy = std::max(1, rnvp_tile_occupancy(mode, p.TR, p.smem_bytes));
  auto ins = d->programs.emplace(key, p);
  *out = &ins.first->second;
  return 0;
}

// ------------------------------------------------------- small utility kernels
__global__ void pack_kernel(const float* __restrict__ flat, float* __restrict__ packed,
                            const int* __restrict__ p2f, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    int f = p2f[i];
    packed[i] = f >= 0 ? flat[f] : 0.0f;
  }
}
// tcgen05 weight images: TF32 round-to-nearest "hi" part, fp32 remainder "lo", or the plain value
__global__ void pack_mma_kernel(const float* __restrict__ flat, float* __restrict__ img, const int* __restrict__ m2f, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const int raw = m2f[i];
    float out = 0.0f;
    if (raw >= 0) {
      const int m = raw & ~RNVP_IMG_SCALED;
      const float v = (raw & RNVP_IMG_SCALED) ? flat[m >> 2] * RNVP_TANH_PRESCALE : flat[m >> 2];
      const uint32_t h = (__float_as_uint(v) + 0x1000u) & 0xFFFFE000u;          // round_tf32, see tc05.cuh
      const uint32_t l = (__float_as_uint(v - __uint_as_float(h)) + 0x1000u) & 0xFFFFE000u;
      const int code = m & 3;
      out = code == 0 ? __uint_as_float(h) : (code == 1 ? __uint_as_float(l) : v);
    }
    img[i] = out;
  }
}
__global__ void unpack_kernel(const float* __restrict__ gpacked, float* __restrict__ gflat,
                              const int* __restrict__ f2p, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    int p = f2p[i];
    gflat[i] = p >= 0 ? gpacked[p] : 0.0f;
  }
}
// torch.optim.Adam single-tensor update (torch/optim/adam.py _single_tensor_adam), fused with the
// gradient gather from the packed accumulator (or a reference-layout gradient), the refresh of the
// packed parameter copy, the re-zeroing of the accumulator and the hand-off of the step's loss.
__global__ void adam_kernel(float* __restrict__ theta, float* __restrict__ packed, float* __restrict__ gpacked,
                            const float* __restrict__ gflat_in, float* __restrict__ m, float* __restrict__ v,
                            float* __restrict__ gflat_out, const int* __restrict__ f2p, const int* __restrict__ f2p2,
                            const int* __restrict__ f2m, float* __restrict__ mma_img, int n, float grad_scale,
                            float wd, float one_minus_b1, float b2, float one_minus_b2, float step_size,
                            float bc2_sqrt, float eps, int zero_gpacked, float* loss_src, float* loss_dst,
                            float loss_scale) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && loss_src) {
    if (loss_dst) *loss_dst = *loss_src * loss_scale;
    if (zero_gpacked) *loss_src = 0.0f;
  }
  if (i >= n) return;
  const int p = f2p[i];
  float g;
  if (gflat_in) g = gflat_in[i] * grad_scale;
  else {
    g = p >= 0 ? gpacked[p] * grad_scale : 0.0f;
    if (zero_gpacked && p >= 0) gpacked[p] = 0.0f;
  }
  if (gflat_out) gflat_out[i] = g;
  float mi = m[i], vi = v[i];
  const RnvpAdamCoef k{wd, one_minus_b1, b2, one_minus_b2, step_size, bc2_sqrt, eps};
  const float th = rnvp_adam_update(g, theta[i], mi, vi, k);
  m[i] = mi; v[i] = vi; theta[i] = th;
  if (p >= 0) packed[p] = th;
  if (f2p2) {
    const int p2 = f2p2[i];
    if (p2 >= 0) packed[p2] = th;
  }
  if (f2m) {                                           // TF32 hi / lo images of the tcgen05 kernels (see tc05.cuh)
    const int4 mm = reinterpret_cast<const int4*>(f2m)[i];
    const uint32_t h = (__float_as_uint(th) + 0x1000u) & 0xFFFFE000u;
    const float fh = __uint_as_float(h), fl = __uint_as_float((__float_as_uint(th - fh) + 0x1000u) & 0xFFFFE000u);
    if ((mm.x >= 0 && (mm.x & RNVP_IMG_SCALED)) || (mm.y >= 0 && (mm.y & RNVP_IMG_SCALED))) {
      // forward W1 image of a tanh flow: 2 log2(e) * theta (see build_mma_map)
      const float ts = th * RNVP_TANH_PRESCALE;
      const uint32_t hs = (__float_as_uint(ts) + 0x1000u) & 0xFFFFE000u;
      const float fhs = __uint_as_float(hs), fls = __uint_as_float((__float_as_uint(ts - fhs) + 0x1000u) & 0xFFFFE000u);
      if (mm.x >= 0) mma_img[mm.x & ~RNVP_IMG_SCALED] = fhs;
      if (mm.y >= 0) mma_img[mm.y & ~RNVP_IMG_SCALED] = fls;
    } else {
      if (mm.x >= 0) mma_img[mm.x] = fh;
      if (mm.y >= 0) mma_img[mm.y] = fl;
    }
    if (mm.z >= 0) mma_img[mm.z & ~RNVP_IMG_SCALED] = fh;
    if (mm.w >= 0) mma_img[mm.w & ~RNVP_IMG_SCALED] = fl;
  }
}

int check_desc(const rnvp_desc* d) { return d ? 0 : fail(RNVP_EINVAL, "null descriptor"); }

// kernel families, numbered as rnvp_plan_info reports them
enum Family { FAMILY_TILE = 0, FAMILY_SMALL = 1, FAMILY_MMA = 2 };

// The family that runs mode `mode` (0 forward, 1 inverse, 2 fit step) of a flow: the one place that reads the path and
// the eligibility flags to choose.  The planner keeps the two eligible sets disjoint (mma_ok needs D > 8, small_ok
// needs D <= 8: rnvp_planner.h build_layout), so the order of the two tests below decides nothing.
Family family(const rnvp_desc* d, int mode) {
  // the tcgen05 fit step (forward + backward sweeps, then the weight-gradient sweep) needs the transposed weight images
  if (d->mma_ok && d->path != 1 && (mode != 2 || d->m_wt_floats > 0)) return FAMILY_MMA;
  // the small-flow fit kernel (one launch, no workspace) has a layer limit and three small-layout arrays in shared memory
  if (d->small_ok && (mode != 2 || (d->L <= rnvp_small_fit_max_layers() && d->small_floats * 12 + 4096 <= d->max_smem)))
    return FAMILY_SMALL;
  return FAMILY_TILE;
}

// One call of the row kernels as an entry point makes it; run_tile, run_small and run_mma fill their kernel's arguments
// from it.
struct RowCall {
  const float *packed = nullptr, *X = nullptr, *C = nullptr;   // X: input rows, or nullptr when an inverse draws them
  const long long* idx = nullptr;                              // optional row gather
  long long N = 0;
  int l0 = 0, l1 = 0;                                          // layer range
  float *out_x = nullptr, *out_logdet = nullptr, *out_logp = nullptr;
  unsigned long long seed = 0;                                 // drawn latent rows are keyed on row_offset + row
  long long row_offset = 0;
  // fit step (mode 2)
  float *gpacked = nullptr, *loss_sum = nullptr;
  float scale = 0.f;
  void* workspace = nullptr;
  int64_t workspace_bytes = 0;
  const RnvpFusedAdam* fused = nullptr;                        // small-flow fit step of one CTA: Adam fused behind it
};

// Argument rules of the row entry points, reported under the entry point's name: the packed parameters, the input rows
// unless the call draws them, the output rows of an inverse, the gradient accumulator of a fit step, and C exactly when
// the flow is conditional.
int check_rows(const rnvp_desc* d, const char* fn, int mode, const RowCall& c, bool draws) {
  if (c.N < 0 || c.row_offset < 0 || !c.packed || (mode == 2 && !c.gpacked) ||
      (c.N > 0 && ((!draws && !c.X) || (mode == 1 && !c.out_x))))
    return fail(RNVP_EINVAL, std::string(fn) + (draws ? ": bad argument" : ": null buffer"));
  if (c.N > 0 && (d->Cd > 0) != (c.C != nullptr))
    return fail(RNVP_EINVAL, std::string(fn) + ": C must be given iff cond_size > 0");
  return 0;
}

int run_tile(const rnvp_desc* d, int mode, const RowCall& c, cudaStream_t stream) {
  Program* p = nullptr;
  int rc = get_program(d, mode, c.l0, c.l1, &p);
  if (rc) return rc;
  const int R = 8 * p->TR;
  const long long n_tiles = (c.N + R - 1) / R;
  if (n_tiles > 0x7fffffffLL) return fail(RNVP_EINVAL, "too many rows for one launch");
  int grid = (int)std::min<long long>(n_tiles, (long long)d->num_sms * p->occupancy);
  RnvpKArgs a{};
  if (mode == 2) {
    const long long per_cta = (long long)p->stash_per_cta * 4;
    const long long fit = per_cta > 0 ? c.workspace_bytes / per_cta : grid;
    if (!c.workspace || fit < 1) return fail(RNVP_EINVAL, "rnvp_backward: workspace too small (see rnvp_workspace_bytes)");
    grid = (int)std::min<long long>(grid, fit);
    a.stash = (float*)c.workspace;
    a.stash_per_cta = p->stash_per_cta;
  }
  a.packed = c.packed; a.X = c.X; a.C = c.C; a.idx = c.idx; a.N = c.N;
  a.out_x = c.out_x; a.out_logdet = c.out_logdet; a.out_logp = c.out_logp;
  a.gpacked = c.gpacked; a.loss_sum = c.loss_sum; a.scale = c.scale;
  a.seed = c.seed; a.row_offset = c.row_offset;
  a.ops = p->d_ops; a.chunks = p->d_chunks; a.n_ops = p->n_ops; a.n_chunks = p->n_chunks; a.n_tiles = (int)n_tiles;
  a.D = d->D; a.Cd = d->Cd; a.sm = p->sm;
  cudaError_t e = rnvp_launch_tile(mode, p->TR, a, grid, p->smem_bytes, stream);
  return e == cudaSuccess ? 0 : cuda_fail(e, "tile kernel launch");
}

int run_small(const rnvp_desc* d, int mode, const RowCall& c, cudaStream_t stream) {
  RnvpSmallArgs a{};
  a.packed_small = c.packed + d->small_off;
  a.X = c.X; a.C = c.C; a.idx = c.idx; a.N = c.N;
  a.out_x = c.out_x; a.out_logdet = c.out_logdet; a.out_logp = c.out_logp;
  a.D = d->D; a.Cd = d->Cd; a.H = d->hidden[0]; a.rec = d->srec; a.small_floats = d->small_floats;
  a.l0 = c.l0; a.l1 = c.l1;
  a.gpacked = c.gpacked; a.s2g = d->d_s2g; a.loss_sum = c.loss_sum; a.scale = c.scale;
  a.seed = c.seed; a.row_offset = c.row_offset;
  if (c.fused) {
    if (mode != 2 || c.N > rnvp_small_fit_rows_per_block()) return fail(RNVP_EINVAL, "fused Adam needs a single-CTA fit step");
    a.fuse_adam = 1;
    a.ad = *c.fused;
  }
  const long long rpb = mode == 2 ? rnvp_small_fit_rows_per_block() : rnvp_small_rows_per_block();
  const long long blocks = (c.N + rpb - 1) / rpb;
  const int grid = (int)std::min<long long>(blocks, (long long)d->num_sms * (mode == 2 ? 16 : 8));
  cudaError_t e = rnvp_launch_small(d->sNE, d->sNC, d->act, mode, a, grid, (size_t)d->small_floats * 4, stream);
  return e == cudaSuccess ? 0 : cuda_fail(e, "small-flow kernel launch");
}

long long* g_wg_trace = nullptr;    // development aid: wait accounting of -DRNVP_WG_TRACE builds, see rnvp_debug_set_trace
// rows covered by the record / stash arrays of a tensor-core fit step: whole 128-row tiles of the sweep kernel, so that
// the weight-gradient sweep never reads an unwritten record
int64_t fit_npad(int64_t N) { return (N + 127) / 128 * 128; }
// record stride of the activation records exchanged between the backward sweep and the weight-gradient sweep
int wgrad_rec_floats(const rnvp_desc* d) {
  const int K1P = (d->mDH + d->Cd + 7) & ~7;
  return 2 * d->hidden[0] + K1P + 2 * d->mDH;               // multiple of 8: an even number of float4 column groups
}

int run_mma(const rnvp_desc* d, int mode, const RowCall& c, cudaStream_t stream) {
  RnvpWideArgs a{};
  a.wimg = c.packed + d->mma_off;
  a.X = c.X; a.C = c.C; a.idx = c.idx; a.N = c.N;
  a.out_x = c.out_x; a.out_logdet = c.out_logdet; a.out_logp = c.out_logp;
  a.Cd = d->Cd; a.H = d->hidden[0]; a.l0 = c.l0; a.l1 = c.l1;
  a.layer_floats = d->m_layer_floats; a.w1_floats = d->m_w1_floats; a.w2_floats = d->m_w2_floats;
  a.loss_sum = c.loss_sum; a.L_total = d->L; a.scale = c.scale;
  a.seed = c.seed; a.row_offset = c.row_offset; a.Dreal = d->D;
  if (mode == 2) {
    // forward + backward sweeps in one launch (per-layer records to the workspace), then the weight-gradient sweep
    const int64_t npad = fit_npad(c.N);
    const int64_t stash_f = npad * d->L * 2 * d->mDH, rec_f = (int64_t)d->L * npad * wgrad_rec_floats(d);   // both blocked by 32 rows
    if (!c.workspace || c.workspace_bytes < (stash_f + rec_f) * 4)
      return fail(RNVP_EINVAL, "rnvp_backward: workspace too small (see rnvp_workspace_bytes)");
    a.stash = (float*)c.workspace; a.records = a.stash + stash_f;
    a.do_bwd = 1; a.rec = wgrad_rec_floats(d); a.Npad = npad; a.wt_floats = d->m_wt_floats;
  }
  // one 128-row tile per CTA, two threads per row, weight images streamed per chunk step (rnvp_wide.cu)
  const long long tiles = (c.N + 127) / 128;
  if (tiles > 0x7fffffffLL) return fail(RNVP_EINVAL, "too many rows for one launch");
  a.n_tiles = (int)tiles;
  const long long ctas = (long long)d->num_sms * rnvp_wide_ctas_per_sm(d->mDH);   // DH <= 32: two CTAs per SM
  cudaError_t e = rnvp_launch_wide(d->mDH, d->act, mode, a, (int)std::min<long long>(tiles, ctas), stream);
  if (e != cudaSuccess) return cuda_fail(e, "tcgen05 streamed kernel launch");
  return mode == 2 ? rnvp_wgrad_sweep(d, c.packed, a.Npad, a.records, c.gpacked, stream) : 0;
}

// a row call on the family that runs it, after the checks all three share
int run(const rnvp_desc* d, int mode, const RowCall& c, cudaStream_t stream) {
  if (c.l0 < 0 || c.l1 > d->L || c.l0 >= c.l1) return fail(RNVP_EINVAL, "bad layer range");
  if (c.N <= 0) return 0;
  switch (family(d, mode)) {
    case FAMILY_MMA: return run_mma(d, mode, c, stream);
    case FAMILY_SMALL: return run_small(d, mode, c, stream);
    default: return run_tile(d, mode, c, stream);
  }
}

}  // namespace

// ===================================================================== C ABI
extern "C" {

int rnvp_version(void) { return 100; }
const char* rnvp_last_error(void) { return g_err.c_str(); }
}  // extern "C"

// rnvp_last_error() for the entry points of other translation units (rnvp_metrics.cu)
int rnvp_fail(int code, const char* msg) { return fail(code, msg); }

extern "C" {

int rnvp_desc_create(int D, int Cd, int L, int n_hidden, const int* hidden, int act, rnvp_desc** out) {
  if (!out) return fail(RNVP_EINVAL, "out is null");
  *out = nullptr;
  if (D < 1 || Cd < 0 || L < 1 || n_hidden < 1 || n_hidden > RNVP_MAX_HIDDEN || !hidden)
    return fail(RNVP_EINVAL, "bad flow shape");
  if (act != RNVP_ACT_TANH && act != RNVP_ACT_RELU) return fail(RNVP_EINVAL, "act must be RNVP_ACT_TANH or RNVP_ACT_RELU");
  for (int q = 0; q < n_hidden; ++q)
    if (hidden[q] < 1) return fail(RNVP_EINVAL, "hidden width must be >= 1");
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
  if (prop.major != 10) {
    char msg[160];
    snprintf(msg, sizeof(msg), "librnvp_b200 is built for sm_100a only; device %d is sm_%d%d", dev, prop.major, prop.minor);
    return fail(RNVP_ENODEVICE, msg);
  }
  rnvp_desc* d = new rnvp_desc();
  d->D = D; d->Cd = Cd; d->L = L; d->nh = n_hidden; d->act = act;
  for (int q = 0; q < n_hidden; ++q) d->hidden[q] = hidden[q];
  d->device = dev;
  d->num_sms = prop.multiProcessorCount;
  d->max_smem = (int)prop.sharedMemPerBlockOptin;
  build_layout(d);
  if (d->P >= 0x7fffffffLL) { delete d; return fail(RNVP_ESHAPE, "flow too large (>= 2^31 parameters)"); }
  std::vector<int> p2f, f2p, f2p2;
  build_maps(d, p2f, f2p);
  build_small_map(d, p2f, f2p2);
  if (d->small_ok) {
    std::vector<int> s2g(d->small_floats, -1);
    for (size_t f = 0; f < f2p2.size() && f < f2p.size(); ++f)
      if (f2p2[f] >= 0 && f2p[f] >= 0) s2g[f2p2[f] - d->small_off] = f2p[f];
    e = cudaMalloc(&d->d_s2g, sizeof(int) * s2g.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_s2g, s2g.data(), sizeof(int) * s2g.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&d->d_f2p2, sizeof(int) * f2p2.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_f2p2, f2p2.data(), sizeof(int) * f2p2.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { rnvp_desc_destroy(d); return cuda_fail(e, "descriptor tables"); }
  }
  if (d->mma_ok) {
    std::vector<int> m2f;
    build_mma_map(d, m2f);
    std::vector<int> f2m(4 * (size_t)d->P, -1);       // per parameter: hi, lo, hi (transposed image), lo (transposed image)
    for (size_t m = 0; m < m2f.size(); ++m)
      if (m2f[m] >= 0 && (m2f[m] & 3) < 2) {
        const int v = m2f[m] & ~RNVP_IMG_SCALED;
        int* slot = &f2m[4 * (size_t)(v >> 2) + (v & 3)];
        if (*slot >= 0) slot += 2;
        *slot = (int)m | (m2f[m] & RNVP_IMG_SCALED);       // the slot remembers whether its image holds the pre-scaled value
      }
    e = cudaMalloc(&d->d_m2f, sizeof(int) * m2f.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_m2f, m2f.data(), sizeof(int) * m2f.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&d->d_f2m, sizeof(int) * f2m.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_f2m, f2m.data(), sizeof(int) * f2m.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { rnvp_desc_destroy(d); return cuda_fail(e, "descriptor tables"); }
  }
  if (d->nh == 1) {
    std::vector<RnvpWgradLayer> wl(d->L);
    for (int i = 0; i < d->L; ++i) {
      const LinearGeom& g0 = d->layers[i].lin[0];
      const LinearGeom& g1 = d->layers[i].lin[1];
      for (int net = 0; net < 2; ++net) {
        wl[i].w1_off[net] = g0.w_off[net]; wl[i].b1_off[net] = g0.b_off[net];
        wl[i].w2_off[net] = g1.w_off[net]; wl[i].b2_off[net] = g1.b_off[net];
      }
      wl[i].Ks1 = g0.Ks; wl[i].Ks2 = g1.Ks;
      wl[i].nK = d->layers[i].nK; wl[i].nT = d->layers[i].nT;
    }
    e = cudaMalloc(&d->d_wg, sizeof(RnvpWgradLayer) * wl.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_wg, wl.data(), sizeof(RnvpWgradLayer) * wl.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { rnvp_desc_destroy(d); return cuda_fail(e, "descriptor tables"); }
  }
  e = cudaMalloc(&d->d_p2f, sizeof(int) * p2f.size());
  if (e == cudaSuccess) e = cudaMalloc(&d->d_f2p, sizeof(int) * std::max<size_t>(f2p.size(), 1));
  if (e == cudaSuccess) e = cudaMemcpy(d->d_p2f, p2f.data(), sizeof(int) * p2f.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d->d_f2p, f2p.data(), sizeof(int) * f2p.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { rnvp_desc_destroy(d); return cuda_fail(e, "descriptor tables"); }
  // programs of the FP32 kernels over the full layer range: built now, so that the hot entry points never allocate
  // (shapes the tile planner cannot fit are reported when such a program is actually needed)
  {
    Program* p = nullptr;
    for (int mode = 0; mode <= 2; ++mode) get_program(d, mode, 0, d->L, &p);
    g_err.clear();
  }
  *out = d;
  return 0;
}

void rnvp_desc_destroy(rnvp_desc* d) {
  if (!d) return;
  for (auto& kv : d->programs) {
    cudaFree(kv.second.d_ops);
    cudaFree(kv.second.d_chunks);
  }
  cudaFree(d->d_p2f);
  cudaFree(d->d_f2p);
  cudaFree(d->d_f2p2);
  cudaFree(d->d_s2g);
  cudaFree(d->d_m2f);
  cudaFree(d->d_f2m);
  cudaFree(d->d_wg);
  delete d;
}

int64_t rnvp_param_count(const rnvp_desc* d) { return d ? d->P : -1; }
int64_t rnvp_packed_count(const rnvp_desc* d) { return d ? d->packed : -1; }
int64_t rnvp_grad_count(const rnvp_desc* d) { return d ? d->packed_tile : -1; }

int64_t rnvp_workspace_bytes(const rnvp_desc* d, int64_t N) {
  if (!d) return -1;
  const Family f = family(d, 2);
  if (f == FAMILY_SMALL) return 16;                     // the row-per-thread fit kernel keeps its stash in local memory
  if (f == FAMILY_MMA) {
    const int64_t npad = fit_npad(std::max<int64_t>(N, 1));
    return (npad * d->L * 2 * d->mDH + (int64_t)d->L * npad * wgrad_rec_floats(d)) * 4;
  }
  Program* p = nullptr;
  if (get_program(d, 2, 0, d->L, &p)) return -1;
  return (int64_t)p->stash_per_cta * 4 * d->num_sms * p->occupancy;
}

int rnvp_param_tensors(const rnvp_desc* d, int64_t* offsets, int max_tensors) {
  if (check_desc(d)) return RNVP_EINVAL;
  int k = 0;
  for (int i = 0; i < d->L; ++i)
    for (int net = 0; net < 2; ++net)
      for (int q = 0; q <= d->nh; ++q) {
        const LinearGeom& g = d->layers[i].lin[q];
        if (offsets && k + 2 <= max_tensors) {
          offsets[2 * k] = g.flat_w[net]; offsets[2 * k + 1] = (int64_t)g.in_full * g.out_full;
          offsets[2 * k + 2] = g.flat_b[net]; offsets[2 * k + 3] = g.out_full;
        }
        k += 2;
      }
  return k;
}

int rnvp_plan_info(const rnvp_desc* d, int mode, int* tile_rows, int* smem_bytes, int* n_ops, int* kernel_family) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (mode < 0 || mode == 3 || mode > 4) return fail(RNVP_EINVAL, "mode must be 0, 1, 2 or 4");
  Program* p = nullptr;
  int rc = get_program(d, mode == 4 ? 2 : mode, 0, d->L, &p);
  if (rc) return rc;
  if (tile_rows) *tile_rows = 8 * p->TR;
  if (smem_bytes) *smem_bytes = (int)p->smem_bytes;
  if (n_ops) *n_ops = p->n_ops;
  // pseudo-mode 4: does the whole fit step run on the tensor cores (sweeps + weight gradients)?
  if (kernel_family) *kernel_family = mode == 4 ? (family(d, 2) == FAMILY_MMA ? 2 : 0) : family(d, mode);
  return 0;
}

int rnvp_pack_params(const rnvp_desc* d, const float* d_flat, float* d_packed, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (!d_flat || !d_packed) return fail(RNVP_EINVAL, "null buffer");
  const int n = (int)d->packed_gather;
  pack_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_flat, d_packed, d->d_p2f, n);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && d->mma_ok) {
    const long long m = d->mma_floats;
    pack_mma_kernel<<<(unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_flat, d_packed + d->mma_off, d->d_m2f, m);
    e = cudaGetLastError();
  }
  return e == cudaSuccess ? 0 : cuda_fail(e, "pack_kernel");
}

int rnvp_unpack_grads(const rnvp_desc* d, const float* d_gpacked, float* d_gflat, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (!d_gpacked || !d_gflat) return fail(RNVP_EINVAL, "null buffer");
  const int n = (int)d->P;
  unpack_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_gpacked, d_gflat, d->d_f2p, n);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "unpack_kernel");
}

int rnvp_forward(const rnvp_desc* d, const float* d_packed, const float* d_X, const float* d_C,
                 const int64_t* d_idx, int64_t N, int layer_begin, int layer_end, float* d_z, float* d_logdet,
                 float* d_logp, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  RowCall c;
  c.packed = d_packed; c.X = d_X; c.C = d_C; c.idx = (const long long*)d_idx; c.N = N; c.l0 = layer_begin; c.l1 = layer_end;
  c.out_x = d_z; c.out_logdet = d_logdet; c.out_logp = d_logp;
  const int rc = check_rows(d, "rnvp_forward", 0, c, false);
  return rc ? rc : run(d, 0, c, (cudaStream_t)stream);
}

int rnvp_inverse(const rnvp_desc* d, const float* d_packed, const float* d_Y, const float* d_C, int64_t N,
                 int layer_begin, int layer_end, float* d_X, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  RowCall c;
  c.packed = d_packed; c.X = d_Y; c.C = d_C; c.N = N; c.l0 = layer_begin; c.l1 = layer_end;
  c.out_x = d_X;
  const int rc = check_rows(d, "rnvp_inverse", 1, c, false);
  return rc ? rc : run(d, 1, c, (cudaStream_t)stream);
}

int rnvp_sample(const rnvp_desc* d, const float* d_packed, const float* d_C, int64_t N, uint64_t seed, int64_t row_offset,
                float* d_X, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  RowCall c;
  c.packed = d_packed; c.C = d_C; c.N = N; c.l1 = d->L;
  c.out_x = d_X; c.seed = seed; c.row_offset = row_offset;
  const int rc = check_rows(d, "rnvp_sample", 1, c, true);
  return rc ? rc : run(d, 1, c, (cudaStream_t)stream);
}

int rnvp_backward(const rnvp_desc* d, const float* d_packed, const float* d_X, const float* d_C,
                  const int64_t* d_idx, int64_t N, float scale, float* d_gpacked, float* d_logp_sum, float* d_logp,
                  void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  RowCall c;
  c.packed = d_packed; c.X = d_X; c.C = d_C; c.idx = (const long long*)d_idx; c.N = N; c.l1 = d->L;
  c.out_logp = d_logp; c.gpacked = d_gpacked; c.loss_sum = d_logp_sum; c.scale = scale;
  c.workspace = d_workspace; c.workspace_bytes = workspace_bytes;
  const int rc = check_rows(d, "rnvp_backward", 2, c, false);
  return rc ? rc : run(d, 2, c, (cudaStream_t)stream);
}

int rnvp_adam_step(const rnvp_desc* d, float* d_flat, float* d_packed, float* d_gpacked, const float* d_gflat_in,
                   float* d_exp_avg, float* d_exp_avg_sq, float* d_gflat_out, float grad_scale, double lr,
                   double beta1, double beta2, double eps, double weight_decay, int64_t step, int zero_gpacked,
                   float* d_loss_src, float* d_loss_dst, float loss_scale, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (!d_flat || !d_packed || (!d_gpacked && !d_gflat_in) || !d_exp_avg || !d_exp_avg_sq)
    return fail(RNVP_EINVAL, "rnvp_adam_step: null buffer");
  if (step < 1) return fail(RNVP_EINVAL, "rnvp_adam_step: step is 1-based");
  // scalar step math in double, as torch does on the host
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  const float step_size = (float)(lr / bc1);
  const float bc2_sqrt = (float)sqrt(bc2);
  const int n = (int)d->P;
  adam_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      d_flat, d_packed, d_gpacked, d_gflat_in, d_exp_avg, d_exp_avg_sq, d_gflat_out, d->d_f2p, d->d_f2p2,
      d->mma_ok ? d->d_f2m : nullptr, d_packed + d->mma_off, n, grad_scale,
      (float)weight_decay, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), step_size, bc2_sqrt, (float)eps,
      zero_gpacked, d_loss_src, d_loss_dst, loss_scale);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : cuda_fail(e, "adam_kernel");
}

int rnvp_fit_epoch(const rnvp_desc* d, float* d_flat, float* d_packed, float* d_gpacked, float* d_exp_avg, float* d_exp_avg_sq,
                   const float* d_X, const float* d_C, const int64_t* d_perm, int64_t n, int64_t batch_size, double lr,
                   double beta1, double beta2, double eps, double weight_decay, int64_t step0, float* d_loss_slot,
                   float* d_losses, void* d_workspace, int64_t workspace_bytes, void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (n < 0 || batch_size < 1 || step0 < 0 || !d_perm || !d_losses || !d_loss_slot) return fail(RNVP_EINVAL, "rnvp_fit_epoch: bad argument");
  // A small-flow step of at most one CTA's rows is ONE launch: the fit kernel with the Adam update fused behind it (no
  // packed-gradient round trip; d_gpacked and the loss slot stay zero, as the two-launch path leaves them).  Arguments it
  // cannot take go to rnvp_backward and rnvp_adam_step, which report them.
  const bool fuse = family(d, 2) == FAMILY_SMALL && (d->Cd > 0) == (d_C != nullptr) && d_X && d_flat && d_packed &&
                    d_exp_avg && d_exp_avg_sq;
  int64_t s = 0;
  for (int64_t b0 = 0; b0 < n; b0 += batch_size, ++s) {
    const int64_t nb = std::min(batch_size, n - b0);
    if (fuse && nb <= rnvp_small_fit_rows_per_block()) {
      const int64_t step = step0 + s + 1;
      const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
      RnvpFusedAdam ad;
      ad.theta = d_flat; ad.packed = d_packed; ad.m = d_exp_avg; ad.v = d_exp_avg_sq;
      ad.f2p = d->d_f2p; ad.f2p2 = d->d_f2p2; ad.n = (int)d->P; ad.small_off = (int)d->small_off;
      ad.k = RnvpAdamCoef{(float)weight_decay, (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)(lr / bc1),
                          (float)sqrt(bc2), (float)eps};
      ad.loss_dst = d_losses + s; ad.loss_scale = -1.0f / (float)nb;
      RowCall c;
      c.packed = d_packed; c.X = d_X; c.C = d_C; c.idx = (const long long*)(d_perm + b0); c.N = nb; c.l1 = d->L;
      c.gpacked = d_gpacked; c.loss_sum = d_loss_slot; c.scale = -1.0f / (float)nb; c.fused = &ad;
      int rc = run(d, 2, c, (cudaStream_t)stream);
      if (rc) return rc;
      continue;
    }
    int rc = rnvp_backward(d, d_packed, d_X, d_C, d_perm + b0, nb, -1.0f / (float)nb, d_gpacked, d_loss_slot, nullptr, d_workspace,
                           workspace_bytes, stream);
    if (rc) return rc;
    rc = rnvp_adam_step(d, d_flat, d_packed, d_gpacked, nullptr, d_exp_avg, d_exp_avg_sq, nullptr, 1.0f, lr, beta1, beta2, eps,
                        weight_decay, step0 + s + 1, 1, d_loss_slot, d_losses + s, -1.0f / (float)nb, stream);
    if (rc) return rc;
  }
  return 0;
}

int rnvp_wgrad_record_floats(const rnvp_desc* d) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (!d->mma_ok) return fail(RNVP_ESHAPE, "rnvp_wgrad_record_floats: not a tcgen05-eligible flow");
  return wgrad_rec_floats(d);
}

int rnvp_wgrad_sweep(const rnvp_desc* d, const float* d_packed, int64_t Npad, const float* d_records, float* d_gpacked,
                     void* stream) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (!d->mma_ok || d->m_wt_floats == 0)
    return fail(RNVP_ESHAPE, "rnvp_wgrad_sweep: needs a flow whose fit step runs on the tensor cores (a tcgen05 flow with D <= 64, "
                             "or with H a multiple of 128)");
  if (!d_records || !d_gpacked || !d_packed) return fail(RNVP_EINVAL, "rnvp_wgrad_sweep: null buffer");
  if (Npad <= 0 || Npad % 32) return fail(RNVP_EINVAL, "rnvp_wgrad_sweep: Npad must be a positive multiple of 32");
  const int K1P = (d->mDH + d->Cd + 7) & ~7, TP = d->mDH;
  {
    // tcgen05 sweep: one CTA per (layer, block of 128 hidden units of [nn_t | nn_s], row slice), one wave of CTAs
    RnvpWgradTcArgs a;
    a.gR = d_records; a.rec = wgrad_rec_floats(d); a.Npad = Npad; a.H = d->hidden[0];
    a.K1P8 = K1P; a.K1 = d->mDH + d->Cd; a.TP = TP; a.Cd = d->Cd;
    a.n_mblocks = (2 * d->hidden[0] + 127) / 128;
    const int NU = TP == 16 ? 32 : (TP == 32 ? 48 : 96);           // dW1 tile columns of the three kernel variants (>= K1P8)
    const int rows = rnvp_wgrad_tc_rows(NU, TP);                   // rows per stage of that variant (the last stage may be short)
    const long long stages = (Npad + rows - 1) / rows;
    {
      // Row slices per (layer, unit block), cut on stage boundaries.  One wave of CTAs leaves num_sms % (L * n_mblocks) SMs
      // idle (c3: 128 CTAs on 148 SMs); cutting finer fills whole waves but every CTA pays a fixed prologue (W2^T image,
      // pipeline fill) and flush worth about `fixed` stages (wait accounting of CTA 0, tools/trace_wgrad.py: 2.7-3.9 stages
      // of 64 rows on c3; about 10 of 32 rows).  Pick the slice count with the best modelled efficiency.
      const double fixed = rows == 64 ? 4.0 : 10.0;
      const long long pairs = (long long)d->L * a.n_mblocks;
      double best = 0.0;
      int best_s = 1;
      for (long long s = 1; s <= std::min<long long>(stages, 64); ++s) {
        const long long ctas = pairs * s, waves = (ctas + d->num_sms - 1) / d->num_sms, per = (stages + s - 1) / s;
        const double eff = (double)ctas / (double)(waves * d->num_sms) * (double)per / ((double)per + fixed);
        if (eff > best * 1.005) { best = eff; best_s = (int)s; }
      }
      a.n_slices = best_s;
    }
    a.gpacked = d_gpacked; a.packed = d_packed; a.act = d->act; a.layers = d->d_wg; a.trace = g_wg_trace;
    { const char* o = getenv("RNVP_WG_ONE_ISSUER"); a.one_issuer = (o && atoi(o)) ? 1 : 0; }
    { const char* o = getenv("RNVP_WG_SLICES"); if (o && atoi(o) > 0) a.n_slices = (int)std::min<long long>(stages, atoi(o)); }
    cudaError_t e = rnvp_launch_wgrad_tc(NU, TP, a, d->L * a.n_mblocks * a.n_slices, (cudaStream_t)stream);
    return e == cudaSuccess ? 0 : cuda_fail(e, "rnvp_wgrad_tc_kernel");
  }
}

int rnvp_debug_set_trace(void* d_buf) { g_wg_trace = (long long*)d_buf; return 0; }

int rnvp_set_path(rnvp_desc* d, int path) {
  if (check_desc(d)) return RNVP_EINVAL;
  if (path < 0 || path > 2) return fail(RNVP_EINVAL, "path must be 0 (auto), 1 (fp32 kernels) or 2 (tcgen05 where eligible)");
  d->path = path;
  return 0;
}

int rnvp_mma_selftest(const float* d_A, const float* d_B, float* d_D, int N, int K, int passes, void* stream) {
  if (!d_A || !d_B || !d_D) return fail(RNVP_EINVAL, "rnvp_mma_selftest: null buffer");
  if (N < 16 || N > 256 || N % 16 || K < 8 || K > 64 || K % 8 || (passes != 1 && passes != 3 && passes != 4 && passes != 5))
    return fail(RNVP_EINVAL, "rnvp_mma_selftest: need N%16==0 in [16,256], K%8==0 in [8,64], passes 1 or 3");
  cudaError_t e = rnvp_launch_mma_selftest(d_A, d_B, d_D, N, K, passes, (cudaStream_t)stream);
  return e == cudaSuccess ? 0 : cuda_fail(e, "mma_selftest_kernel");
}

}  // extern "C"
