// tcgen05 path for WIDE flows (BASELINE configs[4]: D = 128, Cd = 32, H = 512; also D = 64 flows whose weight images do
// not fit shared memory): fused forward (log-density) and inverse (sampling) passes with the conditioner weights STREAMED.
//
// The weight images of a whole coupling layer do not stay resident in shared memory: a layer's images are 1.36 MB (c5),
// a row is 128 + 32 floats and the hidden layer has 2 x 512 units, so:
//   * one persistent CTA per SM owns ONE 128-row tile at a time; TMEM holds u = [x_K, c, 1] (hi/lo, 2 x K1PMAX columns), a
//     double-buffered GEMM1 accumulator chunk (D1 / A_hi in place, A_lo; 2 x 2 x CU columns) and the GEMM2 accumulators
//     [D2 | C2] (2 x NTP columns) -- 464 of 512 columns for c5;
//   * the hidden units are processed in chunk steps of CU = 32 units, nn_t's chunks first (t parked in registers), then
//     nn_s's; per chunk step the TMA producer (warp 0) streams the W1 chunk image [hi | lo], the W2 chunk image
//     [hi | lo] (and, at the first chunk of a net, its b2 image) from the L2-resident packed buffer into a 4-stage ring
//     (43 KB per stage for c5: every SM reads the same 1.36 MB per tile-layer -- 29 B/cycle/SM, under the L2 cap);
//   * the MMA issuer (warp 1, one elected lane) runs GEMM1 of chunk step cc+1 BEFORE it waits for the activations of chunk
//     step cc, so the tensor core works on the next chunk while the epilogue warps turn the current one into tanh(.);
//     error-compensated TF32 split A_hi*B_hi + A_lo*B_hi + A_hi*B_lo (corrections first in GEMM1, merged A_hi x [B_hi ; B_lo]
//     in GEMM2);
//   * warps 2-9 are the epilogue: TWO THREADS PER ROW (a thread cannot hold a 128-D row): thread (row, half) owns half of
//     the transformed and half of the conditioning features, writes its half of u, converts its 16 columns of every D1
//     chunk and applies the coupling to its 32 features; the two partial log-dets / squared norms meet in shared memory.
//   MODE 2 (fit step): the forward sweep additionally stashes (x_T, s) per layer and writes h = act(.) and u = [x_K, c] into
//   the activation record of (layer, row) (rnvp_wgrad_tc.cu); the same CTA then walks the layers BACKWARDS with the same
//   thread ownership, streaming the transposed chunk images: delta2 from the stash -> TMEM (hi/lo, 4 DH columns), per chunk
//   step dh = delta2 W2 (tensor core), delta1 = dh * act'(h), du += delta1 W1[:, x_K] (merged A_hi x [B_hi ; B_lo]); delta2
//   completes the record, and rnvp_wgrad_tc_kernel contracts the records over rows.  h comes back from the record through
//   the ring (DH = 16 / 64): each backward stage also carries the tile's h chunk (4 bulk copies of 4 KB, issued up to four
//   chunk steps ahead), once the tile's forward stores are fenced for the async proxy (WB_RF); DH = 32 has no room for the
//   larger stages and loads h into registers before it waits for dh.
// Reference semantics: RealNVPLayer.f / .g (realnvp.py:73-129) looped as in nflow.py:109-115 / 142-143; MODE 2 is the
// autograd backward of loss = -nf.log_prob(X, C) (realnvp.py:246-250) up to the weight-gradient contraction.
#include <cuda_runtime.h>
#include <stdint.h>
#include "tc05.cuh"
#include "rnvp_wide.h"
#include "rnvp_philox.cuh"

namespace {
using namespace tc05;
#ifdef RNVP_SPLIT_RN
#define SPLIT_A split_tf32
#else
#define SPLIT_A split_tf32_raw_hi          // A operands (TMEM): see tc05.cuh
#endif

constexpr int WD_THREADS = 320;       // warp 0 TMA producer, warp 1 MMA issuer, warps 2-9 epilogue (TMEM lane quarter = warp % 4)
constexpr int WD_STAGES = 4;          // weight ring depth (chunk steps in flight)

template <int ACT>
__device__ __forceinline__ float act_wide(float v) {
  if (ACT == 1) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v));        // v = 2 log2(e) * pre-activation: the W1 image is pre-scaled (rnvp_planner.h)
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
  }
  return fmaxf(v, 0.0f);
}
// exp(x) = 2^(x*log2e) on the MUFU with the argument's rounding error compensated: t = rn(x*log2e), r = x*log2e - t
// (exact residual through FMA + the low part of log2e), exp = ex2(t)*(1 + r*ln2).  ~2 ulp in 6 instructions, against ~25 for expf()
__device__ __forceinline__ float exp_wide(float x) {
  const float t = x * 1.4426950216293335f;
  const float r = fmaf(x, 1.9259629911266175e-8f, fmaf(x, 1.4426950216293335f, -t));
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(t));
  return fmaf(e, r * 0.6931471805599453f, e);
}

// W consecutive TMEM columns of this thread's lane (W = 8 or 16)
template <int W>
__device__ __forceinline__ void tmem_ld_w(uint32_t taddr, uint32_t (&r)[W]) {
  if constexpr (W == 16) tmem_ld_x16(taddr, r);
  else tmem_ld_x8(taddr, r);
}

// barrier indices: ring full / empty first, then the tile hand-offs
enum { WB_WF = 0, WB_WE = WD_STAGES, WB_UF = 2 * WD_STAGES, WB_D1F0, WB_D1F1, WB_AF0, WB_AF1, WB_D2F, WB_XF, WB_XE, WB_COUNT };
// one more barrier where h rides in the ring: the tile's forward sweep has written all its activation records (the
// backward stages copy h out of them).  Appended, so that the layout of the other kernels stays as it is
constexpr int WB_RF = WB_COUNT;

// h rides in the backward ring stage (fit step): the stage carries the tile's h chunk next to the W2T / W1T images.  Not
// at DH = 32, whose two CTAs per SM cannot hold four 32 KB stages each; that shape loads h from the record into registers.
__host__ __device__ constexpr bool wide_hring(int DH, int mode) { return mode == 2 && DH != 32; }
// floats of one ring stage: forward [W1 chunk | W2 chunk | b2 of a net], backward [W2T chunk | W1T chunk (| h chunk)]
__host__ __device__ constexpr int wide_stage_floats(int DH, int CDMAX, int mode) {
  const int CU = 32, K1PMAX = (DH + CDMAX + 1 + 7) & ~7, NTP = (DH + 15) & ~15;
  const int fwd = 2 * CU * K1PMAX + 2 * NTP * CU + 2 * NTP * 8;
  const int bwd = 2 * (2 * NTP * CU) + (wide_hring(DH, mode) ? 128 * CU : 0);
  return ((fwd > bwd ? fwd : bwd) + 31) & ~31;
}

// DH <= 32: two CTAs per SM (256 TMEM columns each).  DH = 16 keeps the double-buffered D1 / dh chunk ring; DH = 32 only fits
// with ONE ring buffer (forward 240, backward 256 columns): the GEMM1 of the next chunk step is then issued behind this
// step's GEMM2 instead of ahead of it, and the second CTA on the SM fills the gap.
#ifndef RNVP_WIDE32_CTAS
#define RNVP_WIDE32_CTAS 2
#endif
template <int DH, int CDMAX, int CU, int ACT, int MODE>
__global__ void __launch_bounds__(WD_THREADS, DH == 16 ? 2 : (DH == 32 ? RNVP_WIDE32_CTAS : 1)) rnvp_wide_kernel(const __grid_constant__ RnvpWideArgs a) {
  constexpr int K1PMAX = (DH + CDMAX + 1 + 7) & ~7;
  constexpr int NTP = (DH + 15) & ~15;
  constexpr int NB1 = (DH == 32 && RNVP_WIDE32_CTAS == 2) ? 1 : 2;      // buffers of the D1 (forward) / dh (backward) chunk ring
  constexpr int HALF = DH / 2;                         // features of each parity class owned by one thread of a row pair
  // TMEM columns
  constexpr int U_HI = 0, U_LO = K1PMAX, D1B = 2 * K1PMAX;               // D1 ring: buffer b at D1B + b*2*CU: [D1/A_hi | A_lo]
  constexpr int D2C = D1B + 2 * NB1 * CU, C2C = D2C + NTP, TCOLS = C2C + NTP;
  static_assert(TCOLS <= 512, "TMEM budget");
  static_assert(DH % 16 == 0 && (K1PMAX - DH) % 8 == 0 && CU == 32, "layout assumptions");
  // backward sweep (MODE 2): delta2 hi / lo (2 DH columns each), the dh / delta1 chunk ring, the du accumulators [main | corr]
  constexpr int E2H = 0, E2L = 2 * DH, DHB = 4 * DH, DUM = DHB + 2 * NB1 * CU, DUC = DUM + NTP;
  static_assert(DUC + NTP <= 512, "TMEM budget (backward)");
  // D = 32 flows need 224 columns in either sweep: two CTAs share an SM (256 columns each, 80 registers per thread)
  constexpr int TALLOC = (TCOLS <= 256 && DUC + NTP <= 256) ? 256 : 512;
  constexpr int CW = HALF >= 16 ? 16 : 8;               // columns per coupling / gradient piece

  extern __shared__ __align__(128) float sm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = a.H, Cd = a.Cd, D = a.Dreal;           // D: features per row in memory; 2 * DH slots (padded shapes: D < 2 * DH)
  const bool exact = D == 2 * DH;
  const int NC = H / CU, NCS = 2 * NC;                  // chunk steps per layer: nn_t chunks, then nn_s chunks
  const int K1P = (DH + Cd + 1 + 7) & ~7;
  const int nL = a.l1 - a.l0;
  const int w1c = 2 * CU * K1P;                         // floats of one W1 chunk image [hi | lo]
  constexpr int W2C = 2 * NTP * CU, B2C = 2 * NTP * 8;  // W2 chunk image [hi | lo]; b2 image of one net [hi | lo]
  constexpr bool HRING = wide_hring(DH, MODE);
  constexpr int stage_floats = wide_stage_floats(DH, CDMAX, MODE);
  constexpr int HCH = 2 * W2C;                          // h chunk of a backward stage: [record block q][8 column groups][32][4]
  const bool do_bwd = MODE == 2 && a.do_bwd;
  const int n_sweeps = do_bwd ? 2 : 1;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + WD_STAGES * stage_floats);
  float* xch = reinterpret_cast<float*>(bars + WB_COUNT + (HRING ? 1 : 0));   // [128][2]: partial (logdet, |z|^2) of the second half-thread
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xch + 256);

  if (warp == 1) tmem_alloc(tmem_slot, TALLOC);
  if (tid == 0) {
    for (int s = 0; s < WD_STAGES; ++s) { mbar_init(&bars[WB_WF + s], 1); mbar_init(&bars[WB_WE + s], 1); }
    mbar_init(&bars[WB_UF], 256);
    mbar_init(&bars[WB_D1F0], 1); mbar_init(&bars[WB_D1F1], 1);
    mbar_init(&bars[WB_AF0], 256); mbar_init(&bars[WB_AF1], 256);
    mbar_init(&bars[WB_D2F], 1);
    mbar_init(&bars[WB_XF], 128); mbar_init(&bars[WB_XE], 128);       // row-pair exchange of the partial log-dets / norms
    if (HRING) mbar_init(&bars[WB_RF], 256);
    mbar_fence_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = *tmem_slot;
  const int my_tiles = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer: one ring stage per chunk step
    if (lane == 0) {
      long long step = 0;
      const uint32_t w1c_bytes = (uint32_t)w1c * 4u, w2c_bytes = (uint32_t)W2C * 4u, b2_bytes = (uint32_t)B2C * 4u;
      constexpr uint32_t h_bytes = HRING ? 128u * CU * 4u : 0u;
      // h chunk of backward chunk step cc of layer i into ring stage st: columns [col0, col0 + CU) of the tile's four 32-row
      // record blocks, one contiguous 4 KB range each (rnvp_wgrad_tc.cu layout), kept in the record's slot order
      auto copy_h = [&](int st, long long tile, int i, int cc) {
        const int net = cc >= NC ? 1 : 0, col0 = net * H + (cc - net * NC) * CU;
        const size_t blk = (size_t)(a.rec >> 2) * 128;
        const float* src = a.records + ((size_t)i * (size_t)(a.Npad >> 5) + (size_t)tile * 4) * blk + (size_t)(col0 >> 2) * 128;
        float* dst = sm + (size_t)st * stage_floats + HCH;
#pragma unroll
        for (int q = 0; q < 4; ++q) bulk_g2s(dst + q * CU * 32, src + q * blk, CU * 32 * 4u, &bars[WB_WF + st]);
      };
      for (int it = 0; it < my_tiles; ++it)
        for (int sw = 0; sw < n_sweeps; ++sw)
          for (int li = 0; li < nL; ++li) {
            const int i = (MODE == 1 || sw == 1) ? a.l1 - 1 - li : a.l0 + li;
            const float* L0 = a.wimg + (size_t)i * a.layer_floats;
            const float* W2 = L0 + a.w1_floats;
            const float* B2 = W2 + (size_t)4 * NTP * H;
            const float* W2T = W2 + a.w2_floats;                   // streamed backward images: [cc][hi | lo][CU x NTP]
            const float* W1T = W2T + a.wt_floats;                  //                           [cc][hi | lo][NTP x CU]
            for (int cc = 0; cc < NCS; ++cc, ++step) {
              const int st = (int)(step % WD_STAGES);
              if (step >= WD_STAGES) mbar_wait_relaxed(&bars[WB_WE + st], (uint32_t)((step / WD_STAGES - 1) & 1));
              const int net = cc >= NC ? 1 : 0, c = cc - net * NC;
              float* dst = sm + (size_t)st * stage_floats;
              if (sw == 0) {
                const bool with_b2 = c == 0;
                mbar_expect_tx(&bars[WB_WF + st], w1c_bytes + w2c_bytes + (with_b2 ? b2_bytes : 0u));
                bulk_g2s(dst, L0 + (size_t)cc * w1c, w1c_bytes, &bars[WB_WF + st]);
                bulk_g2s(dst + 2 * CU * K1PMAX, W2 + (size_t)(c * 2 + net) * W2C, w2c_bytes, &bars[WB_WF + st]);
                if (with_b2) bulk_g2s(dst + 2 * CU * K1PMAX + W2C, B2 + (size_t)net * B2C, b2_bytes, &bars[WB_WF + st]);
              } else {
                mbar_expect_tx(&bars[WB_WF + st], 2 * w2c_bytes + h_bytes);
                bulk_g2s(dst, W2T + (size_t)cc * W2C, w2c_bytes, &bars[WB_WF + st]);
                bulk_g2s(dst + W2C, W1T + (size_t)cc * W2C, w2c_bytes, &bars[WB_WF + st]);
                if constexpr (HRING) {
                  // the forward sweep wrote h with generic stores: the async-proxy copies wait for WB_RF.  The first
                  // stages of the sweep get their images at once (they are armed for the h bytes too) and their h once
                  // the forward sweep is done, so the turn from forward to backward does not wait for the images
                  const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
                  const int k = li * NCS + cc, k_first = nL * NCS < WD_STAGES ? nL * NCS : WD_STAGES;
                  if (k >= k_first) copy_h(st, tile, i, cc);
                  else if (k + 1 == k_first) {
                    mbar_wait(&bars[WB_RF], (uint32_t)(it & 1));
                    for (int k0 = 0; k0 < k_first; ++k0)
                      copy_h((int)((step - k + k0) % WD_STAGES), tile, a.l1 - 1 - k0 / NCS, k0 % NCS);
                  }
                }
              }
            }
          }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const bool leader = elect_one();
    const uint32_t idesc1 = idesc_tf32(128, CU), idesc2 = idesc_tf32(128, NTP), idesc2m = idesc_tf32(128, 2 * NTP);
    const uint32_t lbo = (128u >> 4) << 16;
    const uint32_t hi1 = ((uint32_t)(K1P >> 2) * 128u >> 4) | (1u << 14);       // SBO of the W1 chunk image, descriptor version 1
    const uint32_t hi2 = ((uint32_t)(CU >> 2) * 128u >> 4) | (1u << 14);        // W2 chunk image: [NTP (x2) rows x CU]
    const uint32_t hib = (256u >> 4) | (1u << 14);                              // b2 image: K = 8
    const uint32_t chunk1 = (uint32_t)(CU * K1P) * 4u >> 4;                     // one hi (or lo) W1 chunk, 16 B units
    const int nk1 = K1P >> 3;
    const int k_one = (DH + Cd) & ~7;                                           // u slice holding the constant one
    auto desc = [](uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; };
    const uint32_t sm_lo = ((smem_u32(sm) & 0x3FFFFu) >> 4) | lbo;
    const uint32_t stage16 = (uint32_t)stage_floats * 4u >> 4;
    // GEMM1 of a chunk step into D1 buffer `buf`: [u_lo W1_hi + u_hi W1_lo] + u_hi W1_hi (corrections first)
    auto gemm1 = [&](int st, int buf) {
      const uint32_t bh = sm_lo + (uint32_t)st * stage16, bl = bh + chunk1;
      const uint32_t d = tbase + D1B + buf * 2 * CU;
#pragma unroll
      for (int j = 0; j < K1PMAX / 8; ++j)
        if (j < nk1) mma_tf32_ts(d, tbase + U_LO + 8 * j, desc(bh + 16u * j, hi1), idesc1, j ? 1u : 0u);
#pragma unroll
      for (int j = 0; j < K1PMAX / 8; ++j)
        if (j < nk1) mma_tf32_ts(d, tbase + U_HI + 8 * j, desc(bl + 16u * j, hi1), idesc1, 1u);
#pragma unroll
      for (int j = 0; j < K1PMAX / 8; ++j)
        if (j < nk1) mma_tf32_ts(d, tbase + U_HI + 8 * j, desc(bh + 16u * j, hi1), idesc1, 1u);
    };
    // GEMM2 of chunk c of a net: [D2 | C2] (+)= A_hi x [W2_hi ; W2_lo]  (one MMA of N = 2 NTP), C2 += A_lo x W2_hi; the first
    // chunk seeds [D2 | C2] with 1 x [b2_hi ; b2_lo]
    auto gemm2 = [&](int st, int buf, int c) {
      const uint32_t w2 = sm_lo + (uint32_t)st * stage16 + ((uint32_t)(2 * CU * K1PMAX) * 4u >> 4);
      const uint32_t b2 = w2 + ((uint32_t)W2C * 4u >> 4);
      const uint32_t ah = tbase + D1B + buf * 2 * CU, al = ah + CU;
      if (c == 0) mma_tf32_ts(tbase + D2C, tbase + U_HI + k_one, desc(b2, hib), idesc2m, 0u);
#pragma unroll
      for (int j = 0; j < CU / 8; ++j) mma_tf32_ts(tbase + C2C, al + 8 * j, desc(w2 + 16u * j, hi2), idesc2, 1u);
#pragma unroll
      for (int j = 0; j < CU / 8; ++j) mma_tf32_ts(tbase + D2C, ah + 8 * j, desc(w2 + 16u * j, hi2), idesc2m, 1u);
    };
    // backward sweep (MODE 2).  gemmA: dh chunk = delta2_net W2_net[:, chunk]  (A = delta2 hi / lo in TMEM, B = W2T chunk image
    // [CU units x NTP]); gemmB: [DUM | DUC] += delta1 x [W1T_hi ; W1T_lo], DUC += delta1_lo x W1T_hi (B = W1T chunk image
    // [NTP x CU], the same shape as the forward W2 chunk)
    const uint32_t hiT = ((uint32_t)(NTP >> 2) * 128u >> 4) | (1u << 14);       // SBO of the W2T chunk image (K = NTP)
    auto gemmA = [&](int st, int buf, int net) {
      const uint32_t bh = sm_lo + (uint32_t)st * stage16, bl = bh + ((uint32_t)(CU * NTP) * 4u >> 4);
      const uint32_t d = tbase + DHB + buf * 2 * CU;
      const uint32_t eh = tbase + E2H + net * DH, el = tbase + E2L + net * DH;
#pragma unroll
      for (int j = 0; j < DH / 8; ++j) mma_tf32_ts(d, el + 8 * j, desc(bh + 16u * j, hiT), idesc1, j ? 1u : 0u);
#pragma unroll
      for (int j = 0; j < DH / 8; ++j) mma_tf32_ts(d, eh + 8 * j, desc(bl + 16u * j, hiT), idesc1, 1u);
#pragma unroll
      for (int j = 0; j < DH / 8; ++j) mma_tf32_ts(d, eh + 8 * j, desc(bh + 16u * j, hiT), idesc1, 1u);
    };
    auto gemmB = [&](int st, int buf, int cc) {
      const uint32_t w1t = sm_lo + (uint32_t)st * stage16 + ((uint32_t)W2C * 4u >> 4);
      const uint32_t ah = tbase + DHB + buf * 2 * CU, al = ah + CU;
#pragma unroll
      for (int j = 0; j < CU / 8; ++j) mma_tf32_ts(tbase + DUM, ah + 8 * j, desc(w1t + 16u * j, hi2), idesc2m, (cc | j) ? 1u : 0u);
#pragma unroll
      for (int j = 0; j < CU / 8; ++j) mma_tf32_ts(tbase + DUC, al + 8 * j, desc(w1t + 16u * j, hi2), idesc2, 1u);
    };
    uint32_t ph_u = 0, ph_a = 0, ph_w = 0;              // ph_a / ph_w: one bit per buffer / stage
    long long step = 0;
    for (int it = 0; it < my_tiles; ++it) {
      for (int li = 0; li < nL; ++li) {
        mbar_wait(&bars[WB_UF], ph_u); ph_u ^= 1;
        {
          const int st = (int)(step % WD_STAGES);
          mbar_wait(&bars[WB_WF + st], (ph_w >> st) & 1u); ph_w ^= 1u << st;
          fence_after_sync();
          if (leader) { gemm1(st, 0); mma_commit(&bars[WB_D1F0]); }
          __syncwarp();
        }
        for (int cc = 0; cc < NCS; ++cc, ++step) {
          const int st = (int)(step % WD_STAGES), buf = cc & (NB1 - 1);
          auto next_gemm1 = [&]() {           // GEMM1 of chunk step cc + 1 into the other (NB1 = 2) or the same (NB1 = 1) buffer
            const int st1 = (int)((step + 1) % WD_STAGES), nb = (cc + 1) & (NB1 - 1);
            mbar_wait(&bars[WB_WF + st1], (ph_w >> st1) & 1u); ph_w ^= 1u << st1;
            fence_after_sync();
            if (leader) { gemm1(st1, nb); mma_commit(&bars[WB_D1F0 + nb]); }
            __syncwarp();
          };
          // two buffers: the next chunk's GEMM1 first, the tensor core stays busy during this chunk's epilogue
          if (NB1 == 2 && cc + 1 < NCS) next_gemm1();
          mbar_wait(&bars[WB_AF0 + buf], (ph_a >> buf) & 1u); ph_a ^= 1u << buf;
          fence_after_sync();
          if (leader) {
            const int net = cc >= NC ? 1 : 0;
            gemm2(st, buf, cc - net * NC);
            mma_commit(&bars[WB_WE + st]);                       // both GEMMs that read this ring stage are issued
            if (cc + 1 == NC || cc + 1 == NCS) mma_commit(&bars[WB_D2F]);
          }
          __syncwarp();
          // one buffer: the next GEMM1 overwrites the A operand this GEMM2 reads -- issued behind it (MMAs execute in order)
          if (NB1 == 1 && cc + 1 < NCS) next_gemm1();
        }
      }
      if (do_bwd) {
        for (int li = 0; li < nL; ++li) {
          mbar_wait(&bars[WB_UF], ph_u); ph_u ^= 1;           // delta2 of the layer staged in TMEM
          {
            const int st = (int)(step % WD_STAGES);
            mbar_wait(&bars[WB_WF + st], (ph_w >> st) & 1u); ph_w ^= 1u << st;
            fence_after_sync();
            if (leader) { gemmA(st, 0, 0); mma_commit(&bars[WB_D1F0]); }
            __syncwarp();
          }
          for (int cc = 0; cc < NCS; ++cc, ++step) {
            const int st = (int)(step % WD_STAGES), buf = cc & (NB1 - 1);
            auto next_gemmA = [&]() {
              const int st1 = (int)((step + 1) % WD_STAGES), nb = (cc + 1) & (NB1 - 1);
              mbar_wait(&bars[WB_WF + st1], (ph_w >> st1) & 1u); ph_w ^= 1u << st1;
              fence_after_sync();
              if (leader) { gemmA(st1, nb, (cc + 1) >= NC ? 1 : 0); mma_commit(&bars[WB_D1F0 + nb]); }
              __syncwarp();
            };
            if (NB1 == 2 && cc + 1 < NCS) next_gemmA();
            mbar_wait(&bars[WB_AF0 + buf], (ph_a >> buf) & 1u); ph_a ^= 1u << buf;
            fence_after_sync();
            if (leader) {
              gemmB(st, buf, cc);
              mma_commit(&bars[WB_WE + st]);
              if (cc + 1 == NCS) mma_commit(&bars[WB_D2F]);       // du of the layer complete
            }
            __syncwarp();
            if (NB1 == 1 && cc + 1 < NCS) next_gemmA();
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: two threads per row
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const uint32_t trow = tbase + ((uint32_t)(quarter * 32) << 16);
    const int rin = quarter * 32 + lane;                 // row inside the tile
    uint32_t ph_d1 = 0, ph_d2 = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const long long tile = (long long)blockIdx.x + (long long)it * gridDim.x;
      const long long row = tile * 128 + rin;
      const bool valid = row < a.N;
      const long long src = valid ? (a.idx ? a.idx[row] : row) : 0;
      // this thread's features: [half*DH, (half+1)*DH) of the row = HALF even-indexed (xa) and HALF odd-indexed (xb) ones
      float xa[HALF], xb[HALF], ld = 0.0f;
#pragma unroll
      for (int m = 0; m < HALF / 2; ++m) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        const int j0 = half * DH + 4 * m;                 // first of this float4's feature slots
        if (MODE == 1 && a.X == nullptr) { if (valid && j0 < D) v = rnvp_rng::normal4(a.seed, a.row_offset + row, half * (DH / 4) + m); }
        else if (valid && exact) v = __ldg(reinterpret_cast<const float4*>(a.X + src * D + half * DH) + m);
        else if (valid) {                                 // padded shape: row stride D, scalar guarded loads
          const float* xr = a.X + src * D;
          v.x = j0 + 0 < D ? __ldg(xr + j0 + 0) : 0.f; v.y = j0 + 1 < D ? __ldg(xr + j0 + 1) : 0.f;
          v.z = j0 + 2 < D ? __ldg(xr + j0 + 2) : 0.f; v.w = j0 + 3 < D ? __ldg(xr + j0 + 3) : 0.f;
        }
        if (!exact) {                                     // slots beyond the row stay exactly zero (their weights are zero too)
          if (j0 + 0 >= D) v.x = 0.f;
          if (j0 + 1 >= D) v.y = 0.f;
          if (j0 + 2 >= D) v.z = 0.f;
          if (j0 + 3 >= D) v.w = 0.f;
        }
        xa[2 * m] = v.x; xb[2 * m] = v.y; xa[2 * m + 1] = v.z; xb[2 * m + 1] = v.w;
      }
      // activation records of (layer i, this row): [layer][block of 32 rows][column group of 4][32 slots][4 floats], slot =
      // (row % 32) ^ (group & 7) (rnvp_wgrad_tc.cu): a warp-level float4 access covers 512 contiguous bytes
      const int K1P8 = (DH + Cd + 7) & ~7;
      auto rec_base = [&](int i) -> float* {
        return a.records + (((size_t)i * (size_t)(a.Npad >> 5) + (size_t)(row >> 5)) * (size_t)(a.rec >> 2)) * 128;
      };
      auto rec_st = [&](float* rb, int col, float4 v) {
        const int cg = col >> 2;
        *reinterpret_cast<float4*>(rb + cg * 128 + ((lane ^ (cg & 7)) << 2)) = v;
      };
      // forward stash of this kernel's own backward sweep: [block of 32 rows][layer][float4 group (2 DH / 4)][32 rows][4]
      auto stash_ptr = [&](int i, int group) -> float* {
        return a.stash + (((size_t)(row >> 5) * a.L_total + i) * (2 * DH / 4) + group) * 128 + lane * 4;
      };
      // static part of u: [c | 1 | 0...] at columns DH.. of U_HI / U_LO, written once per tile; the 8-column pieces are
      // shared out between the two threads of the row
#pragma unroll
      for (int e0 = 0; e0 < K1PMAX - DH; e0 += 8) {
        if (((e0 >> 3) & 1) == half) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int k = e0 + j;
            float v = 0.0f;
            if (k < Cd && valid) v = __ldg(a.C + src * Cd + k);
            if (k == Cd) v = 1.0f;
            split_tf32(v, hi[j], lo[j]);          // u (24-48 values per row-layer): the fully rounded split
          }
          tmem_st_x8(trow + U_HI + DH + e0, hi);
          tmem_st_x8(trow + U_LO + DH + e0, lo);
          if (MODE == 2 && do_bwd && DH + e0 < K1P8) {
            // the condition part of u = [x_K, c] is the same for every layer: written into all records of the row now
            float4 c0, c1;
            c0.x = (e0 + 0 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 0) : 0.f; c0.y = (e0 + 1 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 1) : 0.f;
            c0.z = (e0 + 2 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 2) : 0.f; c0.w = (e0 + 3 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 3) : 0.f;
            c1.x = (e0 + 4 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 4) : 0.f; c1.y = (e0 + 5 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 5) : 0.f;
            c1.z = (e0 + 6 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 6) : 0.f; c1.w = (e0 + 7 < Cd && valid) ? __ldg(a.C + src * Cd + e0 + 7) : 0.f;
            for (int i = a.l0; i < a.l1; ++i) {
              rec_st(rec_base(i), 2 * H + DH + e0, c0);
              rec_st(rec_base(i), 2 * H + DH + e0 + 4, c1);
            }
          }
        }
      }

      auto layer = [&](float (&xT)[HALF], float (&xK)[HALF], int i) {
        // ---- this thread's half of the conditioning features -> u (hi / lo) in TMEM
#pragma unroll
        for (int e0 = 0; e0 < HALF; e0 += 8) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) split_tf32(xK[e0 + j], hi[j], lo[j]);
          tmem_st_x8(trow + U_HI + half * HALF + e0, hi);
          tmem_st_x8(trow + U_LO + half * HALF + e0, lo);
        }
        tmem_wait_st();
        fence_before_sync();
        mbar_arrive(&bars[WB_UF]);
        if (MODE == 2 && do_bwd) {               // x_K half of u -> record (the weight-gradient sweep contracts it with delta1)
          float* rb = rec_base(i);
#pragma unroll
          for (int m = 0; m < HALF / 4; ++m)
            rec_st(rb, 2 * H + half * HALF + 4 * m, make_float4(xK[4 * m], xK[4 * m + 1], xK[4 * m + 2], xK[4 * m + 3]));
        }
        float tpark[HALF];
        for (int cc = 0; cc < NCS; ++cc) {
          const int buf = cc & (NB1 - 1);
          mbar_wait(&bars[WB_D1F0 + buf], (ph_d1 >> buf) & 1u); ph_d1 ^= 1u << buf;
          fence_after_sync();
          {
            // this thread's 16 columns of the chunk: D1 -> act -> A_hi (in place), A_lo
            const uint32_t d1 = trow + D1B + buf * 2 * CU + 16 * half;
            uint32_t r[16], lo[16];
            tmem_ld_x16(d1, r);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 16; ++j) r[j] = __float_as_uint(act_wide<ACT>(__uint_as_float(r[j])));
            if (MODE == 2 && do_bwd) {
              // h goes to the activation record now: the backward sweep and the weight-gradient sweep read it back.  Chunk
              // step cc holds units (cc % NC) * CU .. of net cc / NC; this thread has columns 16 * half .. of the chunk
              const int net = cc >= NC ? 1 : 0;
              float* rb = rec_base(i);
              const int col0 = net * H + (cc - net * NC) * CU + 16 * half;
#pragma unroll
              for (int m = 0; m < 4; ++m)
                rec_st(rb, col0 + 4 * m, make_float4(__uint_as_float(r[4 * m]), __uint_as_float(r[4 * m + 1]),
                                                     __uint_as_float(r[4 * m + 2]), __uint_as_float(r[4 * m + 3])));
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) SPLIT_A(__uint_as_float(r[j]), r[j], lo[j]);
            tmem_st_x16(d1, r);
            tmem_st_x16(d1 + CU, lo);
          }
          tmem_wait_st();
          fence_before_sync();
          mbar_arrive(&bars[WB_AF0 + buf]);
          if (cc + 1 == NC) {                    // nn_t complete: t = D2 + C2 into registers (the nn_s GEMM2 overwrites them)
            mbar_wait(&bars[WB_D2F], ph_d2); ph_d2 ^= 1;
            fence_after_sync();
#pragma unroll
            for (int e0 = 0; e0 < HALF; e0 += CW) {
              uint32_t tv[CW], tc[CW];
              tmem_ld_w<CW>(trow + D2C + half * HALF + e0, tv);
              tmem_ld_w<CW>(trow + C2C + half * HALF + e0, tc);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < CW; ++j) tpark[e0 + j] = __uint_as_float(tv[j]) + __uint_as_float(tc[j]);
            }
            fence_before_sync();                 // ordered before this thread's next a_full arrival, which releases D2 / C2
          }
        }
        // ---- s complete -> coupling on this thread's transformed features
        mbar_wait(&bars[WB_D2F], ph_d2); ph_d2 ^= 1;
        fence_after_sync();
#pragma unroll
        for (int e0 = 0; e0 < HALF; e0 += CW) {
          uint32_t sv[CW], sc[CW];
          tmem_ld_w<CW>(trow + D2C + half * HALF + e0, sv);
          tmem_ld_w<CW>(trow + C2C + half * HALF + e0, sc);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < CW; ++j) {
            const float s = __uint_as_float(sv[j]) + __uint_as_float(sc[j]);
            const float t = tpark[e0 + j];
            if (MODE == 2) { sv[j] = __float_as_uint(s); sc[j] = __float_as_uint(xT[e0 + j]); }      // stash s and x_T
            if (MODE != 1) { xT[e0 + j] = fmaf(xT[e0 + j], exp_wide(s), t); ld += s; }
            else xT[e0 + j] = (xT[e0 + j] - t) * exp_wide(-s);
          }
          if (MODE == 2 && do_bwd) {
#pragma unroll
            for (int m = 0; m < CW / 4; ++m) {
              *reinterpret_cast<float4*>(stash_ptr(i, (half * HALF + e0) / 4 + m)) =
                  make_float4(__uint_as_float(sc[4 * m]), __uint_as_float(sc[4 * m + 1]), __uint_as_float(sc[4 * m + 2]),
                              __uint_as_float(sc[4 * m + 3]));
              *reinterpret_cast<float4*>(stash_ptr(i, DH / 4 + (half * HALF + e0) / 4 + m)) =
                  make_float4(__uint_as_float(sv[4 * m]), __uint_as_float(sv[4 * m + 1]), __uint_as_float(sv[4 * m + 2]),
                              __uint_as_float(sv[4 * m + 3]));
            }
          }
        }
        fence_before_sync();                     // the next layer's first GEMM2 (after the next a_full) overwrites D2 / C2
      };
      for (int li = 0; li < nL; ++li) {
        const int i = MODE != 1 ? a.l0 + li : a.l1 - 1 - li;
        if ((i & 1) == 0) layer(xa, xb, i);              // even layer transforms the even features
        else layer(xb, xa, i);
      }
      if (HRING && do_bwd) {
        // this thread's h record stores of the tile, ordered before the producer's async-proxy copies of them
        asm volatile("fence.proxy.async.global;" ::: "memory");
        mbar_arrive(&bars[WB_RF]);
      }

      if (valid && a.out_x) {
        if (exact) {
#pragma unroll
          for (int m = 0; m < HALF / 2; ++m)
            reinterpret_cast<float4*>(a.out_x + row * D + half * DH)[m] = make_float4(xa[2 * m], xb[2 * m], xa[2 * m + 1], xb[2 * m + 1]);
        } else {
          float* orow = a.out_x + row * D;
#pragma unroll
          for (int m = 0; m < HALF / 2; ++m) {
            const int j0 = half * DH + 4 * m;
            if (j0 + 0 < D) orow[j0 + 0] = xa[2 * m];
            if (j0 + 1 < D) orow[j0 + 1] = xb[2 * m];
            if (j0 + 2 < D) orow[j0 + 2] = xa[2 * m + 1];
            if (j0 + 3 < D) orow[j0 + 3] = xb[2 * m + 1];
          }
        }
      }
      if (MODE != 1) {
        float q = 0.0f;
#pragma unroll
        for (int e = 0; e < HALF; ++e) { q = fmaf(xa[e], xa[e], q); q = fmaf(xb[e], xb[e], q); }
        // the second thread of the row hands its partial sums to the first
        float lp = 0.0f;
        if (half == 1) {
          if (it > 0) mbar_wait(&bars[WB_XE], (uint32_t)((it - 1) & 1));          // the first threads have read the previous tile's sums
          xch[2 * rin] = ld; xch[2 * rin + 1] = q;
          mbar_arrive(&bars[WB_XF]);
        } else {
          mbar_wait(&bars[WB_XF], (uint32_t)(it & 1));
          const float ldt = ld + xch[2 * rin], qt = q + xch[2 * rin + 1];
          mbar_arrive(&bars[WB_XE]);
          if (valid) {
            lp = ldt - 0.5f * (D * 1.8378770664093453f + qt);
            if (a.out_logdet) a.out_logdet[row] = ldt;
            if (a.out_logp) a.out_logp[row] = lp;
          }
        }
        if (MODE == 2 && a.loss_sum && half == 0) {
#pragma unroll
          for (int m = 16; m >= 1; m >>= 1) lp += __shfl_xor_sync(0xffffffffu, lp, m);
          if (lane == 0) atomicAdd(a.loss_sum, lp);
        }
      }

      // ================================================================ backward sweep (fit step)
      if constexpr (MODE == 2) {
        if (do_bwd) {
          // gradient of scale * sum_rows logp w.r.t. the current activations: g_z = -scale * z, g_logdet = scale
          const float gld = valid ? a.scale : 0.0f;
          float ga[HALF], gb[HALF];
#pragma unroll
          for (int e = 0; e < HALF; ++e) { ga[e] = -gld * xa[e]; gb[e] = -gld * xb[e]; }
          auto layer_bwd = [&](float (&gT)[HALF], float (&gK)[HALF], int i) {
            float* rb = rec_base(i);
            if (i > a.l0) {       // the next layer's stash block of this thread's rows: pull it into L2 now
#pragma unroll
              for (int m = 0; m < HALF / 4; ++m) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(stash_ptr(i - 1, half * HALF / 4 + m)));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(stash_ptr(i - 1, DH / 4 + half * HALF / 4 + m)));
              }
            }
            // ---- x_T and s of this layer from the forward stash; delta2 (hi / lo) -> TMEM and -> record; new g_T
#pragma unroll
            for (int e0 = 0; e0 < HALF; e0 += 8) {
              uint32_t th[8], tl[8], sh[8], sl[8];
              float d2t[8], d2s[8];
#pragma unroll
              for (int m = 0; m < 2; ++m) {
                const float4 xv = *reinterpret_cast<const float4*>(stash_ptr(i, (half * HALF + e0) / 4 + m));
                const float4 sv = *reinterpret_cast<const float4*>(stash_ptr(i, DH / 4 + (half * HALF + e0) / 4 + m));
                const float xs4[4] = {xv.x, xv.y, xv.z, xv.w}, ss4[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
                for (int q2 = 0; q2 < 4; ++q2) {
                  const int e = e0 + 4 * m + q2;
                  const float es = exp_wide(ss4[q2]);
                  d2t[4 * m + q2] = gT[e];                                   // dL/dt
                  d2s[4 * m + q2] = fmaf(gT[e] * xs4[q2], es, gld);          // dL/ds = g_y * x * exp(s) + g_logdet
                  gT[e] *= es;                                               // dL/dx_T
                  SPLIT_A(d2t[4 * m + q2], th[4 * m + q2], tl[4 * m + q2]);
                  SPLIT_A(d2s[4 * m + q2], sh[4 * m + q2], sl[4 * m + q2]);
                }
              }
              tmem_st_x8(trow + E2H + half * HALF + e0, th);
              tmem_st_x8(trow + E2L + half * HALF + e0, tl);
              tmem_st_x8(trow + E2H + DH + half * HALF + e0, sh);
              tmem_st_x8(trow + E2L + DH + half * HALF + e0, sl);
              rec_st(rb, 2 * H + K1P8 + half * HALF + e0, make_float4(d2t[0], d2t[1], d2t[2], d2t[3]));
              rec_st(rb, 2 * H + K1P8 + half * HALF + e0 + 4, make_float4(d2t[4], d2t[5], d2t[6], d2t[7]));
              rec_st(rb, 2 * H + K1P8 + DH + half * HALF + e0, make_float4(d2s[0], d2s[1], d2s[2], d2s[3]));
              rec_st(rb, 2 * H + K1P8 + DH + half * HALF + e0 + 4, make_float4(d2s[4], d2s[5], d2s[6], d2s[7]));
            }
            tmem_wait_st();
            fence_before_sync();
            mbar_arrive(&bars[WB_UF]);
            // ---- chunk steps: delta1 = dh * act'(h), dh from the tensor core, h from the record the forward sweep wrote
            // ring step of chunk step 0, modulo 2^32: only its stage and phase (step % 2 WD_STAGES) are used
            const uint32_t step0 = ((uint32_t)(2 * it + 1) * (uint32_t)nL + (uint32_t)(a.l1 - 1 - i)) * (uint32_t)NCS;
            for (int cc = 0; cc < NCS; ++cc) {
              const int buf = cc & (NB1 - 1), net = cc >= NC ? 1 : 0;
              const int col0 = net * H + (cc - net * NC) * CU + 16 * half;
              uint32_t hv[16];
              if constexpr (!HRING) {
#pragma unroll
                for (int m = 0; m < 4; ++m) {         // issued before the wait for dh: the L2 / HBM latency hides behind the MMAs
                  const int cg = (col0 >> 2) + m;
                  const float4 v = *reinterpret_cast<const float4*>(rb + cg * 128 + ((lane ^ (cg & 7)) << 2));
                  hv[4 * m] = __float_as_uint(v.x); hv[4 * m + 1] = __float_as_uint(v.y);
                  hv[4 * m + 2] = __float_as_uint(v.z); hv[4 * m + 3] = __float_as_uint(v.w);
                }
              }
              mbar_wait(&bars[WB_D1F0 + buf], (ph_d1 >> buf) & 1u); ph_d1 ^= 1u << buf;
              fence_after_sync();
              if constexpr (HRING) {
                // h from the ring stage of this chunk step (already full: its gemmA has completed).  The stage is not
                // refilled under these reads: they complete before this thread's WB_AF arrival below, the issuer commits
                // the stage's WB_WE only behind the gemmB that waits for that arrival, and the producer refills the stage
                // only after WB_WE
                const uint32_t s = step0 + (uint32_t)cc;
                const int st = (int)(s % WD_STAGES);
                mbar_wait(&bars[WB_WF + st], (uint32_t)((s / WD_STAGES) & 1));
                const float* hs = sm + (size_t)st * stage_floats + HCH + quarter * (CU * 32);
#pragma unroll
                for (int m = 0; m < 4; ++m) {         // same slot order as the record: conflict-free 512-byte warp reads
                  const int cg = (col0 >> 2) + m;
                  const float4 v = *reinterpret_cast<const float4*>(hs + (cg & 7) * 128 + ((lane ^ (cg & 7)) << 2));
                  hv[4 * m] = __float_as_uint(v.x); hv[4 * m + 1] = __float_as_uint(v.y);
                  hv[4 * m + 2] = __float_as_uint(v.z); hv[4 * m + 3] = __float_as_uint(v.w);
                }
              }
              const uint32_t d1 = trow + DHB + buf * 2 * CU + 16 * half;
              uint32_t dh[16], lo[16];
              tmem_ld_x16(d1, dh);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float h = __uint_as_float(hv[j]);
                const float dp = ACT == 1 ? fmaf(-h, h, 1.0f) : (h > 0.0f ? 1.0f : 0.0f);
                SPLIT_A(__uint_as_float(dh[j]) * dp, dh[j], lo[j]);
              }
              tmem_st_x16(d1, dh);
              tmem_st_x16(d1 + CU, lo);
              tmem_wait_st();
              fence_before_sync();
              mbar_arrive(&bars[WB_AF0 + buf]);
            }
            // ---- du -> g_x_K (this thread's half of the conditioning features)
            mbar_wait(&bars[WB_D2F], ph_d2); ph_d2 ^= 1;
            fence_after_sync();
#pragma unroll
            for (int e0 = 0; e0 < HALF; e0 += CW) {
              uint32_t um[CW], uc[CW];
              tmem_ld_w<CW>(trow + DUM + half * HALF + e0, um);
              tmem_ld_w<CW>(trow + DUC + half * HALF + e0, uc);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < CW; ++j) gK[e0 + j] += __uint_as_float(um[j]) + __uint_as_float(uc[j]);
            }
            fence_before_sync();
          };
          for (int li = 0; li < nL; ++li) {
            const int i = a.l1 - 1 - li;
            if ((i & 1) == 0) layer_bwd(ga, gb, i);
            else layer_bwd(gb, ga, i);
          }
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tbase, TALLOC);
}

template <int DH, int CDMAX>
cudaError_t launch_wide_shape(int act, int mode, const RnvpWideArgs& a, int grid, size_t smem, cudaStream_t st) {
#define RNVP_WIDE_LAUNCH(ACT_, MODE_)                                                                       \
  {                                                                                                          \
    auto k = rnvp_wide_kernel<DH, CDMAX, 32, ACT_, MODE_>;                                                   \
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);         \
    if (e != cudaSuccess) return e;                                                                          \
    k<<<grid, WD_THREADS, smem, st>>>(a);                                                                    \
    return cudaGetLastError();                                                                               \
  }
  if (act == 1 && mode == 0) RNVP_WIDE_LAUNCH(1, 0)
  if (act == 1 && mode == 1) RNVP_WIDE_LAUNCH(1, 1)
  if (act == 1 && mode == 2) RNVP_WIDE_LAUNCH(1, 2)
  if (act == 2 && mode == 0) RNVP_WIDE_LAUNCH(2, 0)
  if (act == 2 && mode == 1) RNVP_WIDE_LAUNCH(2, 1)
  if (act == 2 && mode == 2) RNVP_WIDE_LAUNCH(2, 2)
#undef RNVP_WIDE_LAUNCH
  return cudaErrorInvalidValue;
}

}  // namespace

// the fit step (mode 2) of DH = 16 / 64 has the larger backward stages that carry h; log-prob and sample keep the smaller ones
size_t rnvp_wide_smem_bytes(int DH, int CDMAX, int mode) {
  return WD_STAGES * (size_t)wide_stage_floats(DH, CDMAX, mode) * 4 + 8 * (WB_COUNT + (wide_hring(DH, mode) ? 1 : 0)) +
         256 * 4 + 64;
}

int rnvp_wide_ctas_per_sm(int DH) { return DH == 16 ? 2 : (DH == 32 ? RNVP_WIDE32_CTAS : 1); }

cudaError_t rnvp_launch_wide(int DH, int act, int mode, const RnvpWideArgs& a, int grid, cudaStream_t st) {
  if (DH == 64) return launch_wide_shape<64, 32>(act, mode, a, grid, rnvp_wide_smem_bytes(64, 32, mode), st);
  if (DH == 32) return launch_wide_shape<32, 16>(act, mode, a, grid, rnvp_wide_smem_bytes(32, 16, mode), st);
  if (DH == 16) return launch_wide_shape<16, 16>(act, mode, a, grid, rnvp_wide_smem_bytes(16, 16, mode), st);
  return cudaErrorInvalidValue;
}
