// Weight-gradient sweep of the fit step on the 5th-generation tensor cores (tcgen05 / TMEM).
//
// The backward sweep (rnvp_wide.cu) owns ROWS (two threads per row), so what it leaves behind per (layer, row) is row-major:
//     record = [ h (2H: nn_t | nn_s) | u = [x_K, c] (K1P8) | delta2 (2*TP: t | s) ]
// while the weight gradients are contractions OVER ROWS:
//     dW1[j][k] = sum_r delta1[r][j] u[r][k]     db1[j] = sum_r delta1[r][j]     delta1 = (delta2 W2) * act'(h)
//     dW2[e][j] = sum_r delta2[r][e] h[r][j]     db2[e] = sum_r delta2[r][e]
// tcgen05.mma contracts over the COLUMNS of its A operand (TMEM lane = output row), so this kernel works in the transposed
// world: one TMEM lane per HIDDEN UNIT.  A CTA owns (layer, block of 128 units of the concatenated list [nn_t | nn_s], row
// slice) and streams its rows in stages of 32:
//   warp 12     TMA producer: three bulk copies per stage (this block's h columns, u, delta2) into a raw ring
//   warps 2-3   converters: u and delta2 -> K-major operand tiles with K = rows (a 4-byte transposing scatter, conflict
//               free through a padded K-group stride), TF32 hi (the raw fp32: the tensor core reads its upper 19 bits) and
//               lo = v - trunc(v); delta2 also as the [rows x e] operand of the dh product; db2 partial sums in registers
//   warps 0-1   MMA issuers (one elected lane each; warp 0: dh^T and dW1, warp 1: dW2): dh^T[unit][row] = W2^T-image (TMEM, loaded once) x delta2  (3-pass split);
//               then dW1 += delta1^T (TMEM) x u and dW2^T += h^T (TMEM) x delta2, main products and split corrections in
//               separate TMEM accumulators
//   warps 4-11  unit owners (two threads per TMEM lane = hidden unit, 16 of the stage's 32 rows each): dh^T from TMEM, h
//               from the raw ring, delta1 = dh*act'(h), write delta1^T and h^T (hi/lo) back to TMEM as the A operands, db1
//               in a register; every WT_FOLD stages they drain the accumulators into fp32 register sums (the tensor core
//               TRUNCATES when it accumulates, so chains are kept short -- tools/mma_rounding_probe.py) and at the end
//               flush everything with red.global.add
// Nets share a lane block through a block-diagonal trick: the W2^T image of a unit holds its own net's W2 column in its
// net's half of K = [e_t | e_s] and zeros in the other half, and dW2^T is accumulated against both halves of delta2 (the
// foreign half is never written out).  Any H (multiple of 16) therefore maps onto ceil(2H / 128) lane blocks.
//
// Records are stored in blocks of 32 rows as [layer][block][column group of 4][32 slots][4] with slot = row ^ (group & 7):
// the row-per-thread writer stores 512 contiguous bytes per warp instruction, a block's column range is ONE contiguous
// bulk copy, and both the per-unit 4-byte reads (lanes = units) and the per-row 16-byte reads (lanes = rows) of this
// kernel are bank-conflict free.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include "rnvp_wgrad.h"
#include "tc05.cuh"

namespace {
using namespace tc05;

constexpr int WT_ROWS = 32;                 // rows per stage = rows per record block = K of one stage's gradient products
constexpr int WT_THREADS = 416;             // warps 0-1 issuers, 2-3 converters, 4-11 unit owners, 12 TMA producer
constexpr int WT_KG = 36;                   // floats between K-groups (4 rows) of a K-major-over-rows tile: 144 B, so that the
                                            // transposing 4-byte stores of a warp (lanes = rows) hit 32 different banks
constexpr int WT_NG = 8 * WT_KG;            // floats between 8-column groups (SBO = 1152 B)
#ifndef RNVP_WT_FOLD
#define RNVP_WT_FOLD 8
#endif
constexpr int WT_FOLD = RNVP_WT_FOLD;       // stages per accumulator chain (32 accumulations of K = 8).  Measured on the c3 step
                                            // (fit kernels, M rows/s | gradient error / max|grad|, bound 2e-5): 4: 68.4 | 3.5e-6,
                                            // 8: 69.3 | 4.0e-6, 16: 69.9 | 4.4e-6 (c5 sweep vs fp64 4.3e-6 of its 5e-6 bound), 32: fails

// Wait accounting (development aid, compile with -DRNVP_WG_TRACE; rnvp_debug_set_trace): when a trace buffer is set, every role of CTA 0 sums the cycles
// it spends in each of its mbarrier waits and writes the totals at the end: trace[role * 8 + k] (role 0 issuer A, 1 issuer
// B, 2 converter warp 2, 3 owner warp 4, 4 producer; k = wait site, 7 = total cycles of the role's loop).
#ifdef RNVP_WG_TRACE
struct WaitAcc {
  long long t[8];
  bool on;
  __device__ __forceinline__ void init(bool enable) { on = enable; for (int k = 0; k < 8; ++k) t[k] = 0; }
  __device__ __forceinline__ void wait(uint64_t* bar, uint32_t parity, int k, bool relaxed = false) {
    if (!on) {
      if (relaxed) tc05::mbar_wait_relaxed(bar, parity);
      else tc05::mbar_wait(bar, parity);
      return;
    }
    const long long t0 = clock64();
    if (relaxed) tc05::mbar_wait_relaxed(bar, parity);
    else tc05::mbar_wait(bar, parity);
    t[k] += clock64() - t0;
  }
  __device__ __forceinline__ void flush(long long* out, int role, long long total) {
    if (!on) return;
    t[7] = total;
    for (int k = 0; k < 8; ++k) out[role * 8 + k] = t[k];
  }
};
#else
// production build: the accounting compiles away (even a disabled accumulator array costs registers in every role, and this
// kernel is sensitive to that: a 720-byte per-thread event log made it 2x slower)
struct WaitAcc {
  static constexpr bool on = false;
  long long t[8];
  __device__ __forceinline__ void init(bool) {}
  __device__ __forceinline__ void wait(uint64_t* bar, uint32_t parity, int, bool relaxed = false) {
    if (relaxed) tc05::mbar_wait_relaxed(bar, parity);
    else tc05::mbar_wait(bar, parity);
  }
  __device__ __forceinline__ void flush(long long*, int, long long) {}
};
#endif

__device__ __forceinline__ float lo_part(float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

// NU: columns of the dW1 tile (>= K1P8, multiple of 16); K1P8: u columns of a record; TP: delta2 columns per net (multiple of 16)
// NBUF: TMEM staging buffers; NOP: operand buffers in shared memory; NSLOT: raw ring depth
template <int NU, int TP, int NBUF, int NOP, int NSLOT, bool SINGLE>
__global__ void __launch_bounds__(SINGLE ? 384 : WT_THREADS, 1) rnvp_wgrad_tc_kernel(const __grid_constant__ RnvpWgradTcArgs a) {
  // TMEM column map.  Per net the gradient accumulators sit side by side, [main | corr]: A_hi x [B_hi ; B_lo] is ONE MMA of
  // twice the width (the hi and lo operand tiles are adjacent in shared memory), A_lo x B_hi adds into the corr half.
  // SINGLE (wide flows, H % 128 == 0: every lane block belongs to one net): only the block's own net's delta2 / W2 columns
  // are staged, and main products and corrections share ONE accumulator per product (TMEM columns: 416 for c5)
  constexpr int NN = SINGLE ? 1 : 2;
  constexpr bool MERGED = !SINGLE;
  constexpr int NTHR = SINGLE ? 384 : WT_THREADS;          // SINGLE: one issuer (warp 0), the TMA producer takes warp 1: 12 warps, 168 registers
  const bool one_issuer = SINGLE || a.one_issuer;
  constexpr int W2H = 0, W2L = NN * TP, STG0 = 2 * NN * TP, STGW = 128;         // staging: DH/D1H +0, D1L +32, HH +64, HL +96
  constexpr int ACC1 = STG0 + NBUF * STGW, ACC2 = ACC1 + (MERGED ? 2 * NU : NU), TCOLS = ACC2 + (MERGED ? 4 * TP : TP);
  static_assert(TCOLS <= 512, "TMEM budget");
  static_assert(NU % 16 == 0 && TP % 16 == 0, "N of an M=128 MMA is a multiple of 16");
  constexpr int UB = (NU / 8) * WT_NG, EBN = (TP / 8) * WT_NG, DK = WT_ROWS * NN * TP;  // floats of one hi (or lo) tile
  constexpr int OPF = 2 * UB + 2 * NN * EBN + 2 * DK;                             // floats of one operand buffer
  // operand buffer: [u_hi | u_lo | e_t_hi | e_t_lo | e_s_hi | e_s_lo | dk_hi | dk_lo]
  constexpr int RAW_H = WT_ROWS * 128, RAW_E = WT_ROWS * NN * TP;
  const int K1P8 = a.K1P8;                                      // u columns of a record (multiple of 8, <= NU)
  const int RAW_U = WT_ROWS * K1P8, RAW = RAW_H + RAW_U + RAW_E;

  extern __shared__ __align__(128) float sm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = a.H, H2 = 2 * H;
  const int per_layer = a.n_mblocks * a.n_slices;
  const int layer = blockIdx.x / per_layer, rem = blockIdx.x - layer * per_layer;
  const int mb = rem / a.n_slices, slice = rem - mb * a.n_slices;
  const int ncols_h = min(128, H2 - 128 * mb);                  // this block's hidden units (h columns 128*mb ..)
  const int net_lo = (128 * mb >= H) ? 1 : 0, net_hi = (128 * mb + ncols_h > H) ? 1 : 0;   // nets present in this lane block
  float* raw = sm;
  float* op = sm + NSLOT * RAW;
  uint64_t* bars = reinterpret_cast<uint64_t*>(op + NOP * OPF);
  uint64_t* b_full = bars;                    // [NSLOT] raw slot filled (TMA bytes)
  uint64_t* b_empty = b_full + NSLOT;         // [NSLOT] raw slot drained: 2 converter warps + 8 owner warps
  uint64_t* b_conv = b_empty + NSLOT;         // [NOP]   operand buffer converted (64 threads)
  uint64_t* b_opfree = b_conv + NOP;          // [NOP]   gradient MMAs of the stage done (one tcgen05.commit per issuer)
  uint64_t* b_dh = b_opfree + NOP;            // [NBUF]  dh^T ready, and the dW1 products that read this staging buffer done
  uint64_t* b_hfree = b_dh + NBUF;            // [NBUF]  the dW2 products that read this staging buffer done
  uint64_t* b_afull = b_hfree + NBUF;         // [NBUF]  delta1^T / h^T staged in TMEM (256 owner threads)
  uint64_t* b_accfull = b_afull + NBUF;       // [1]     an accumulator chain is complete (one commit per issuer)
  uint64_t* b_accfree = b_accfull + 1;        // [1]     ... and drained into registers (256 owner threads)
  uint64_t* b_img = b_accfree + 1;            // [1]     W2^T image staged in TMEM (256 owner threads), once per kernel
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_img + 1);

  const long long blocks_total = a.Npad / WT_ROWS;
  const long long blk0 = blocks_total * slice / a.n_slices, blk1 = blocks_total * (slice + 1) / a.n_slices;
  const int nst = (int)(blk1 - blk0);                            // stages of this CTA

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 0) {
    for (int s = 0; s < NSLOT; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 10); }
    for (int b = 0; b < NOP; ++b) { mbar_init(&b_conv[b], 64); mbar_init(&b_opfree[b], one_issuer ? 1 : 2); }
    for (int b = 0; b < NBUF; ++b) { mbar_init(&b_dh[b], 1); mbar_init(&b_hfree[b], 1); mbar_init(&b_afull[b], 256); }
    mbar_init(b_accfull, one_issuer ? 1 : 2); mbar_init(b_accfree, 256); mbar_init(b_img, 256);
    mbar_fence_init();
  }
  // zero the operand buffers once: padding columns (K1P8..NU) and padding K-groups are never written again
  for (int i = tid; i < NOP * OPF; i += NTHR) op[i] = 0.0f;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = *tmem_slot;
  const size_t block_floats = (size_t)WT_ROWS * a.rec;
  const float* gblk = a.gR + ((size_t)layer * blocks_total + blk0) * block_floats;
  auto desc = [](uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) { return smem_desc_kmajor_nosw(addr, lbo_bytes, sbo_bytes); };
  constexpr uint32_t LBO = WT_KG * 4u, SBO = WT_NG * 4u, KS = 2 * WT_KG * 4u;      // K-major-over-rows tiles: one K step = 8 rows = 2 K-groups

  if (warp == 0) {
    // ------------------------------------------------------------------ issuer A: dh^T and dW1
    mbar_wait(b_img, 0);                                       // the owners have staged the W2^T image in TMEM
    fence_after_sync();
    const bool leader = elect_one();
    const uint32_t idesc_dh = idesc_tf32(128, WT_ROWS), idesc_u = idesc_tf32(128, NU), idesc_u2 = idesc_tf32(128, 2 * NU);
    const uint32_t op_addr = smem_u32(op);
    const int kj0 = SINGLE ? 0 : net_lo * (TP / 8), kj1 = SINGLE ? TP / 8 : (net_hi + 1) * (TP / 8);   // K steps of the dh product that are not all-zero
    // dh^T of stage s -> staging buffer s % NBUF: A = W2^T image (TMEM), B = delta2 [N = rows, K = 2TP] (core-matrix tiled)
    auto issue_dh = [&](int s) {
      const int b = s % NBUF, ob = s % NOP;
      const uint32_t dk_hi = op_addr + (uint32_t)(ob * OPF + 2 * UB + 2 * NN * EBN) * 4u, dk_lo = dk_hi + (uint32_t)DK * 4u;
      const uint32_t d = tbase + STG0 + b * STGW;
      constexpr uint32_t SBOD = (NN * TP / 4) * 128u;
#pragma unroll
      for (int j = 0; j < NN * TP / 8; ++j)
        if (j >= kj0 && j < kj1) mma_tf32_ts(d, tbase + W2L + 8 * j, desc(dk_hi + 256u * j, 128u, SBOD), idesc_dh, j > kj0 ? 1u : 0u);
#pragma unroll
      for (int j = 0; j < NN * TP / 8; ++j)
        if (j >= kj0 && j < kj1) mma_tf32_ts(d, tbase + W2H + 8 * j, desc(dk_lo + 256u * j, 128u, SBOD), idesc_dh, 1u);
#pragma unroll
      for (int j = 0; j < NN * TP / 8; ++j)
        if (j >= kj0 && j < kj1) mma_tf32_ts(d, tbase + W2H + 8 * j, desc(dk_hi + 256u * j, 128u, SBOD), idesc_dh, 1u);
    };
    uint32_t ph_conv = 0, ph_afull = 0, ph_accfree = 0;          // one phase bit per ring entry
    WaitAcc wa; wa.init((a.trace != nullptr && blockIdx.x == 0));
    const long long tstart = clock64();
    for (int s = 0; s < NBUF && s < nst; ++s) {                  // prologue: dh^T of the first NBUF stages
      const int ob = s % NOP;
      wa.wait(&b_conv[ob], (ph_conv >> ob) & 1u, 0); ph_conv ^= 1u << ob;
      fence_after_sync();
      if (leader) { issue_dh(s); mma_commit(&b_dh[s % NBUF]); }
      __syncwarp();
    }
    for (int s = 0; s < nst; ++s) {
      const int b = s % NBUF, ob = s % NOP;
      const bool first_in_grp = (s % WT_FOLD) == 0, last_in_grp = (s % WT_FOLD) == WT_FOLD - 1 || s == nst - 1;
      if (first_in_grp && s > 0) { wa.wait(b_accfree, ph_accfree, 1); ph_accfree ^= 1; }
      wa.wait(&b_afull[b], (ph_afull >> b) & 1u, 2); ph_afull ^= 1u << b;
      fence_after_sync();
      if (leader) {
        const uint32_t ub = op_addr + (uint32_t)(ob * OPF) * 4u;
        const uint32_t stg = tbase + STG0 + b * STGW;
        const long long tq0 = wa.on ? clock64() : 0;
#pragma unroll
        for (int j = 0; j < WT_ROWS / 8; ++j) {
          const uint32_t acc = (first_in_grp && j == 0) ? 0u : 1u;
          if (MERGED) {
            mma_tf32_ts(tbase + ACC1, stg + 0 + 8 * j, desc(ub + KS * j, LBO, SBO), idesc_u2, acc);               // d1_hi x [u_hi ; u_lo]
            mma_tf32_ts(tbase + ACC1 + NU, stg + 32 + 8 * j, desc(ub + KS * j, LBO, SBO), idesc_u, 1u);           // d1_lo x u_hi
          } else {
            mma_tf32_ts(tbase + ACC1, stg + 0 + 8 * j, desc(ub + KS * j, LBO, SBO), idesc_u, acc);                // d1_hi x u_hi
            mma_tf32_ts(tbase + ACC1, stg + 32 + 8 * j, desc(ub + KS * j, LBO, SBO), idesc_u, 1u);                // d1_lo x u_hi
            mma_tf32_ts(tbase + ACC1, stg + 0 + 8 * j, desc(ub + (uint32_t)UB * 4u + KS * j, LBO, SBO), idesc_u, 1u);   // d1_hi x u_lo
          }
        }
        if (wa.on) wa.t[4] += clock64() - tq0;
        if (one_issuer) {
          const uint32_t eb = ub + (uint32_t)(2 * UB) * 4u;
          const uint32_t idesc_e = idesc_tf32(128, TP), idesc_e2 = idesc_tf32(128, 2 * TP);
#pragma unroll
          for (int j = 0; j < WT_ROWS / 8; ++j) {
            const uint32_t acc = (first_in_grp && j == 0) ? 0u : 1u;
            if (MERGED) {
              for (int n = net_lo; n <= net_hi; ++n) {
                const uint32_t ebn = eb + (uint32_t)(n * 2 * EBN) * 4u, d2 = tbase + ACC2 + n * 2 * TP;
                mma_tf32_ts(d2, stg + 64 + 8 * j, desc(ebn + KS * j, LBO, SBO), idesc_e2, acc);
                mma_tf32_ts(d2 + TP, stg + 96 + 8 * j, desc(ebn + KS * j, LBO, SBO), idesc_e, 1u);
              }
            } else {
              mma_tf32_ts(tbase + ACC2, stg + 64 + 8 * j, desc(eb + KS * j, LBO, SBO), idesc_e, acc);
              mma_tf32_ts(tbase + ACC2, stg + 96 + 8 * j, desc(eb + KS * j, LBO, SBO), idesc_e, 1u);
              mma_tf32_ts(tbase + ACC2, stg + 64 + 8 * j, desc(eb + (uint32_t)EBN * 4u + KS * j, LBO, SBO), idesc_e, 1u);
            }
          }
          mma_commit(&b_hfree[b]);
        }
        mma_commit(&b_opfree[ob]);
        if (last_in_grp) mma_commit(b_accfull);
      }
      __syncwarp();
      if (s + NBUF < nst) {                      // dh^T of the stage that will reuse this staging buffer
        const int ob2 = (s + NBUF) % NOP;
        wa.wait(&b_conv[ob2], (ph_conv >> ob2) & 1u, 0); ph_conv ^= 1u << ob2;
        fence_after_sync();
        if (leader) {
          const long long tq0 = wa.on ? clock64() : 0;
          issue_dh(s + NBUF);
          if (wa.on) wa.t[5] += clock64() - tq0;
          mma_commit(&b_dh[b]);
          if (wa.on) wa.t[6] += clock64() - tq0;
        }
        __syncwarp();
      }
    }
    if (leader) wa.flush(a.trace, 0, clock64() - tstart);
  } else if (warp == 1 && !SINGLE) {
    // ------------------------------------------------------------------ issuer B: dW2 (issuing, not the tensor pipe, bounds
    // these small MMAs -- ~35 cycles each -- so the gradient products are split over two issuing threads)
    const bool leader = elect_one();
    int nst_b = nst;
    const uint32_t idesc_e = idesc_tf32(128, TP), idesc_e2 = idesc_tf32(128, 2 * TP);
    const uint32_t op_addr = smem_u32(op);
    uint32_t ph_afull = 0, ph_accfree = 0;
    if (a.one_issuer) nst_b = 0;
    WaitAcc wa; wa.init((a.trace != nullptr && blockIdx.x == 0));
    const long long tstart = clock64();
    for (int s = 0; s < nst_b; ++s) {
      const int b = s % NBUF, ob = s % NOP;
      const bool first_in_grp = (s % WT_FOLD) == 0, last_in_grp = (s % WT_FOLD) == WT_FOLD - 1 || s == nst - 1;
      if (first_in_grp && s > 0) { wa.wait(b_accfree, ph_accfree, 1); ph_accfree ^= 1; }
      wa.wait(&b_afull[b], (ph_afull >> b) & 1u, 2); ph_afull ^= 1u << b;
      fence_after_sync();
      if (leader) {
        const uint32_t eb = op_addr + (uint32_t)(ob * OPF + 2 * UB) * 4u;
        const uint32_t stg = tbase + STG0 + b * STGW;
#pragma unroll
        for (int j = 0; j < WT_ROWS / 8; ++j) {
          const uint32_t acc = (first_in_grp && j == 0) ? 0u : 1u;
          if (MERGED) {
            for (int n = net_lo; n <= net_hi; ++n) {
              const uint32_t ebn = eb + (uint32_t)(n * 2 * EBN) * 4u, d2 = tbase + ACC2 + n * 2 * TP;
              mma_tf32_ts(d2, stg + 64 + 8 * j, desc(ebn + KS * j, LBO, SBO), idesc_e2, acc);                // h_hi x [e_hi ; e_lo]
              mma_tf32_ts(d2 + TP, stg + 96 + 8 * j, desc(ebn + KS * j, LBO, SBO), idesc_e, 1u);             // h_lo x e_hi
            }
          } else {
            mma_tf32_ts(tbase + ACC2, stg + 64 + 8 * j, desc(eb + KS * j, LBO, SBO), idesc_e, acc);          // h_hi x e_hi
            mma_tf32_ts(tbase + ACC2, stg + 96 + 8 * j, desc(eb + KS * j, LBO, SBO), idesc_e, 1u);           // h_lo x e_hi
            mma_tf32_ts(tbase + ACC2, stg + 64 + 8 * j, desc(eb + (uint32_t)EBN * 4u + KS * j, LBO, SBO), idesc_e, 1u);   // h_hi x e_lo
          }
        }
        mma_commit(&b_opfree[ob]);
        mma_commit(&b_hfree[b]);
        if (last_in_grp) mma_commit(b_accfull);
      }
      __syncwarp();
    }
    if (leader) wa.flush(a.trace, 1, clock64() - tstart);
  } else if (warp == (SINGLE ? 1 : 12)) {
    // ------------------------------------------------------------------ TMA producer: three bulk copies per stage
    if (lane == 0) {
      const uint32_t bytes_h = (uint32_t)(WT_ROWS * ncols_h) * 4u;
      WaitAcc wa; wa.init((a.trace != nullptr && blockIdx.x == 0));
      const long long tstart = clock64();
      for (int s = 0; s < nst; ++s) {
        const int slot = s % NSLOT;
        if (s >= NSLOT) wa.wait(&b_empty[slot], (uint32_t)((s / NSLOT - 1) & 1), 0, true);
        const float* src = gblk + (size_t)s * block_floats;
        float* dst = raw + slot * RAW;
        mbar_expect_tx(&b_full[slot], bytes_h + (uint32_t)(RAW_U + RAW_E) * 4u);
        bulk_g2s(dst, src + (size_t)WT_ROWS * 128 * mb, bytes_h, &b_full[slot]);
        bulk_g2s(dst + RAW_H, src + (size_t)WT_ROWS * H2, (uint32_t)RAW_U * 4u, &b_full[slot]);
        bulk_g2s(dst + RAW_H + RAW_U, src + (size_t)WT_ROWS * (H2 + K1P8 + (SINGLE ? net_lo * TP : 0)), (uint32_t)RAW_E * 4u, &b_full[slot]);
      }
      wa.flush(a.trace, 4, clock64() - tstart);
    }
  } else if (warp < 4) {
    // ------------------------------------------------------------------ converters (lanes = rows)
    const int cw = warp - 2;
    constexpr int NCGE = (NN * TP) / 4, NUW = (NU / 4 + 1) / 2, NEW = NCGE / 2;
    const int NCGU = K1P8 / 4;
    const int cg_u0 = H2 >> 2, cg_e0 = (H2 + K1P8 + (SINGLE ? net_lo * TP : 0)) >> 2;                  // global column-group index (the slot swizzle uses it)
    float db2[NEW][4];
#pragma unroll
    for (int i = 0; i < NEW; ++i) db2[i][0] = db2[i][1] = db2[i][2] = db2[i][3] = 0.0f;
    const int r = lane;
    const int koff = (r >> 2) * WT_KG + (r & 3);                           // K-major-over-rows: K-group, position in group
    uint32_t ph_full = 0, ph_free = 0;
    WaitAcc wa; wa.init((a.trace != nullptr && blockIdx.x == 0) && warp == 2);
    const long long tstart = clock64();
    for (int s = 0; s < nst; ++s) {
      const int slot = s % NSLOT, ob = s % NOP;
      wa.wait(&b_full[slot], (ph_full >> slot) & 1u, 0); ph_full ^= 1u << slot;
      const float* R = raw + slot * RAW;
      // all of this warp's column groups are loaded before the first store (independent loads in flight)
      float4 vu[NUW], ve[NEW];
#pragma unroll
      for (int i = 0; i < NUW; ++i) {
        const int cg = cw + 2 * i;
        vu[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cg < NCGU) vu[i] = *reinterpret_cast<const float4*>(R + RAW_H + cg * 128 + ((r ^ ((cg_u0 + cg) & 7)) << 2));
      }
#pragma unroll
      for (int i = 0; i < NEW; ++i) {
        const int cg = cw + 2 * i;
        ve[i] = *reinterpret_cast<const float4*>(R + RAW_H + RAW_U + cg * 128 + ((r ^ ((cg_e0 + cg) & 7)) << 2));
      }
      if (s >= NOP) { wa.wait(&b_opfree[ob], (ph_free >> ob) & 1u, 1); ph_free ^= 1u << ob; }      // the MMAs that read this buffer are done
      float* ub_hi = op + ob * OPF;
      float* eb = ub_hi + 2 * UB;
      float* dk_hi = eb + 2 * NN * EBN;
#pragma unroll
      for (int i = 0; i < NUW; ++i) {
        const int cg = cw + 2 * i;
        if (cg < NCGU) {
          const float vv[4] = {vu[i].x, vu[i].y, vu[i].z, vu[i].w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int n = 4 * cg + q, o = (n >> 3) * WT_NG + (n & 7) * 4 + koff;
            ub_hi[o] = vv[q];
            ub_hi[UB + o] = lo_part(vv[q]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < NEW; ++i) {
        const int cg = cw + 2 * i;
        const float vv[4] = {ve[i].x, ve[i].y, ve[i].z, ve[i].w};
        const int net = (4 * cg) / TP;
        float* en_hi = eb + net * 2 * EBN;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int n = 4 * cg + q - net * TP, o = (n >> 3) * WT_NG + (n & 7) * 4 + koff;
          en_hi[o] = vv[q];
          en_hi[EBN + o] = lo_part(vv[q]);
          db2[i][q] += vv[q];
        }
        // operand of the dh product: [N = rows, K = 2TP], core matrices of 8 rows x 4 columns
        const int o2 = (r >> 3) * (NN * TP / 4) * 32 + cg * 32 + (r & 7) * 4;
        *reinterpret_cast<float4*>(dk_hi + o2) = ve[i];
        *reinterpret_cast<float4*>(dk_hi + DK + o2) = make_float4(lo_part(vv[0]), lo_part(vv[1]), lo_part(vv[2]), lo_part(vv[3]));
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // generic-proxy stores -> tensor-core reads
      mbar_arrive(&b_conv[ob]);
      __syncwarp();
      if (lane == 0) mbar_arrive(&b_empty[slot]);
    }
    if (lane == 0) wa.flush(a.trace, 2, clock64() - tstart);
    // db2[e] = sum over this CTA's rows of delta2[:, e]; the CTA of lane block 0 contributes it
    if ((SINGLE ? 128 * mb == net_lo * H : mb == 0) && nst > 0) {
      const RnvpWgradLayer& lw = a.layers[layer];
#pragma unroll
      for (int i = 0; i < NEW; ++i) {
        const int cg = cw + 2 * i;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float v = db2[i][q];
#pragma unroll
          for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
          const int e = 4 * cg + q, nl = e / TP, ee = e - nl * TP, net = SINGLE ? net_lo : nl;
          if (lane == 0 && ee < lw.nT) atomicAdd(a.gpacked + lw.b2_off[net] + ee, v);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ unit owners: two threads per TMEM lane (= hidden unit)
    const int half = (warp - 4) >> 2;                           // rows 16*half .. 16*half+15 of every stage
    const int m = (warp & 3) * 32 + lane;                       // lane of the block; warp % 4 = TMEM lane quarter
    const int q = 128 * mb + m;                                 // index in the concatenated unit list [nn_t | nn_s]
    const bool valid = q < H2;
    const int net = (valid && q >= H) ? 1 : 0, unit = valid ? q - net * H : 0;
    const uint32_t trow = tbase + ((uint32_t)((warp & 3) * 32) << 16);
    const RnvpWgradLayer& lw = a.layers[layer];
    // W2^T image of this unit: its own net's half of K = [e_t | e_s] holds W2[e][unit], the other half zeros
    {
      const float* w2 = a.packed + lw.w2_off[net];
#pragma unroll
      for (int e0 = half * (NN * TP / 2); e0 < (half + 1) * (NN * TP / 2); e0 += 8) {   // the two threads of a lane share the image columns
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int e = e0 + j, en = SINGLE ? net : e / TP, ee = SINGLE ? e : e - en * TP;
          float v = 0.0f;
          if (valid && en == net && ee < lw.nT) v = w2[ee * lw.Ks2 + unit];
          hi[j] = __float_as_uint(v);
          lo[j] = __float_as_uint(lo_part(v));
        }
        tmem_st_x8(trow + W2H + e0, hi);
        tmem_st_x8(trow + W2L + e0, lo);
      }
      tmem_wait_st();
      fence_before_sync();
    }
    mbar_arrive(b_img);                                          // the image is in place (issuer A waits for all 256 owners)
    // half 0 keeps the running sums of dW1 (this unit's row), half 1 those of dW2 (this unit's column, own net)
    constexpr int NS = NU > TP ? NU : TP;
    float sum[NS];
#pragma unroll
    for (int j = 0; j < NS; ++j) sum[j] = 0.0f;
    float db1 = 0.0f;
    const bool is_tanh = a.act == 1;
    const int hcg = m >> 2, hq = m & 3;
    uint32_t ph_full = 0, ph_dh = 0, ph_hfree = 0, ph_acc = 0;
    WaitAcc wa; wa.init((a.trace != nullptr && blockIdx.x == 0) && warp == 4);
    const long long tstart = clock64();
    uint32_t hh[16];
    // h of stage s (this unit, this thread's 16 rows) from the raw ring; releases the slot for this warp
    auto load_h = [&](int s) {
      const int slot = s % NSLOT;
      wa.wait(&b_full[slot], (ph_full >> slot) & 1u, 0); ph_full ^= 1u << slot;
      const float* Rh = raw + slot * RAW + hcg * 128 + hq;
#pragma unroll
      for (int r = 0; r < 16; ++r) hh[r] = __float_as_uint(Rh[((16 * half + r) ^ (hcg & 7)) << 2]);
      if (!valid) {
#pragma unroll
        for (int r = 0; r < 16; ++r) hh[r] = 0u;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&b_empty[slot]);
    };
    if (nst > 0) load_h(0);
    for (int s = 0; s < nst; ++s) {
      const int b = s % NBUF;
      wa.wait(&b_dh[b], (ph_dh >> b) & 1u, 1); ph_dh ^= 1u << b;
      if (s >= NBUF) { wa.wait(&b_hfree[b], (ph_hfree >> b) & 1u, 2); ph_hfree ^= 1u << b; }    // issuer B is done with this buffer
      fence_after_sync();
      const uint32_t stg = trow + STG0 + b * STGW + 16 * half;
      uint32_t dh[16], lo[16];
      tmem_ld_x16(stg, dh);
      tmem_wait_ld();
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const float h = __uint_as_float(hh[r]);
        const float dp = is_tanh ? fmaf(-h, h, 1.0f) : (h > 0.0f ? 1.0f : 0.0f);
        const float d1 = __uint_as_float(dh[r]) * dp;
        db1 += d1;
        dh[r] = __float_as_uint(d1);
        lo[r] = __float_as_uint(lo_part(d1));
      }
      tmem_st_x16(stg, dh);
      tmem_st_x16(stg + 32, lo);
#pragma unroll
      for (int r = 0; r < 16; ++r) lo[r] = __float_as_uint(lo_part(__uint_as_float(hh[r])));
      tmem_st_x16(stg + 64, hh);
      tmem_st_x16(stg + 96, lo);
      tmem_wait_st();
      fence_before_sync();
      mbar_arrive(&b_afull[b]);
      if (s + 1 < nst) load_h(s + 1);             // overlaps with the issuers' work on this stage
      // drain a finished accumulator chain into the fp32 register sums
      if ((s % WT_FOLD) == WT_FOLD - 1 || s == nst - 1) {
        wa.wait(b_accfull, ph_acc, 3); ph_acc ^= 1;
        fence_after_sync();
        if (half == 0) {
#pragma unroll
          for (int j0 = 0; j0 < NU; j0 += 16) {
            uint32_t vm[16], vc[16];
            tmem_ld_x16(trow + ACC1 + j0, vm);
            if (MERGED) tmem_ld_x16(trow + ACC1 + NU + j0, vc);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 16; ++j) sum[j0 + j] += MERGED ? __uint_as_float(vm[j]) + __uint_as_float(vc[j]) : __uint_as_float(vm[j]);
          }
        } else {
          const uint32_t acc = trow + ACC2 + (MERGED ? net * 2 * TP : 0);
#pragma unroll
          for (int j0 = 0; j0 < TP; j0 += 16) {
            uint32_t vm[16], vc[16];
            tmem_ld_x16(acc + j0, vm);
            if (MERGED) tmem_ld_x16(acc + TP + j0, vc);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 16; ++j) sum[j0 + j] += MERGED ? __uint_as_float(vm[j]) + __uint_as_float(vc[j]) : __uint_as_float(vm[j]);
          }
        }
        fence_before_sync();
        mbar_arrive(b_accfree);
      }
    }
    if (lane == 0) wa.flush(a.trace, 3, clock64() - tstart);
    // ---- flush: this unit's row of dW1 (half 0), its column of dW2 (half 1), db1 (both halves' partial sums)
    if (nst > 0 && valid) {
      if (half == 0) {
        float* gw1 = a.gpacked + lw.w1_off[net] + (size_t)unit * lw.Ks1;
        if (lw.nK == a.TP) {   // exact shape: u = [x_K | c] has the packed row's column order
#pragma unroll
          for (int j = 0; j < NU; j += 4)
            if (j < a.K1)      // K1 = |K| + Cd real columns; the packed row is padded to a multiple of 4
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gw1 + j), "f"(sum[j]), "f"(sum[j + 1]),
                           "f"(sum[j + 2]), "f"(sum[j + 3]) : "memory");
        } else {               // padded shape: the record's x_K part has TP slots, the packed row only |K|
#pragma unroll
          for (int j = 0; j < NU; ++j) {
            if (j < lw.nK) atomicAdd(gw1 + j, sum[j]);
            else if (j >= a.TP && j < a.TP + a.Cd) atomicAdd(gw1 + lw.nK + (j - a.TP), sum[j]);
          }
        }
      } else {
        float* gw2 = a.gpacked + lw.w2_off[net] + unit;
#pragma unroll
        for (int e = 0; e < TP; ++e)
          if (e < lw.nT) atomicAdd(gw2 + (size_t)e * lw.Ks2, sum[e]);
      }
      atomicAdd(a.gpacked + lw.b1_off[net] + unit, db1);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, 512);
}

template <int NU, int TP, int NBUF, int NOP, int NSLOT, bool SINGLE = false>
cudaError_t launch_tc(const RnvpWgradTcArgs& a, int grid, cudaStream_t st) {
  if (a.K1P8 > NU || a.K1P8 % 8) return cudaErrorInvalidValue;
  auto k = rnvp_wgrad_tc_kernel<NU, TP, NBUF, NOP, NSLOT, SINGLE>;
  const size_t smem = rnvp_wgrad_tc_smem_bytes(NU, TP, NBUF, NOP, NSLOT, a.K1P8, SINGLE ? 1 : 2);
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k<<<grid, SINGLE ? 384 : WT_THREADS, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace

size_t rnvp_wgrad_tc_smem_bytes(int NU, int TP, int NBUF, int NOP, int NSLOT, int K1P8, int NN) {
  const size_t raw = (size_t)WT_ROWS * (128 + K1P8 + NN * TP);
  const size_t opf = 2 * (size_t)(NU / 8) * WT_NG + 2 * NN * (size_t)(TP / 8) * WT_NG + 2 * (size_t)WT_ROWS * NN * TP;
  return (NSLOT * raw + NOP * opf) * 4 + 8 * (2 * NSLOT + 2 * NOP + 3 * NBUF + 3) + 64;
}

// D <= 32 flows: NU 32, TP 16.  D <= 64: NU 48, TP 32 (one staging buffer: TMEM columns).  D <= 128: NU 96, TP 64, single-net
// lane blocks (H a multiple of 128).  K1P8 = ceil8(DH + Cd) <= NU is a run-time value.
// ring depths measured on c3 (tools/wg_time.py): raw ring 4 / operand buffers 4 = 0.59 ms, 7 / 2 = 0.61, 6 / 3 = 0.59, 4 / 2 = 0.61:
// the sweep is not bound by bytes in flight
cudaError_t rnvp_launch_wgrad_tc(int NU, int TP, const RnvpWgradTcArgs& a, int grid, cudaStream_t st) {
  if (NU == 32 && TP == 16) return launch_tc<32, 16, 2, 4, 4>(a, grid, st);
  if (NU == 48 && TP == 32) return launch_tc<48, 32, 1, 2, 3>(a, grid, st);
  if (NU == 96 && TP == 64 && a.H % 128 == 0) return launch_tc<96, 64, 1, 2, 2, true>(a, grid, st);
  return cudaErrorInvalidValue;
}
