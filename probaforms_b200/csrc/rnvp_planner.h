// Host-only planner for the fused RealNVP tile kernels: flow geometry, the packed parameter
// layout and its index maps, and the per-tile op program (see rnvp_plan.h).  No CUDA calls in
// here, so the same code is compiled into librnvp_b200.so (rnvp_api.cu) and into the test-only
// host emulator (tests/emul/rnvp_emul.cpp) that checks the programs without a GPU.
#pragma once
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <vector>

#include "rnvp_plan.h"

namespace rnvp_planner {

inline int ceil4(int k) { return (k + 3) & ~3; }
// row stride == 4 (mod 8) floats: 8 consecutive rows hit 8 distinct 16-byte bank groups (LDS.128)
inline int pad_stride(int k) {
  int c = ceil4(k);
  return (c % 8 == 4) ? c : c + 4;
}
inline int pow2ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

struct LinearGeom {
  int in_dim, out_dim;      // compacted dims (mask-aware for the first / last Linear)
  int in_full, out_full;    // reference dims
  int Kc, Ks, rows_p;
  int w_off[2], b_off[2];   // packed offsets per net (t, s)
  int64_t flat_w[2], flat_b[2];
};
struct LayerGeom {
  int par, nK, nT;          // T = {j : j%2 == par}, K = {j : j%2 == 1-par}
  std::vector<LinearGeom> lin;
};

struct FlowGeom {
  int D, Cd, L, nh, act;
  int hidden[RNVP_MAX_HIDDEN];
  int max_smem = 232448;     // bytes of opt-in dynamic shared memory per CTA (sm_100: 227 KB)
  std::vector<LayerGeom> layers;
  int64_t P = 0, packed = 0;     // packed = tile layout + (optional) small-flow layout
  int64_t packed_tile = 0;       // floats of the tile-kernel layout (the gradient accumulator covers only this)
  // row-per-thread small-flow layout (rnvp_small.cu): one hidden layer, ceil(D/2) <= 4, Cd <= 4
  bool small_ok = false;
  int sNE = 0, sNC = 0, srec = 0, snet = 0, small_floats = 0;
  int64_t small_off = 0;
  int64_t packed_gather = 0;     // floats covered by the plain gather map p2f (tile + small layouts)
  // tcgen05 layout (rnvp_wide.cu): one hidden layer, 8 < D <= 128; TF32 hi/lo images of the weights in the no-swizzle
  // K-major core-matrix layout, per layer [W1 chunks | W2 chunks | b2 | W2T chunks | W1T chunks]
  bool mma_ok = false;
  int mDH = 0, mCDMAX = 0, mCU = 0, mK1P = 0, mNTP = 0;
  int m_w1_floats = 0, m_w2_floats = 0, m_b2_floats = 0, m_layer_floats = 0;
  int m_wt_floats = 0;   // transposed images for the backward sweep (W2T then W1T, m_wt_floats each), 0 if not built
  int64_t mma_off = 0, mma_floats = 0;
};

// ------------------------------------------------------------------ layout
inline void build_layout(FlowGeom* d) {
  const int D = d->D, Cd = d->Cd, nh = d->nh;
  int64_t flat = 0;
  int packed = 0;
  d->layers.resize(d->L);
  for (int i = 0; i < d->L; ++i) {
    LayerGeom& lg = d->layers[i];
    lg.par = i & 1;                       // mask_i[j] = (j+i)%2 == 0  <=>  j%2 == i%2
    lg.nT = (D - lg.par + 1) / 2;         // #j in [0,D) with j%2 == par
    lg.nK = D - lg.nT;
    lg.lin.resize(nh + 1);
    // reference order: nn_t (all Linears) then nn_s (realnvp.py:69-70)
    for (int net = 0; net < 2; ++net)
      for (int q = 0; q <= nh; ++q) {
        LinearGeom& g = lg.lin[q];
        g.in_full = q == 0 ? D + Cd : d->hidden[q - 1];
        g.out_full = q == nh ? D : d->hidden[q];
        g.flat_w[net] = flat;
        flat += (int64_t)g.in_full * g.out_full;
        g.flat_b[net] = flat;
        flat += g.out_full;
      }
    for (int q = 0; q <= nh; ++q) {
      LinearGeom& g = lg.lin[q];
      g.in_dim = q == 0 ? lg.nK + Cd : d->hidden[q - 1];
      g.out_dim = q == nh ? lg.nT : d->hidden[q];
      g.Kc = ceil4(g.in_dim);
      g.Ks = pad_stride(g.in_dim);
      g.rows_p = lg.nT == 0 ? 0 : ceil4(g.out_dim);
      for (int net = 0; net < 2; ++net) { g.w_off[net] = packed; packed += g.rows_p * g.Ks; }
      for (int net = 0; net < 2; ++net) { g.b_off[net] = packed; packed += g.rows_p; }
    }
  }
  d->P = flat;
  d->packed_tile = std::max(packed, 4);
  d->packed = d->packed_tile;
  // small-flow layout
  const int ne = (D + 1) / 2;
  d->small_ok = false;
  if (nh == 1 && ne <= 4 && Cd <= 4) {
    d->sNE = ne <= 1 ? 1 : (ne <= 2 ? 2 : 4);
    d->sNC = Cd == 0 ? 0 : (Cd <= 1 ? 1 : (Cd <= 2 ? 2 : 4));
    d->srec = ceil4(2 * d->sNE + d->sNC + 1);
    d->snet = d->hidden[0] * d->srec + ceil4(d->sNE);
    const int64_t total = (int64_t)d->L * 2 * d->snet;
    if (total * 4 <= 64 * 1024) {
      d->small_ok = true;
      d->small_floats = (int)total;
      d->small_off = d->packed_tile;
      d->packed = d->small_off + total;
    }
  }
  d->packed_gather = d->packed;
  // tcgen05 layout
  d->mma_ok = false;
  if (nh == 1 && D > 8 && D <= 128) {
    // the kernels are built for DH = D/2 in {16, 32, 64}; any other D (odd ones included) runs as the next larger shape
    // with zero-weight padding features: |K|, |T| <= DH, the images hold zeros beyond them, the row loads are guarded
    const int DH = D <= 32 ? 16 : (D <= 64 ? 32 : 64), H = d->hidden[0];
    const int CDMAX = DH == 16 ? 16 : (DH == 32 ? 16 : 32), CU = 32;
    const int K1P = (DH + Cd + 1 + 7) & ~7, NTP = (DH + 15) & ~15;
    const int64_t w1 = (int64_t)4 * H * K1P, w2 = (int64_t)4 * NTP * H;
    // The weight images are streamed per chunk step, so no shape needs them to fit shared memory.  DH = 16 flows still run
    // on the tensor cores only where the whole-layer images would fit: that rule decides which flows take the tcgen05 path.
    const bool fits = DH >= 32 || (w1 + w2 + 32 * NTP) * 4 + 2048 <= d->max_smem;
    if (Cd <= CDMAX && H % CU == 0 && H >= CU && fits) {
      d->mma_ok = true;
      d->mDH = DH; d->mCDMAX = CDMAX; d->mCU = CU; d->mK1P = K1P; d->mNTP = NTP;
      d->m_b2_floats = 32 * NTP;                               // 2 nets x [hi | lo] x [NTP x 8]
      d->m_w1_floats = (int)w1; d->m_w2_floats = (int)w2 + d->m_b2_floats;  // b2 images ride with the W2 copy
      // backward sweep: per chunk step (net, chunk of CU units) a W2T block [hi | lo] of [CU x DH] and a W1T block [hi | lo]
      // of [NTP x CU]; for DH = 64 the tcgen05 weight-gradient sweep needs whole 128-unit lane blocks per net
      d->m_wt_floats = (DH < 64 || H % 128 == 0) ? 4 * H * NTP : 0;
      d->m_layer_floats = d->m_w1_floats + d->m_w2_floats + 2 * d->m_wt_floats;
      d->mma_off = (d->packed + 31) & ~(int64_t)31;            // 128-byte aligned for the bulk copies
      d->mma_floats = (int64_t)d->L * d->m_layer_floats;
      d->packed = d->mma_off + d->mma_floats;
    }
  }
}

// float offset of element (n, k) of an [N x K] K-major MMA operand in the no-swizzle core-matrix layout
// (8 rows x 16 B core matrices, 128 B each, K-adjacent core matrices contiguous): see tc05.cuh
inline int mma_tiled_off(int n, int k, int K) { return (n >> 3) * (K >> 2) * 32 + (k >> 2) * 32 + (n & 7) * 4 + (k & 3); }

// map of the tcgen05 region: value = 4*flat_index + code (0: TF32 hi image, 1: lo remainder, 2: full fp32), or -1 (zero).
// RNVP_IMG_SCALED (bit 30) marks the entries of the FORWARD W1 image (weights and the b1 column) of a tanh flow: they hold
// 2*log2(e) times the parameter, so that GEMM1 delivers the argument of the tanh's ex2 directly and the epilogue saves one
// multiply per hidden activation.  Nothing else reads that image (the backward products use the transposed images).
constexpr int RNVP_IMG_SCALED = 1 << 30;
constexpr float RNVP_TANH_PRESCALE = 2.8853900817779268f;       // tanh(a) = 1 - 2 / (2^(a * 2 log2 e) + 1)
inline void build_mma_map(const FlowGeom* d, std::vector<int>& m2f) {
  m2f.assign(d->mma_ok ? d->mma_floats : 0, -1);
  if (!d->mma_ok) return;
  const int D = d->D, Cd = d->Cd, H = d->hidden[0], DH = d->mDH, CU = d->mCU, K1P = d->mK1P, NTP = d->mNTP;
  const int NC = H / CU;
  for (int i = 0; i < d->L; ++i) {
    const LayerGeom& lg = d->layers[i];
    const LinearGeom& g0 = lg.lin[0];
    const LinearGeom& g1 = lg.lin[1];
    const int64_t base = (int64_t)i * d->m_layer_floats;
    // W1 image: one block [hi | lo] of CU rows per chunk step; blocks 0..NC-1 are the nn_t chunks, NC..2NC-1 the nn_s chunks
    for (int cc = 0; cc < 2 * NC; ++cc)
      for (int part = 0; part < 2; ++part) {
        const int64_t blk = base + ((int64_t)cc * 2 + part) * (CU * K1P);
        for (int n = 0; n < CU; ++n) {
          const int net = cc / NC;
          const int unit = (cc % NC) * CU + n;
          for (int k = 0; k < K1P; ++k) {
            int64_t f = -1;
            if (k < DH) { const int xk = lg.par == 0 ? 2 * k + 1 : 2 * k; if (xk < D) f = g0.flat_w[net] + (int64_t)unit * (D + Cd) + xk; }
            else if (k < DH + Cd) f = g0.flat_w[net] + (int64_t)unit * (D + Cd) + D + (k - DH);
            else if (k == DH + Cd) f = g0.flat_b[net] + unit;
            if (f >= 0) m2f[blk + mma_tiled_off(n, k, K1P)] = (int)(4 * f + part) | (d->act == 1 ? RNVP_IMG_SCALED : 0);
          }
        }
      }
    // W2 image: chunk c, net, [hi | lo]: rows = transformed features, cols = units of the chunk
    const int64_t base2 = base + d->m_w1_floats;
    for (int c = 0; c < NC; ++c)
      for (int net = 0; net < 2; ++net)
        for (int part = 0; part < 2; ++part) {
          const int64_t blk = base2 + (((int64_t)c * 2 + net) * 2 + part) * (NTP * CU);
          for (int r = 0; r < DH; ++r) {
            const int ft = lg.par == 0 ? 2 * r : 2 * r + 1;
            if (ft >= D) continue;
            for (int kk = 0; kk < CU; ++kk)
              m2f[blk + mma_tiled_off(r, kk, CU)] = (int)(4 * (g1.flat_w[net] + (int64_t)ft * H + c * CU + kk) + part);
          }
        }
    // b2 images: per net [hi | lo] of an [NTP x 8] operand; column (DH+Cd)%8 holds b2, the rest is zero.  Multiplied
    // with the 8-column u slice that contains the constant one it seeds the GEMM2 accumulator with the bias.
    const int64_t base3 = base2 + (int64_t)4 * NTP * H;
    for (int net = 0; net < 2; ++net)
      for (int part = 0; part < 2; ++part)
        for (int r = 0; r < DH; ++r) {
          const int ft = lg.par == 0 ? 2 * r : 2 * r + 1;
          if (ft >= D) continue;
          m2f[base3 + (net * 2 + part) * (NTP * 8) + mma_tiled_off(r, (DH + Cd) & 7, 8)] = (int)(4 * (g1.flat_b[net] + ft) + part);
        }
    if (d->m_wt_floats) {
      // backward images, indexed by chunk step cc = net * NC + c
      const int64_t base4 = base2 + d->m_w2_floats, base5 = base4 + d->m_wt_floats;
      for (int net = 0; net < 2; ++net)
        for (int c = 0; c < NC; ++c)
          for (int part = 0; part < 2; ++part) {
            const int64_t cc = (int64_t)net * NC + c;
            const int64_t o2 = base4 + (cc * 2 + part) * ((int64_t)CU * NTP);     // W2T block: [CU units x NTP (e, K)]
            const int64_t o1 = base5 + (cc * 2 + part) * ((int64_t)NTP * CU);     // W1T block: [NTP (x_K col) x CU units (K)]
            for (int un = 0; un < CU; ++un)
              for (int e = 0; e < DH; ++e) {
                const int unit = c * CU + un;
                const int ft = lg.par == 0 ? 2 * e : 2 * e + 1;            // transformed feature e
                const int xk = lg.par == 0 ? 2 * e + 1 : 2 * e;            // conditioning feature e
                if (ft < D) m2f[o2 + mma_tiled_off(un, e, NTP)] = (int)(4 * (g1.flat_w[net] + (int64_t)ft * H + unit) + part);
                if (xk < D) m2f[o1 + mma_tiled_off(e, un, CU)] = (int)(4 * (g0.flat_w[net] + (int64_t)unit * (D + Cd) + xk) + part);
              }
          }
    }
  }
}

// second flat -> packed map: position of each parameter in the small-flow layout (or -1)
inline void build_small_map(const FlowGeom* d, std::vector<int>& p2f, std::vector<int>& f2p2) {
  f2p2.assign(d->P, -1);
  if (!d->small_ok) return;
  const int D = d->D, Cd = d->Cd, H = d->hidden[0], NE = d->sNE, NC = d->sNC, rec = d->srec;
  for (int i = 0; i < d->L; ++i) {
    const LayerGeom& lg = d->layers[i];
    const LinearGeom& g0 = lg.lin[0];
    const LinearGeom& g1 = lg.lin[1];
    for (int net = 0; net < 2; ++net) {
      const int64_t base = d->small_off + ((int64_t)i * 2 + net) * d->snet;
      auto put = [&](int64_t p, int64_t f) { p2f[p] = (int)f; f2p2[f] = (int)p; };
      for (int j = 0; j < H; ++j) {
        const int64_t u = base + (int64_t)j * rec;
        for (int e = 0; e < NE; ++e) {
          const int fk = lg.par == 0 ? 2 * e + 1 : 2 * e;            // conditioning (keep) feature
          if (fk < D) put(u + e, g0.flat_w[net] + (int64_t)j * (D + Cd) + fk);
          const int ft = lg.par == 0 ? 2 * e : 2 * e + 1;            // transformed feature
          if (ft < D) put(u + NE + NC + 1 + e, g1.flat_w[net] + (int64_t)ft * H + j);
        }
        for (int k = 0; k < NC && k < Cd; ++k) put(u + NE + k, g0.flat_w[net] + (int64_t)j * (D + Cd) + D + k);
        put(u + NE + NC, g0.flat_b[net] + j);
      }
      for (int e = 0; e < NE; ++e) {
        const int ft = lg.par == 0 ? 2 * e : 2 * e + 1;
        if (ft < D) put(base + (int64_t)H * rec + e, g1.flat_b[net] + ft);
      }
    }
  }
}

inline void build_maps(const FlowGeom* d, std::vector<int>& p2f, std::vector<int>& f2p) {
  p2f.assign(d->packed_gather, -1);
  f2p.assign(d->P, -1);
  const int D = d->D, nh = d->nh;
  for (int i = 0; i < d->L; ++i) {
    const LayerGeom& lg = d->layers[i];
    if (lg.nT == 0) continue;
    for (int q = 0; q <= nh; ++q) {
      const LinearGeom& g = lg.lin[q];
      for (int net = 0; net < 2; ++net)
        for (int n = 0; n < g.out_dim; ++n) {
          const int row = q == nh ? 2 * n + lg.par : n;
          for (int k = 0; k < g.in_dim; ++k) {
            int col = k;
            if (q == 0) col = k < lg.nK ? 2 * k + (1 - lg.par) : D + (k - lg.nK);
            const int64_t f = g.flat_w[net] + (int64_t)row * g.in_full + col;
            const int p = g.w_off[net] + n * g.Ks + k;
            p2f[p] = (int)f;
            f2p[f] = p;
          }
          const int64_t fb = g.flat_b[net] + row;
          p2f[g.b_off[net] + n] = (int)fb;
          f2p[fb] = g.b_off[net] + n;
        }
    }
  }
}

// ---------------------------------------------------- micro-tile selection
inline void choose_linear(int rows_p, int Kc, int* tn, int* split) {
  long best = -1;
  const int nkb = std::max(Kc / 4, 1);
  for (int S = 1; S <= 4; S <<= 1) {
    if (S > 1 && nkb < S) continue;
    const int CG = 16 / S;
    for (int TN = 8; TN >= 4; TN -= 4) {
      const int passes = (rows_p + CG * TN - 1) / (CG * TN);
      long cost = (long)passes * TN * ((nkb + S - 1) / S) * 8 + (S > 1 ? TN * 4 * S : 0) + passes * 16;
      if (best < 0 || cost < best) { best = cost; *tn = TN; *split = S; }
    }
  }
}
inline void choose_dgrad(int kout, int rows_p, int* q, int* split) {
  long best = -1;
  const int ncb = std::max((kout + 3) / 4, 1), nnb = std::max(rows_p / 4, 1);
  for (int S = 1; S <= 4; S <<= 1) {
    if (S > 1 && nnb < S) continue;
    const int CG = 16 / S;
    for (int Q = 2; Q >= 1; --Q) {
      const int passes = (ncb + CG * Q - 1) / (CG * Q);
      long cost = (long)passes * Q * ((nnb + S - 1) / S) * 8 + (S > 1 ? Q * 8 * S : 0) + passes * 16;
      if (best < 0 || cost < best) { best = cost; *q = Q; *split = S; }
    }
  }
}
inline void choose_wgrad(int rows_p, int Kc, int R, int* qq, int* split) {
  long best = -1;
  const int nb4 = std::max(rows_p / 4, 1), kb4 = std::max(Kc / 4, 1);
  for (int Q = 2; Q >= 1; --Q) {
    const int tiles = ((nb4 + Q - 1) / Q) * ((kb4 + Q - 1) / Q);
    for (int S = 1; S <= 32 && S <= R; S <<= 1) {
      const int passes = (tiles * S + RNVP_NET_THREADS - 1) / RNVP_NET_THREADS;
      long cost = (long)passes * (Q * Q * (R / S) * 16 + 2 * Q * (R / S) + (S > 1 ? 16 * Q * Q * 5 : 0) + 32);
      if (best < 0 || cost < best) { best = cost; *qq = Q; *split = S; }
    }
  }
}

// ------------------------------------------------------------------ planner
struct Builder {
  const FlowGeom* d;
  int mode, l0, l1, TR, R;
  RnvpSmem sm{};
  std::vector<RnvpOp> ops;
  std::vector<RnvpChunk> chunks;
  std::vector<int> hbuf_off, hbuf_stride;   // hidden activation buffers
  int dbuf_off = -1, dbuf_stride = 0;
  int slot_floats = 0;
  int cap = 7680;            // weight-ring slot capacity in floats (one chunk of both nets)
  int stash_per_cta = 0;
  std::vector<int> stash_off;

  int rows_per_chunk(const LinearGeom& g) const {
    int r = (slot_floats / (2 * (g.Ks + 1))) & ~3;
    return std::min(std::max(r, 4), g.rows_p);
  }

  bool plan_smem(int max_floats) {
    const int D = d->D, Cd = d->Cd, nh = d->nh;
    int maxK1c = 0, maxT = 0, maxK = 0, maxH = 0;
    long max_block = 0;
    int maxKs = 4;
    bool any = false;
    for (int i = l0; i < l1; ++i) {
      const LayerGeom& lg = d->layers[i];
      if (lg.nT == 0) continue;
      any = true;
      maxK1c = std::max(maxK1c, lg.lin[0].Kc);
      maxT = std::max(maxT, lg.nT);
      maxK = std::max(maxK, lg.nK);
      for (const LinearGeom& g : lg.lin) {
        max_block = std::max(max_block, (long)2 * g.rows_p * (g.Ks + 1));
        maxKs = std::max(maxKs, g.Ks);
      }
    }
    for (int q = 0; q < nh; ++q) maxH = std::max(maxH, d->hidden[q]);
    const int CAP = cap;
    slot_floats = (int)std::min<long>(max_block, CAP);
    slot_floats = std::max(slot_floats, 8 * (maxKs + 1));
    slot_floats = ceil4(slot_floats);
    if (!any) slot_floats = 16;

    int off = 0;
    auto take = [&](int n) { int o = off; off += ceil4(n); return o; };
    sm.xs_stride = pad_stride(D);
    sm.xs = take(R * sm.xs_stride);
    sm.cs_stride = pad_stride(std::max(Cd, 1));
    sm.cs = take(Cd > 0 ? R * sm.cs_stride : 4);
    sm.gx = mode >= 2 ? take(R * sm.xs_stride) : 0;
    sm.ub_stride = pad_stride(std::max(maxK1c, 1));
    sm.ub = take(R * sm.ub_stride);
    sm.ld = take(R);
    sm.st_stride = pad_stride(std::max(maxT, 1));
    sm.st_net = R * sm.st_stride;
    sm.st = take(2 * sm.st_net);
    sm.gu_stride = pad_stride(std::max(maxK, 1));
    sm.gu_net = R * sm.gu_stride;
    sm.gu = mode >= 2 ? take(2 * sm.gu_net) : 0;
    hbuf_off.clear();
    hbuf_stride.clear();
    if (mode >= 2) {
      bool chunked = false;
      for (int q = 0; q < nh; ++q) {
        hbuf_stride.push_back(pad_stride(d->hidden[q]));
        hbuf_off.push_back(take(2 * R * hbuf_stride.back()));
      }
      for (int i = l0; i < l1; ++i) {
        const LayerGeom& lg = d->layers[i];
        if (lg.nT == 0) continue;
        for (int q = 1; q <= nh; ++q)
          if (rows_per_chunk(lg.lin[q]) < lg.lin[q].rows_p) chunked = true;
      }
      if (chunked) {
        dbuf_stride = pad_stride(maxH);
        dbuf_off = take(2 * R * dbuf_stride);
      }
    } else {
      const int nb = nh > 1 ? 2 : 1;
      for (int b = 0; b < nb; ++b) {
        hbuf_stride.push_back(pad_stride(maxH));
        hbuf_off.push_back(take(2 * R * hbuf_stride.back()));
      }
    }
    sm.slot_floats = slot_floats;
    sm.wring = take(RNVP_NSLOTS * slot_floats);
    sm.mbar = take(2 * RNVP_NSLOTS);
    sm.red = take(8);
    sm.total_floats = off;
    return off <= max_floats;
  }

  // largest row tile, then largest weight slot, that fits the shared-memory budget
  bool plan_best(int tr_force = 0) {
    static const int caps[3] = {7680, 3840, 1920};
    for (int tr = tr_force > 0 ? tr_force : 8; tr >= 2; tr >>= 1) {
      for (int c = 0; c < 3; ++c) {
        TR = tr; R = 8 * tr; cap = caps[c];
        if (plan_smem(d->max_smem / 4)) return true;
      }
      if (tr_force > 0) break;
    }
    return false;
  }

  RnvpOp base_op(int kind, int layer) const {
    RnvpOp op;
    memset(&op, 0, sizeof(op));
    op.kind = kind;
    op.layer = layer;
    op.chunk = -1;
    op.split = 1;
    if (layer >= 0) {
      const LayerGeom& lg = d->layers[layer];
      op.nK = lg.nK; op.nT = lg.nT; op.par = lg.par;
      op.Kc = lg.lin[0].Kc;
    }
    return op;
  }

  void hidden_buffer(int q, int* off, int* stride) const {
    const int b = mode >= 2 ? q : (q & 1) % (int)hbuf_off.size();
    *off = hbuf_off[b];
    *stride = hbuf_stride[b];
  }

  // Linear q of layer i, both nets, one op per weight row chunk
  void emit_linear(int i, int q, int extra_flags) {
    const LayerGeom& lg = d->layers[i];
    const LinearGeom& g = lg.lin[q];
    const int nh = d->nh;
    const int rc = rows_per_chunk(g);
    for (int n0 = 0; n0 < g.rows_p; n0 += rc) {
      const int rp = std::min(rc, g.rows_p - n0);
      RnvpOp op = base_op(OP_LINEAR, i);
      op.flags = extra_flags;
      op.chunk = (int)chunks.size();
      if (q == 0) { op.a_off = sm.ub; op.a_stride = sm.ub_stride; op.a_net = 0; }
      else { hidden_buffer(q - 1, &op.a_off, &op.a_stride); op.a_net = R * op.a_stride; }
      if (q < nh) { hidden_buffer(q, &op.o_off, &op.o_stride); op.o_net = R * op.o_stride; op.act = d->act; }
      else { op.o_off = sm.st; op.o_stride = sm.st_stride; op.o_net = sm.st_net; op.act = 0; }
      op.rows = std::max(0, std::min(rp, g.out_dim - n0));
      op.rows_p = rp; op.n0 = n0;
      op.K = g.in_dim; op.Kc = g.Kc; op.Ks = g.Ks;
      choose_linear(rp, g.Kc, &op.tn, &op.split);
      ops.push_back(op);
      RnvpChunk c;
      memset(&c, 0, sizeof(c));
      for (int net = 0; net < 2; ++net) { c.w_src[net] = g.w_off[net] + n0 * g.Ks; c.b_src[net] = g.b_off[net] + n0; }
      c.rows_p = rp; c.Ks = g.Ks;
      chunks.push_back(c);
    }
  }

  void emit_dgrad(int i, int q, bool to_gu) {
    const LayerGeom& lg = d->layers[i];
    const LinearGeom& g = lg.lin[q];
    const int nh = d->nh;
    const int rc = rows_per_chunk(g);
    for (int n0 = 0; n0 < g.rows_p; n0 += rc) {
      const int rp = std::min(rc, g.rows_p - n0);
      RnvpOp op = base_op(OP_DGRAD, i);
      op.chunk = (int)chunks.size();
      if (n0 == 0) op.flags |= F_FIRST;
      if (n0 + rp >= g.rows_p) op.flags |= F_LAST;
      // A = delta_q
      if (q == nh) { op.a_off = sm.st; op.a_stride = sm.st_stride; op.a_net = sm.st_net; }
      else { hidden_buffer(q, &op.a_off, &op.a_stride); op.a_net = R * op.a_stride; }
      if (to_gu) {
        op.flags |= F_TO_GU;
        op.o_off = sm.gu; op.o_stride = sm.gu_stride; op.o_net = sm.gu_net;
        op.kout = lg.nK;
        op.act = 0;
        // partial sums of a chunked reduction can live in gu itself
        op.d_off = sm.gu; op.d_stride = sm.gu_stride; op.d_net = sm.gu_net;
      } else {
        hidden_buffer(q - 1, &op.h_off, &op.h_stride);
        op.h_net = R * op.h_stride;
        op.kout = g.in_dim;
        op.act = d->act;
        op.d_off = dbuf_off; op.d_stride = dbuf_stride; op.d_net = R * dbuf_stride;
      }
      op.rows = std::max(0, std::min(rp, g.out_dim - n0));
      op.rows_p = rp; op.n0 = n0;
      op.K = g.in_dim; op.Kc = g.Kc; op.Ks = g.Ks;
      choose_dgrad(op.kout, rp, &op.tn, &op.split);
      ops.push_back(op);
      RnvpChunk c;
      memset(&c, 0, sizeof(c));
      for (int net = 0; net < 2; ++net) { c.w_src[net] = g.w_off[net] + n0 * g.Ks; c.b_src[net] = g.b_off[net] + n0; }
      c.rows_p = rp; c.Ks = g.Ks;
      chunks.push_back(c);
    }
  }

  void emit_wgrad(int i, int q) {
    const LayerGeom& lg = d->layers[i];
    const LinearGeom& g = lg.lin[q];
    const int nh = d->nh;
    RnvpOp op = base_op(OP_WGRAD, i);
    if (q == nh) { op.a_off = sm.st; op.a_stride = sm.st_stride; op.a_net = sm.st_net; }
    else { hidden_buffer(q, &op.a_off, &op.a_stride); op.a_net = R * op.a_stride; }
    if (q == 0) { op.h_off = sm.ub; op.h_stride = sm.ub_stride; op.h_net = 0; }
    else { hidden_buffer(q - 1, &op.h_off, &op.h_stride); op.h_net = R * op.h_stride; }
    op.rows = g.out_dim; op.rows_p = g.rows_p; op.n0 = 0;
    op.K = g.in_dim; op.Kc = g.Kc; op.Ks = g.Ks;
    for (int net = 0; net < 2; ++net) { op.g_w[net] = g.w_off[net]; op.g_b[net] = g.b_off[net]; }
    choose_wgrad(g.rows_p, g.Kc, R, &op.tn, &op.split);
    ops.push_back(op);
  }

  void emit_forward_layer(int i, bool stash) {
    const LayerGeom& lg = d->layers[i];
    ops.push_back(base_op(OP_BUILD_U, i));
    for (int q = 0; q <= d->nh; ++q) emit_linear(i, q, 0);
    RnvpOp c = base_op(OP_COUPLE_F, i);
    c.split = std::min(32, pow2ceil(lg.nT));
    if (stash) { c.flags |= F_STASH; c.stash_off = stash_off[i]; }
    ops.push_back(c);
  }

  void build() {
    const int nh = d->nh;
    ops.clear();
    chunks.clear();
    stash_off.assign(d->L, 0);
    stash_per_cta = 0;
    for (int i = l0; i < l1; ++i) { stash_off[i] = stash_per_cta; stash_per_cta += R * d->layers[i].nT; }
    stash_per_cta = ceil4(std::max(stash_per_cta, 4));

    ops.push_back(base_op(OP_LOAD, -1));
    if (mode == 0 || mode == 2) {
      for (int i = l0; i < l1; ++i)
        if (d->layers[i].nT > 0) emit_forward_layer(i, mode == 2);
      RnvpOp s = base_op(OP_STORE_F, -1);
      s.split = std::min(32, pow2ceil(d->D));
      ops.push_back(s);
    }
    if (mode == 1) {
      for (int i = l1 - 1; i >= l0; --i) {
        if (d->layers[i].nT == 0) continue;
        ops.push_back(base_op(OP_BUILD_U, i));
        for (int q = 0; q <= nh; ++q) emit_linear(i, q, 0);
        ops.push_back(base_op(OP_COUPLE_G, i));
      }
      ops.push_back(base_op(OP_STORE_G, -1));
    }
    if (mode == 2) {
      int prev_with_gu = -1;
      for (int i = l1 - 1; i >= l0; --i) {
        const LayerGeom& lg = d->layers[i];
        if (lg.nT == 0) continue;
        RnvpOp b = base_op(OP_BUILD_U, i);
        b.flags = F_RESTORE;
        b.stash_off = stash_off[i];
        if (prev_with_gu == i + 1) b.flags |= F_ADDGU;
        ops.push_back(b);
        for (int q = 0; q < nh; ++q) emit_linear(i, q, 0);
        emit_linear(i, nh, F_NET_S_ONLY);
        ops.push_back(base_op(OP_COUPLE_B, i));
        for (int q = nh; q >= 0; --q) {
          emit_wgrad(i, q);
          if (q > 0) emit_dgrad(i, q, false);
          else if (i > l0 && lg.nK > 0) { emit_dgrad(i, 0, true); prev_with_gu = i; }
        }
      }
    }
  }
};


}  // namespace rnvp_planner
