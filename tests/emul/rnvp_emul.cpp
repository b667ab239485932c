// TEST INFRASTRUCTURE ONLY -- host emulator of the per-tile op programs.
//
// The build container has no GPU, so this executes the *same* program the planner
// (probaforms_b200/csrc/rnvp_planner.h) hands to the CUDA tile kernel, op by op, with plain scalar
// loops over an emulated shared-memory array that starts out as NaN (any read of a location the
// program never wrote poisons the result).  It checks the planner -- offsets, strides, chunking,
// stash, flags, packed layout maps -- against the oracle before GPU time is spent; it says nothing
// about the device micro-kernels, which only the -m gpu tests cover.  Never loaded by the product.
#include <math.h>
#include <stdio.h>
#include <limits>
#include <vector>

#include "../../probaforms_b200/csrc/rnvp_planner.h"

using namespace rnvp_planner;

namespace {

struct Emu {
  const FlowGeom* g;
  Builder* b;
  std::vector<float> sm, packed, gpacked, stash, slot;
  const float *X, *C;
  const long long* idx;
  long long N;
  float scale;
  float *out_x, *out_logdet, *out_logp;
  double loss_sum = 0;
  int mode, R;

  float act(float v, int a) const { return a == 1 ? tanhf(v) : (a == 2 ? fmaxf(v, 0.f) : v); }
  float actp(float h, int a) const { return a == 1 ? 1.f - h * h : (a == 2 ? (h > 0.f ? 1.f : 0.f) : 1.f); }

  void load_chunk(const RnvpChunk& c) {
    slot.assign(b->slot_floats, std::numeric_limits<float>::quiet_NaN());
    const int wn = c.rows_p * c.Ks;
    for (int net = 0; net < 2; ++net) {
      for (int i = 0; i < wn; ++i) slot[net * wn + i] = packed[c.w_src[net] + i];
      for (int i = 0; i < c.rows_p; ++i) slot[2 * wn + net * c.rows_p + i] = packed[c.b_src[net] + i];
    }
  }

  void run_tile(long long row0) {
    const RnvpSmem& s = b->sm;
    const int D = g->D, Cd = g->Cd;
    for (const RnvpOp& op : b->ops) {
      if (op.chunk >= 0) load_chunk(b->chunks[op.chunk]);
      switch (op.kind) {
        case OP_LOAD:
          for (int r = 0; r < R; ++r) {
            const long long row = row0 + r;
            const long long src = row < N ? (idx ? idx[row] : row) : -1;
            for (int j = 0; j < D; ++j) sm[s.xs + r * s.xs_stride + j] = src >= 0 ? X[src * D + j] : 0.f;
            for (int j = 0; j < Cd; ++j) sm[s.cs + r * s.cs_stride + j] = src >= 0 ? C[src * Cd + j] : 0.f;
            sm[s.ld + r] = 0.f;
          }
          break;
        case OP_BUILD_U:
          for (int r = 0; r < R; ++r) {
            if (op.flags & F_ADDGU)
              for (int kk = 0; kk < op.nT; ++kk)
                sm[s.gx + r * s.xs_stride + 2 * kk + op.par] +=
                    sm[s.gu + r * s.gu_stride + kk] + sm[s.gu + s.gu_net + r * s.gu_stride + kk];
            if (op.flags & F_RESTORE)
              for (int ii = 0; ii < op.nT; ++ii)
                sm[s.xs + r * s.xs_stride + 2 * ii + op.par] = stash[op.stash_off + r * op.nT + ii];
            for (int kk = 0; kk < op.Kc; ++kk) {
              float v = 0.f;
              if (kk < op.nK) v = sm[s.xs + r * s.xs_stride + 2 * kk + (1 - op.par)];
              else if (kk < op.nK + Cd) v = sm[s.cs + r * s.cs_stride + kk - op.nK];
              sm[s.ub + r * s.ub_stride + kk] = v;
            }
          }
          break;
        case OP_LINEAR:
          for (int net = 0; net < 2; ++net) {
            if ((op.flags & F_NET_S_ONLY) && net == 0) continue;
            const float* W = slot.data() + net * op.rows_p * op.Ks;
            const float* B = slot.data() + 2 * op.rows_p * op.Ks + net * op.rows_p;
            for (int r = 0; r < R; ++r)
              for (int n = 0; n < op.rows_p; ++n) {
                float acc = 0.f;
                for (int k = 0; k < op.Kc; ++k) acc += sm[op.a_off + net * op.a_net + r * op.a_stride + k] * W[n * op.Ks + k];
                sm[op.o_off + net * op.o_net + r * op.o_stride + op.n0 + n] = act(acc + B[n], op.act);
              }
          }
          break;
        case OP_COUPLE_F:
          for (int r = 0; r < R; ++r)
            for (int ii = 0; ii < op.nT; ++ii) {
              float& x = sm[s.xs + r * s.xs_stride + 2 * ii + op.par];
              const float t = sm[s.st + r * s.st_stride + ii], sv = sm[s.st + s.st_net + r * s.st_stride + ii];
              if (op.flags & F_STASH) stash[op.stash_off + r * op.nT + ii] = x;
              x = x * expf(sv) + t;
              sm[s.ld + r] += sv;
            }
          break;
        case OP_COUPLE_G:
          for (int r = 0; r < R; ++r)
            for (int ii = 0; ii < op.nT; ++ii) {
              float& x = sm[s.xs + r * s.xs_stride + 2 * ii + op.par];
              const float t = sm[s.st + r * s.st_stride + ii], sv = sm[s.st + s.st_net + r * s.st_stride + ii];
              x = (x - t) * expf(-sv);
            }
          break;
        case OP_STORE_F:
          for (int r = 0; r < R; ++r) {
            const bool valid = row0 + r < N;
            float q = 0.f;
            for (int j = 0; j < D; ++j) { const float z = sm[s.xs + r * s.xs_stride + j]; q += z * z; }
            const float ld = sm[s.ld + r];
            const float lp = ld - 0.5f * (D * 1.8378770664093453f + q);
            if (valid) {
              if (mode == 0 && out_x) for (int j = 0; j < D; ++j) out_x[(row0 + r) * D + j] = sm[s.xs + r * s.xs_stride + j];
              if (out_logdet) out_logdet[row0 + r] = ld;
              if (out_logp) out_logp[row0 + r] = lp;
              loss_sum += lp;
            }
            if (mode == 2) {
              sm[s.ld + r] = valid ? scale : 0.f;
              for (int j = 0; j < D; ++j) sm[s.gx + r * s.xs_stride + j] = valid ? -scale * sm[s.xs + r * s.xs_stride + j] : 0.f;
            }
          }
          break;
        case OP_STORE_G:
          for (int r = 0; r < R; ++r)
            if (row0 + r < N) for (int j = 0; j < D; ++j) out_x[(row0 + r) * D + j] = sm[s.xs + r * s.xs_stride + j];
          break;
        case OP_COUPLE_B: {
          const int nTp = (op.nT + 3) & ~3;
          for (int r = 0; r < R; ++r)
            for (int ii = 0; ii < nTp; ++ii) {
              float dt = 0.f, ds = 0.f;
              if (ii < op.nT) {
                float& gy = sm[s.gx + r * s.xs_stride + 2 * ii + op.par];
                const float x = sm[s.xs + r * s.xs_stride + 2 * ii + op.par];
                const float es = expf(sm[s.st + s.st_net + r * s.st_stride + ii]);
                dt = gy; ds = gy * x * es + sm[s.ld + r]; gy = gy * es;
              }
              sm[s.st + r * s.st_stride + ii] = dt;
              sm[s.st + s.st_net + r * s.st_stride + ii] = ds;
            }
        } break;
        case OP_WGRAD:
          for (int net = 0; net < 2; ++net)
            for (int n = 0; n < op.rows_p; ++n) {
              float bsum = 0.f;
              for (int r = 0; r < R; ++r) bsum += sm[op.a_off + net * op.a_net + r * op.a_stride + n];
              gpacked[op.g_b[net] + n] += bsum;
              for (int k = 0; k < op.Kc; ++k) {
                float acc = 0.f;
                for (int r = 0; r < R; ++r)
                  acc += sm[op.a_off + net * op.a_net + r * op.a_stride + n] * sm[op.h_off + net * op.h_net + r * op.h_stride + k];
                gpacked[op.g_w[net] + n * op.Ks + k] += acc;
              }
            }
          break;
        case OP_DGRAD: {
          const int kc = (op.kout + 3) & ~3;
          for (int net = 0; net < 2; ++net) {
            const float* W = slot.data() + net * op.rows_p * op.Ks;
            for (int r = 0; r < R; ++r)
              for (int k = 0; k < kc; ++k) {
                float v = 0.f;
                for (int n = 0; n < op.rows_p; ++n) v += sm[op.a_off + net * op.a_net + r * op.a_stride + op.n0 + n] * W[n * op.Ks + k];
                if (!(op.flags & F_FIRST)) v += sm[op.d_off + net * op.d_net + r * op.d_stride + k];
                if (op.flags & F_LAST) {
                  if (op.flags & F_TO_GU) sm[op.o_off + net * op.o_net + r * op.o_stride + k] = v;
                  else {
                    float& h = sm[op.h_off + net * op.h_net + r * op.h_stride + k];
                    h = v * actp(h, op.act);
                  }
                } else sm[op.d_off + net * op.d_net + r * op.d_stride + k] = v;
              }
          }
        } break;
        default: break;
      }
    }
  }
};

}  // namespace

extern "C" int rnvp_emulate(int mode, int D, int Cd, int L, int nh, const int* hidden, int act, int TR_force,
                            const float* flat, const float* X, const float* C, const long long* idx, long long N,
                            int l0, int l1, float scale, float* out_x, float* out_logdet, float* out_logp,
                            float* gflat, double* loss_sum, int* info /* [TR, smem_bytes, n_ops, n_chunks, packed, ops past a layer's first weight-row chunk] */) {
  FlowGeom g;
  g.D = D; g.Cd = Cd; g.L = L; g.nh = nh; g.act = act;
  for (int q = 0; q < nh; ++q) g.hidden[q] = hidden[q];
  build_layout(&g);
  std::vector<int> p2f, f2p;
  build_maps(&g, p2f, f2p);
  Builder b;
  b.d = &g; b.mode = mode; b.l0 = l0; b.l1 = l1;
  const bool ok = b.plan_best(TR_force);
  if (!ok) return -2;
  b.build();
  if (info) { info[0] = b.TR; info[1] = b.sm.total_floats * 4; info[2] = (int)b.ops.size(); info[3] = (int)b.chunks.size(); info[4] = (int)g.packed;
    info[5] = 0;
    for (const RnvpOp& op : b.ops) info[5] += op.n0 > 0;
  }
  Emu e;
  e.g = &g; e.b = &b; e.mode = mode; e.R = b.R;
  e.X = X; e.C = C; e.idx = idx; e.N = N; e.scale = scale;
  e.out_x = out_x; e.out_logdet = out_logdet; e.out_logp = out_logp;
  const float nan = std::numeric_limits<float>::quiet_NaN();
  e.sm.assign(b.sm.total_floats, nan);
  e.stash.assign(b.stash_per_cta, nan);
  e.packed.assign(g.packed_gather, 0.f);
  for (int64_t p = 0; p < g.packed_gather; ++p) e.packed[p] = p2f[p] >= 0 ? flat[p2f[p]] : 0.f;
  e.gpacked.assign(g.packed_tile, 0.f);
  for (long long row0 = 0; row0 < N; row0 += b.R) e.run_tile(row0);
  if (gflat) for (int64_t f = 0; f < g.P; ++f) gflat[f] = f2p[f] >= 0 ? e.gpacked[f2p[f]] : 0.f;
  if (loss_sum) *loss_sum = e.loss_sum;
  return 0;
}

namespace {
// FNV-1a over raw bytes: a stable fingerprint of a layout map or an op program
uint64_t fnv1a(const void* p, size_t n, uint64_t h = 1469598103934665603ull) {
  const unsigned char* b = (const unsigned char*)p;
  for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
  return h;
}
}  // namespace

// Tensor-core layout and FP32 programs of a one-hidden-layer flow as rnvp_desc_create builds them
// (default max_smem).  out[26]: mma_ok, mDH, mK1P, mNTP, m_w1_floats, m_w2_floats, m_wt_floats, m_layer_floats,
// mma_off, mma_floats, packed, packed_tile, small_ok, digest of build_mma_map's m2f, then per FP32 mode 0, 1, 2:
// planned (0/1), TR, shared-memory bytes, digest of the smem carve-up, ops and chunks.
extern "C" int rnvp_emul_tc_layout(int D, int Cd, int L, int H, int act, long long* out) {
  FlowGeom g;
  g.D = D; g.Cd = Cd; g.L = L; g.nh = 1; g.act = act; g.hidden[0] = H;
  build_layout(&g);
  std::vector<int> m2f;
  build_mma_map(&g, m2f);
  const long long head[14] = {g.mma_ok, g.mDH, g.mK1P, g.mNTP, g.m_w1_floats, g.m_w2_floats, g.m_wt_floats, g.m_layer_floats,
                              g.mma_off, g.mma_floats, g.packed, g.packed_tile, g.small_ok,
                              (long long)fnv1a(m2f.data(), m2f.size() * sizeof(int))};
  for (int k = 0; k < 14; ++k) out[k] = head[k];
  for (int mode = 0; mode < 3; ++mode) {
    long long* o = out + 14 + 4 * mode;
    Builder b;
    b.d = &g; b.mode = mode; b.l0 = 0; b.l1 = L;
    if (!b.plan_best(0)) { o[0] = 0; o[1] = o[2] = o[3] = -1; continue; }
    b.build();
    o[0] = 1; o[1] = b.TR; o[2] = (long long)b.sm.total_floats * 4;
    uint64_t h = fnv1a(&b.sm, sizeof(b.sm));
    h = fnv1a(b.ops.data(), b.ops.size() * sizeof(RnvpOp), h);
    o[3] = (long long)fnv1a(b.chunks.data(), b.chunks.size() * sizeof(RnvpChunk), h);
  }
  return 0;
}

// Which tcgen05 image entries carry RNVP_IMG_SCALED.  out[4]: mapped entries of the forward W1 images, of them the
// scaled ones, mapped entries of every other image, of them the scaled ones.
extern "C" int rnvp_emul_img_scaled(int D, int Cd, int L, int H, int act, long long* out) {
  FlowGeom g;
  g.D = D; g.Cd = Cd; g.L = L; g.nh = 1; g.act = act; g.hidden[0] = H;
  build_layout(&g);
  if (!g.mma_ok) return -1;
  std::vector<int> m2f;
  build_mma_map(&g, m2f);
  for (int k = 0; k < 4; ++k) out[k] = 0;
  for (size_t m = 0; m < m2f.size(); ++m) {
    if (m2f[m] < 0) continue;
    const int q = (int)(m % g.m_layer_floats) < g.m_w1_floats ? 0 : 2;
    out[q] += 1;
    out[q + 1] += (m2f[m] & RNVP_IMG_SCALED) ? 1 : 0;
  }
  return 0;
}

// Row-per-thread small-flow layout of a one-hidden-layer flow as rnvp_desc_create builds it.  head[8]: small_ok, sNE, sNC,
// srec, snet, small_floats, small_off, P.  When small_ok and the buffers are given, s2f[small_floats] receives the flat
// index held by each slot of the small region (or -1) and f2p2[P] the absolute packed index of each parameter's small-layout
// copy (or -1).  Call once with null buffers to learn the sizes.
extern "C" int rnvp_emul_small_layout(int D, int Cd, int L, int H, long long* head, int* s2f, int* f2p2) {
  FlowGeom g;
  g.D = D; g.Cd = Cd; g.L = L; g.nh = 1; g.act = 1; g.hidden[0] = H;
  build_layout(&g);
  const long long h[8] = {g.small_ok, g.sNE, g.sNC, g.srec, g.snet, g.small_floats, g.small_off, g.P};
  for (int k = 0; k < 8; ++k) head[k] = h[k];
  if (!g.small_ok || !s2f || !f2p2) return 0;
  std::vector<int> p2f(g.packed_gather, -1), f2p2v;
  build_small_map(&g, p2f, f2p2v);
  for (int k = 0; k < g.small_floats; ++k) s2f[k] = p2f[g.small_off + k];
  for (int64_t f = 0; f < g.P; ++f) f2p2[f] = f2p2v[f];
  return 0;
}

extern "C" long long rnvp_emul_param_count(int D, int Cd, int L, int nh, const int* hidden) {
  FlowGeom g;
  g.D = D; g.Cd = Cd; g.L = L; g.nh = nh; g.act = 1;
  for (int q = 0; q < nh; ++q) g.hidden[q] = hidden[q];
  build_layout(&g);
  return g.P;
}
