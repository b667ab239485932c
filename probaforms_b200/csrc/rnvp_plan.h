// Shared host/device structures for the fused RealNVP tile kernels.
//
// Vocabulary follows the reference (probaforms/models/realnvp.py): a *flow* is a
// stack of L *coupling layers*; layer i has mask m_i[j] = (j+i)%2 (realnvp.py:199),
// keep-set K_i = {j : m_i[j]=1} (conditioning half, passed through) and
// transform-set T_i = {j : m_i[j]=0}.  Each layer owns two conditioner nets,
// nn_t and nn_s (realnvp.py:69-70), i.e. chains of Linear(+activation).
#pragma once
#include <stdint.h>

#define RNVP_MAX_HIDDEN 8          // max number of hidden layers in a conditioner
#define RNVP_THREADS 256           // threads per CTA: 128 per conditioner net (t, s)
#define RNVP_NET_THREADS 128
#define RNVP_NSLOTS 2              // weight ring depth (TMA bulk copies, mbarrier-tracked)

// ---- op kinds of the per-tile program -------------------------------------
enum RnvpOpKind {
  OP_LOAD = 0,        // rows of X (or noise) and C -> smem
  OP_BUILD_U = 1,     // u = [x_K, c]  (realnvp.py:91-94)  (+ restore x_T / add du in the backward sweep)
  OP_LINEAR = 2,      // one Linear(+act) of nn_t and nn_s, weight chunk from the ring
  OP_COUPLE_F = 3,    // y_T = x_T*exp(s)+t, logdet += sum s   (realnvp.py:99-100)
  OP_COUPLE_G = 4,    // x_T = (y_T-t)*exp(-s)                 (realnvp.py:128)
  OP_STORE_F = 5,     // z, logdet, logp = logdet + N(0,I).log_prob(z)  (nflow.py:115)
  OP_STORE_G = 6,     // x
  OP_COUPLE_B = 8,    // d(coupling): delta2_t, delta2_s, g_x_T
  OP_WGRAD = 9,       // dW, db of one Linear (both nets) -> red.global.add into packed grads
  OP_DGRAD = 10,      // delta_{q-1} = (delta_q W_q) * act'(h_{q-1})  /  du for q = 0
  OP_ADD_GU = 11      // g_x_K += du_t + du_s (only used stand-alone after the last layer processed)
};

enum RnvpOpFlags {
  F_RESTORE = 1,      // BUILD_U: first put x_T back from the stash (backward sweep)
  F_ADDGU = 2,        // BUILD_U: first add the previous layer's du into g_x
  F_STASH = 4,        // COUPLE_F: save x_T of this layer for the backward sweep
  F_FIRST = 8,        // DGRAD: first chunk of the reduction
  F_LAST = 16,        // DGRAD: last chunk of the reduction
  F_TO_GU = 32,       // DGRAD: q = 0, result is du (input gradient), no act'
  F_NET_S_ONLY = 64   // LINEAR: only nn_s needs this output (t is unused in the backward sweep)
};

struct RnvpOp {
  int kind, layer, flags, chunk;      // chunk: index into the tile's weight-chunk sequence, -1 if none
  int a_off, a_stride, a_net;         // A operand (activations / deltas) in smem, float offsets
  int o_off, o_stride, o_net;         // output in smem
  int h_off, h_stride, h_net;         // DGRAD: h_{q-1} (act' and in-place result); WGRAD: the Linear's input
  int d_off, d_stride, d_net;         // DGRAD: partial-sum scratch when the reduction is chunked
  int rows, rows_p, n0;               // weight rows in this chunk (true / padded to 4), first row
  int K, Kc, Ks;                      // in_dim, ceil4(in_dim), weight row stride (== 4 mod 8)
  int tn, split;                      // micro-tile variant and split-K factor (1,2,4)
  int act;                            // 0 none, 1 tanh, 2 relu
  int nK, nT, par, stash_off;         // layer sets: |K|, |T|, parity (T = {j : j%2 == par}), stash offset
  int g_w[2], g_b[2];                 // WGRAD: packed-gradient offsets of W_t, W_s, b_t, b_s
  int kout;                           // DGRAD: number of output columns wanted
  int pad0, pad1, pad2;
};

struct RnvpChunk {
  int w_src[2], b_src[2];             // packed-parameter float offsets (per net) of this row chunk
  int rows_p, Ks;                     // padded rows, row stride
  int pad0, pad1;
};

// smem carve-up (float offsets) chosen by the host planner for one (shape, mode, TR)
struct RnvpSmem {
  int xs, xs_stride;                  // current x  [R][xs_stride]
  int cs, cs_stride;                  // condition  [R][cs_stride]
  int gx;                             // g_x        [R][xs_stride]          (backward)
  int ub, ub_stride;                  // u=[x_K,c]  [R][ub_stride]
  int ld;                             // logdet     [R]
  int st, st_stride, st_net;          // t / s (and delta2)  [2][R][st_stride]
  int gu, gu_stride, gu_net;          // du per net [2][R][gu_stride]        (backward)
  int wring, slot_floats;             // weight ring [NSLOTS][slot_floats]
  int mbar;                           // NSLOTS mbarriers (8 B each), float offset (even)
  int red;                            // 8 floats of CTA reduction scratch
  int total_floats;
};

struct RnvpKArgs {
  const float* packed;                // packed parameters (see rnvp_layout)
  const RnvpOp* ops;
  const RnvpChunk* chunks;
  int n_ops, n_chunks;
  const float* X;                     // [N][D] rows (forward/backward) or noise/latent (inverse)
  const float* C;                     // [N][Cd] or nullptr
  const long long* idx;               // optional row gather (epoch permutation slice), or nullptr
  long long N;
  int n_tiles;
  float* out_x;                       // z (forward) / x (inverse), [N][D] or nullptr
  float* out_logdet;                  // [N] or nullptr
  float* out_logp;                    // [N] or nullptr
  float* gpacked;                     // packed gradient accumulator (backward)
  float* loss_sum;                    // sum over rows of logp (backward), atomically accumulated
  float* stash;                       // per-CTA x_T stash, gridDim.x * stash_per_cta floats
  int stash_per_cta;
  // 16-byte aligned: the tile kernels' register allocation depends on where the fields from here on sit (ptxas -v:
  // rnvp_tile_kernel<2, 0> needs 128 registers with this alignment and 164 without)
  alignas(16) float scale;            // backward: d(out)/d(logp_row); g_logdet = scale, g_z = -z*scale
  int D, Cd;
  // inverse program with X == nullptr: latent rows drawn in-kernel (rnvp_philox.cuh), keyed on row_offset + row
  unsigned long long seed;
  long long row_offset;
  RnvpSmem sm;
};
