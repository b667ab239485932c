// Arguments of the tcgen05 forward / inverse / fit kernel (rnvp_wide.cu).
#pragma once
#include <stdint.h>

struct RnvpWideArgs {
  const float* wimg;           // per layer [W1 image | W2 image | b2 | W2T | W1T], see rnvp_planner.h build_mma_map
  const float* X;              // rows (forward) or latent noise (inverse), [N][D]
  const float* C;              // [N][Cd] or nullptr
  const long long* idx;        // optional row gather
  long long N;
  float* out_x;                // z / x
  float* out_logdet;
  float* out_logp;
  int Cd, H, l0, l1;
  int layer_floats, w1_floats, w2_floats;
  int n_tiles;                 // 128-row tiles
  // MODE 2 (fit step): per layer the row's x_T (before the coupling) and s go to a global stash that the kernel's own
  // backward sweep reads back, blocked by 32 rows: [row / 32][layer][x_T | s as 2 DH / 4 float4 groups][row % 32][4];
  // the sum of logp accumulates atomically
  float* stash;
  float* loss_sum;
  int L_total;                 // layers of the flow (stash block = L_total * 2 * DH * 32 floats)
  // MODE 2 with do_bwd: the kernel continues with the backward sweep (everything but the weight gradients): per (layer,
  // row) it leaves a record [h 2H | u K1P8 | delta2 2*DH] in the blocked records array for rnvp_wgrad_tc_kernel
  int do_bwd;
  float scale;                 // d(out)/d(logp_row): g_logdet = scale, g_z = -scale*z
  float* records;
  int rec;
  long long Npad;
  int wt_floats;               // floats of one transposed image (W2T, then W1T) per layer; 0 unless do_bwd
  // MODE 1 with X == nullptr: latent rows drawn in-kernel (rnvp_philox.cuh), keyed on row_offset + row
  unsigned long long seed;
  long long row_offset;
  int Dreal;                   // features per row in memory (< 2 * DH for padded shapes, the row loads are guarded)
};
