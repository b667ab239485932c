// Arguments of the weight-gradient sweep kernel (rnvp_wgrad_tc.cu).
#pragma once
#include <stdint.h>

struct RnvpWgradLayer {            // where one layer's gradients live in the packed accumulator (tile layout)
  int w1_off[2], b1_off[2];        // first Linear of nn_t / nn_s: rows = hidden units, row stride Ks1
  int w2_off[2], b2_off[2];        // last Linear: rows = transformed features, row stride Ks2
  int Ks1, Ks2;
  int nK, nT;                      // real |K| and |T| of the layer (differ from DH for padded / odd D)
};

// Arguments of the tcgen05 weight-gradient sweep (rnvp_wgrad_tc.cu): records as above but with the 3-bit slot swizzle,
// [L][Npad/32][rec/4][32 slots][4], slot = row ^ (column group & 7)
struct RnvpWgradTcArgs {
  const float* gR;
  int rec;                         // floats per record = 2H + K1P8 + 2*TP
  long long Npad;                  // rows, multiple of 32; padding rows hold zeros in delta2
  int H, K1P8, K1, TP, Cd;         // hidden width; u columns (padded to 8 / real = DH + Cd); delta2 columns per net = DH; cond_size
  int n_slices, n_mblocks;         // grid = L * n_mblocks * n_slices; n_mblocks = ceil(2H / 128)
  float* gpacked;
  const float* packed;
  int act;
  const RnvpWgradLayer* layers;
  long long* trace;                // development aid (rnvp_debug_set_trace): wait accounting of CTA 0
  int one_issuer;                  // development knob: issuer A also issues the dW2 products (issuer B idles)
};
size_t rnvp_wgrad_tc_smem_bytes(int NU, int TP, int ROWS, int NBUF, int NOP, int NSLOT, int K1P8, int NN);
int rnvp_wgrad_tc_rows(int NU, int TP);   // rows per stage of the kernel variant (NU, TP): slices are cut in such stages
