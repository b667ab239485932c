// torch.optim.RMSprop single-tensor update (torch/optim/rmsprop.py _single_tensor_rmsprop; momentum 0, not centred) for
// one parameter: the tail of the ConditionalWGAN fit step (rnvp_wgan.cu).
#pragma once

struct RnvpRmspropCoef {
  float lr, alpha, one_minus_alpha, eps, wd;
};

__device__ __forceinline__ float rnvp_rmsprop_update(float g, float th, float& sq, const RnvpRmspropCoef& k) {
  if (k.wd != 0.0f) g = fmaf(k.wd, th, g);                  // grad.add(param, alpha=weight_decay)
  sq = fmaf(k.one_minus_alpha * g, g, sq * k.alpha);        // square_avg.mul_(alpha).addcmul_(grad, grad, 1-alpha)
  const float avg = __fsqrt_rn(sq) + k.eps;                 // square_avg.sqrt().add_(eps)
  return th + __fdiv_rn(-k.lr * g, avg);                    // param.addcdiv_(grad, avg, value=-lr)
}
