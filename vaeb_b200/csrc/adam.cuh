// Adam (Kingma & Ba 2015, Algorithm 1) in the ascent convention of the reference's rules, with the weight prior folded
// into the gradient as getUpdates does (VAEB.py:389-390).  One definition for the flat kernel (kernels_small.cu) and the
// large-batch tail (tc_tail.cu), so that both compute the same bits per element.
#pragma once
#include <cuda_runtime.h>

// alpha_t = lr / (1 - b1^t) and s2_t = sqrt(1 - b2^t) are computed on the host in double: with them,
// p + alpha_t m / (sqrt(v) / s2_t + eps) is torch.optim.Adam(maximize=True)'s step.
__device__ __forceinline__ void adam1(float& p, float& m, float& v, float g, float alpha_t, float s2_t, float b1,
                                      float b2, float eps, float prior) {
  g -= prior * p;
  m = b1 * m + (1.0f - b1) * g;
  v = b2 * v + (1.0f - b2) * g * g;
  p += alpha_t * m / (sqrtf(v) / s2_t + eps);
}
