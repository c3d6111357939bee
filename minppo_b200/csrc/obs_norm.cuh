// minppo_b200 -- running observation normalization (include/minppo_b200.h, minppo_obs_norm): the per-element transform
// shared by the observation image kernel (adam.cu) and the fused policy step (policy_fused.cuh).
//   s_j = 1 / sqrt(var_j + eps),  y = clamp((x - mean_j) * s_j, -clip, clip)   (clip <= 0: no clamp)
// Every operation is an explicitly rounded fp32 intrinsic, so that NumPy float32 (oracle/ppo_numpy.py normalize_obs)
// reproduces the result bit for bit whatever the compiler's contraction settings.
#pragma once

#include <cuda_runtime.h>

namespace minppo {

__device__ __forceinline__ float obs_norm_scale(float var, float eps) {
  return __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var, eps)));
}

__device__ __forceinline__ float obs_norm_apply(float x, float mean, float scale, float clip) {
  float y = __fmul_rn(__fsub_rn(x, mean), scale);
  if (clip > 0.f) y = fminf(fmaxf(y, -clip), clip);
  return y;
}

}  // namespace minppo
