// GumbelSoftmax logit normalisation, shared by the discrete gripper head (gripper.cu) and the rollout policy's sampler
// (rollout.cu), so both draw the same class from the same logits and uniforms.
#pragma once

namespace tacorl {

// torch: Categorical-family `logits` are stored normalised, logits - logsumexp(logits) (max-shifted)
__device__ __forceinline__ void gr_normalise(float l0, float l1, float& n0, float& n1) {
  const float m = fmaxf(l0, l1);
  const float lse = m + logf(expf(l0 - m) + expf(l1 - m));
  n0 = l0 - lse;
  n1 = l1 - lse;
}

}  // namespace tacorl
