// Discretised-logistic-mixture sample of one action dimension, action_decoder_logistic.py:238-266.  Shared by
// dlm_sample_kernel (losses.cu) and the rollout decoder step (rollout.cu), so both turn the same logits and uniforms
// into the same action bit for bit.
#pragma once

namespace tacorl {

constexpr int kMix = 10;    // n_mixtures (config/networks/action_decoder/logistic.yaml:2)
constexpr float kLogSigMin = -5.f;

// L: one logits row [prob A*10 | mean A*10 | log_scale A*10 | gripper 2]; u1: the 10 Gumbel uniforms of dimension d,
// u2: its logistic uniform, both on [0, 1).
template <typename U1>
__device__ __forceinline__ float dlm_sample_dim(const float* L, int A, int d, U1 u1, float u2) {
  const float r1 = 1e-5f, r2 = 1.f - 1e-5f;
  int best = 0; float bv = -INFINITY;
#pragma unroll
  for (int k = 0; k < kMix; ++k) {
    const float t = (r1 - r2) * u1(k) + r2;
    const float v = L[d * kMix + k] - logf(-logf(t));
    if (v > bv) { bv = v; best = k; }
  }
  const float mu = L[A * kMix + d * kMix + best];
  const float s = fmaxf(L[2 * A * kMix + d * kMix + best], kLogSigMin);
  const float u = (r1 - r2) * u2 + r2;
  return mu + expf(s) * (logf(u) - logf(1.f - u));
}

__device__ __forceinline__ float dlm_gripper(const float* L, int A, float grip_lo, float grip_hi) {
  return (L[3 * A * kMix + 1] > L[3 * A * kMix]) ? grip_hi : grip_lo;
}

}  // namespace tacorl
