// Discrete open/close gripper head of the flat-CQL baseline (SURVEY.md 8f-4):
//   GumbelSoftmax(temperature 0.5, logits) of /root/reference/src/tacorl/utils/distributions.py:15-58 as used by
//   Actor.get_actions / sample_n_with_log_prob / log_prob, networks/actor_critic/actor.py:66-156.
// Only the class index of a draw is ever used by the reference (rsample(hard=True) is followed by argmax, :84-85), so a
// draw is argmax(normalised logits + Gumbel(u)); the log-probability of a class index is log_softmax(logits)[index].
// Noise (the uniforms) is an input, like every other random quantity of this library.
#include "common.cuh"
#include "internal.h"
#include "gripper.cuh"
#include "../../include/tacorl_b200.h"

namespace tacorl {

// index[r] = argmax_c(norm_logits[r % rows0][c] - log(-log(u[r][c]))); ties -> class 0 (torch.argmax: first maximum).
// clamp_u: u clamped to [eps, 1 - eps] first (torch.distributions.utils.clamp_probs, the rsample path).
__global__ void gripper_gumbel_kernel(int rows, int rows0, const float* __restrict__ logits, const float* __restrict__ u,
                                      int clamp_u, float* __restrict__ index, float* __restrict__ action) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int r0 = r % rows0;
  float n0, n1;
  gr_normalise(logits[2 * r0], logits[2 * r0 + 1], n0, n1);
  float u0 = u[2 * r], u1 = u[2 * r + 1];
  if (clamp_u) {
    const float eps = 1.1920928955078125e-07f;       // torch.finfo(torch.float32).eps
    u0 = fminf(fmaxf(u0, eps), 1.f - eps);
    u1 = fminf(fmaxf(u1, eps), 1.f - eps);
  }
  const float s0 = n0 - logf(-logf(u0)), s1 = n1 - logf(-logf(u1));
  const float c = s1 > s0 ? 1.f : 0.f;
  if (index) index[r] = c;
  if (action) action[r] = 2.f * c - 1.f;
}

// logp[r] = log_softmax(logits[r % rows0])[index[r]];  index given as a class id (0 / 1) in a float
__global__ void gripper_logprob_kernel(int rows, int rows0, const float* __restrict__ logits,
                                       const float* __restrict__ index, float* __restrict__ logp) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int r0 = r % rows0;
  const float l0 = logits[2 * r0], l1 = logits[2 * r0 + 1];
  const float m = fmaxf(l0, l1);
  const float lse = logf(expf(l0 - m) + expf(l1 - m));
  logp[r] = (index[r] >= 0.5f ? l1 : l0) - m - lse;
}

// d logits[r][c] = dlogp[r] * ([c == index[r]] - softmax(logits[r])[c])     (rows == rows0)
__global__ void gripper_logprob_bwd_kernel(int rows, const float* __restrict__ logits, const float* __restrict__ index,
                                           const float* __restrict__ dlogp, float* __restrict__ dlogits) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float l0 = logits[2 * r], l1 = logits[2 * r + 1];
  const float m = fmaxf(l0, l1);
  const float e0 = expf(l0 - m), e1 = expf(l1 - m);
  const float inv = 1.f / (e0 + e1);
  const float hot1 = index[r] >= 0.5f ? 1.f : 0.f;
  const float d = dlogp[r];
  dlogits[2 * r] = d * ((1.f - hot1) - e0 * inv);
  dlogits[2 * r + 1] = d * (hot1 - e1 * inv);
}

}  // namespace tacorl

using namespace tacorl;

extern "C" {

int tacorl_gripper_gumbel(int rows, int rows0, const float* logits, const float* u, int clamp_u, float* index,
                          float* action, void* stream) {
  TACORL_REQUIRE(rows >= 0 && rows0 >= 1 && rows % rows0 == 0, "gripper_gumbel: rows %d is not a multiple of %d", rows, rows0);
  TACORL_REQUIRE(logits && u && (index || action), "gripper_gumbel: null pointer");
  if (rows == 0) return 0;
  gripper_gumbel_kernel<<<cdiv(rows, 128), 128, 0, (cudaStream_t)stream>>>(rows, rows0, logits, u, clamp_u, index, action);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_gripper_logprob(int rows, int rows0, const float* logits, const float* index, float* logp, void* stream) {
  TACORL_REQUIRE(rows >= 0 && rows0 >= 1 && rows % rows0 == 0, "gripper_logprob: rows %d is not a multiple of %d", rows, rows0);
  TACORL_REQUIRE(logits && index && logp, "gripper_logprob: null pointer");
  if (rows == 0) return 0;
  gripper_logprob_kernel<<<cdiv(rows, 128), 128, 0, (cudaStream_t)stream>>>(rows, rows0, logits, index, logp);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_gripper_logprob_bwd(int rows, const float* logits, const float* index, const float* dlogp, float* dlogits,
                               void* stream) {
  TACORL_REQUIRE(logits && index && dlogp && dlogits, "gripper_logprob_bwd: null pointer");
  if (rows == 0) return 0;
  gripper_logprob_bwd_kernel<<<cdiv(rows, 128), 128, 0, (cudaStream_t)stream>>>(rows, logits, index, dlogp, dlogits);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
