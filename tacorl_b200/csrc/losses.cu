// Fused loss / distribution kernels.  Every kernel computes the forward value AND the analytic
// gradient w.r.t. its inputs in one pass (the tensors are < 1 MB: these ops are latency-bound, so
// one launch each instead of the ~20-30 aten launches the reference issues; SURVEY.md §2.3).
// Citations are into /root/reference/src/tacorl/.
#include "common.cuh"
#include "internal.h"
#include "dlm_sample.cuh"
#include "../../include/tacorl_b200.h"

namespace tacorl {

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float softplus_acc(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// ------------------------------------------------------------------------------------------
// Discretised-logistic-mixture NLL + gripper cross-entropy, fwd + grad.
// networks/action_decoders/action_decoder_logistic.py:184-235 (_logistic_loss), :114-133 (_loss).
// logits row layout (ld floats): [prob A*10 | mean A*10 | log_scale A*10 | gripper 2], A = act dims.
// One thread per (row, action dim); the dim-0 thread of a row also does the gripper CE.
// row_loss: (rows, A+1) per-term losses (already divided by rows); dlogits same layout as logits.
__global__ void dlm_nll_kernel(int rows, int A, const float* __restrict__ logits, long long ld,
                               const float* __restrict__ actions, long long lda, float half_bin, float log_half_classes,
                               float act_min, float act_max, float gripper_alpha,
                               float* __restrict__ row_loss, float* __restrict__ dlogits, long long ldd) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * A) return;
  const int r = idx / A, d = idx % A;
  const float inv_rows = 1.f / (float)rows;
  const float* L = logits + (long long)r * ld;
  float* G = dlogits ? dlogits + (long long)r * ldd : nullptr;
  const float a = actions[(long long)r * lda + d];
  float lpk[kMix], g_mu[kMix], g_s[kMix], pi[kMix];
  float pmax = -INFINITY;
#pragma unroll
  for (int k = 0; k < kMix; ++k) { pi[k] = L[d * kMix + k]; pmax = fmaxf(pmax, pi[k]); }
  float psum = 0.f;
#pragma unroll
  for (int k = 0; k < kMix; ++k) psum += expf(pi[k] - pmax);
  const float plse = pmax + logf(psum);
  float m = -INFINITY;
#pragma unroll
  for (int k = 0; k < kMix; ++k) {
    const float mu = L[A * kMix + d * kMix + k];
    const float s_raw = L[2 * A * kMix + d * kMix + k];
    const float s = fmaxf(s_raw, kLogSigMin);
    const float inv = expf(-s);
    const float c = a - mu;
    const float P = inv * (c + half_bin), M = inv * (c - half_bin), mid = inv * c;
    float lp, gP = 0.f, gM = 0.f, gm = 0.f, gs_direct = 0.f;
    if (a < act_min + 1e-3f) {
      lp = P - softplus_acc(P); gP = 1.f - sigmoid_acc(P);
    } else if (a > act_max - 1e-3f) {
      lp = -softplus_acc(M); gM = -sigmoid_acc(M);
    } else {
      const float sP = sigmoid_acc(P), sM = sigmoid_acc(M);
      const float delta = sP - sM;
      if (delta > 1e-5f) {
        lp = logf(fmaxf(delta, 1e-12f));
        gP = sP * (1.f - sP) / delta; gM = -sM * (1.f - sM) / delta;
      } else {
        lp = mid - s - 2.f * softplus_acc(mid) - log_half_classes;   // log((num_classes - 1) / 2), :231
        gm = 1.f - 2.f * sigmoid_acc(mid); gs_direct = -1.f;
      }
    }
    g_mu[k] = -inv * (gP + gM + gm);
    g_s[k] = (s_raw >= kLogSigMin) ? (-(gP * P + gM * M + gm * mid) + gs_direct) : 0.f;
    lpk[k] = lp + pi[k] - plse;
    m = fmaxf(m, lpk[k]);
  }
  float se = 0.f;
#pragma unroll
  for (int k = 0; k < kMix; ++k) se += expf(lpk[k] - m);
  const float lse = m + logf(se);
  row_loss[(long long)r * (A + 1) + d] = -lse * inv_rows;
  if (G) {
#pragma unroll
    for (int k = 0; k < kMix; ++k) {
      const float w = expf(lpk[k] - lse);
      const float sm = expf(pi[k] - plse);
      G[d * kMix + k] = -(w - sm) * inv_rows;
      G[A * kMix + d * kMix + k] = -w * g_mu[k] * inv_rows;
      G[2 * A * kMix + d * kMix + k] = -w * g_s[k] * inv_rows;
    }
  }
  if (d == 0) {  // gripper CE: class 0 if action == -1 else 1 (action_decoder_logistic.py:126-131)
    const float g0 = L[3 * A * kMix], g1 = L[3 * A * kMix + 1];
    const int cls = actions[(long long)r * lda + A] > 0.f ? 1 : 0;
    const float mx = fmaxf(g0, g1);
    const float l = mx + logf(expf(g0 - mx) + expf(g1 - mx));
    row_loss[(long long)r * (A + 1) + A] = gripper_alpha * (l - (cls ? g1 : g0)) * inv_rows;
    if (G) {
      const float p0 = expf(g0 - l), p1 = expf(g1 - l);
      G[3 * A * kMix] = gripper_alpha * (p0 - (cls == 0 ? 1.f : 0.f)) * inv_rows;
      G[3 * A * kMix + 1] = gripper_alpha * (p1 - (cls == 1 ? 1.f : 0.f)) * inv_rows;
    }
  }
}

// Mixture sampling, action_decoder_logistic.py:238-266.  u1 (rows,A,10), u2 (rows,A) ~ U[0,1).
// pred: (rows, A+1); hit: (rows) = 1 if predicted gripper sign equals the target's
// (modules/play_lmp/play_lmp_for_rl.py:165-176).
__global__ void dlm_sample_kernel(int rows, int A, const float* __restrict__ logits, long long ld,
                                  const float* __restrict__ u1, const float* __restrict__ u2,
                                  const float* __restrict__ actions, long long lda, float grip_lo,
                                  float grip_hi, float* __restrict__ pred, float* __restrict__ hit) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * A) return;
  const int r = idx / A, d = idx % A;
  const float* L = logits + (long long)r * ld;
  const float* u1d = u1 + ((long long)r * A + d) * kMix;
  pred[(long long)r * (A + 1) + d] = dlm_sample_dim(L, A, d, [&](int k) { return u1d[k]; }, u2[(long long)r * A + d]);
  if (d == 0) {
    const float g = dlm_gripper(L, A, grip_lo, grip_hi);
    pred[(long long)r * (A + 1) + A] = g;
    if (hit && actions) hit[r] = ((g > 0.f ? 1.f : -1.f) == actions[(long long)r * lda + A]) ? 1.f : 0.f;
  }
}

// ------------------------------------------------------------------------------------------
// Gaussian policy head, networks/actor_critic/actor.py:259-266:
//   mean = clamp(raw_m, -9, 9); std = exp(clamp(raw_ls, -5, 2)).   raw: (rows, 2L) = [mean | log_std]
__global__ void gauss_head_fwd_kernel(int rows, int L, const float* __restrict__ raw, float* __restrict__ mean,
                                      float* __restrict__ stdv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * L) return;
  const int r = i / L, c = i % L;
  mean[i] = fminf(fmaxf(raw[(long long)r * 2 * L + c], -9.f), 9.f);
  stdv[i] = expf(fminf(fmaxf(raw[(long long)r * 2 * L + L + c], -5.f), 2.f));
}
__global__ void gauss_head_bwd_kernel(int rows, int L, const float* __restrict__ raw,
                                      const float* __restrict__ stdv, const float* __restrict__ dmean,
                                      const float* __restrict__ dstd, float* __restrict__ draw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * L) return;
  const int r = i / L, c = i % L;
  const float rm = raw[(long long)r * 2 * L + c], rl = raw[(long long)r * 2 * L + L + c];
  draw[(long long)r * 2 * L + c] = (dmean && rm >= -9.f && rm <= 9.f) ? dmean[i] : 0.f;
  draw[(long long)r * 2 * L + L + c] = (dstd && rl >= -5.f && rl <= 2.f) ? dstd[i] * stdv[i] : 0.f;
}

// Plan-recognition head, plan_recognition_tanh_net.py:44-46: raw (rows, 2L) = [mean | var];
//   std = softplus(var) + min_std
__global__ void softplus_head_fwd_kernel(int rows, int L, const float* __restrict__ raw, float min_std,
                                         float* __restrict__ mean, float* __restrict__ stdv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * L) return;
  const int r = i / L, c = i % L;
  mean[i] = raw[(long long)r * 2 * L + c];
  stdv[i] = softplus_acc(raw[(long long)r * 2 * L + L + c]) + min_std;
}
__global__ void softplus_head_bwd_kernel(int rows, int L, const float* __restrict__ raw,
                                         const float* __restrict__ dmean, const float* __restrict__ dstd,
                                         float* __restrict__ draw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * L) return;
  const int r = i / L, c = i % L;
  const float v = raw[(long long)r * 2 * L + L + c];
  draw[(long long)r * 2 * L + c] = dmean ? dmean[i] : 0.f;
  draw[(long long)r * 2 * L + L + c] = dstd ? dstd[i] * (v > 20.f ? 1.f : sigmoid_acc(v)) : 0.f;
}

// ------------------------------------------------------------------------------------------
// Balanced Gaussian KL, modules/play_lmp/play_lmp_for_rl.py:259-285.  Single CTA.
//   kl = alpha * mean_b KL(sg(q)||p) + (1-alpha) * mean_b KL(q||sg(p));  out[0] = kl.
//   Gradients (already weighted and divided by B): dq from the (1-alpha) term, dp from the alpha term.
__global__ void kl_balanced_kernel(int B, int L, const float* __restrict__ mu_q, const float* __restrict__ sd_q,
                                   const float* __restrict__ mu_p, const float* __restrict__ sd_p,
                                   float w_p, float w_q, float* __restrict__ out, float* __restrict__ dmu_q,
                                   float* __restrict__ dsd_q, float* __restrict__ dmu_p, float* __restrict__ dsd_p) {
  __shared__ float red[32];
  float acc = 0.f;
  const float invB = 1.f / (float)B;
  for (int i = threadIdx.x; i < B * L; i += blockDim.x) {
    const float mq = mu_q[i], sq = sd_q[i], mp = mu_p[i], sp = sd_p[i];
    const float vr = (sq / sp) * (sq / sp);
    const float dm = (mq - mp) / sp;
    acc += 0.5f * (vr + dm * dm - 1.f - logf(vr));
    const float isp2 = 1.f / (sp * sp);
    if (dmu_p) {
      dmu_p[i] = w_p * invB * (mp - mq) * isp2;
      dsd_p[i] = w_p * invB * (1.f / sp - (sq * sq + (mq - mp) * (mq - mp)) * isp2 / sp);
      dmu_q[i] = w_q * invB * (mq - mp) * isp2;
      dsd_q[i] = w_q * invB * (-1.f / sq + sq * isp2);
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < (blockDim.x + 31) / 32; ++i) t += red[i];
    out[0] = t * invB * (w_p + w_q);
  }
}

// ------------------------------------------------------------------------------------------
// TanhNormal, utils/distributions.py:61-153.
// rsample: z = mu + std*eps, a = tanh(z)
__global__ void tanh_rsample_fwd_kernel(long long n, const float* __restrict__ mu, const float* __restrict__ sd,
                                        const float* __restrict__ eps, long long bcast, float* __restrict__ a,
                                        float* __restrict__ z, int apply_tanh) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long j = i % bcast;   // mu/std broadcast over a leading sample dim (sample_n)
  const float zz = mu[j] + sd[j] * eps[i];
  if (z) z[i] = zz;
  a[i] = apply_tanh ? tanhf(zz) : zz;
}
// da, dz (either may be null) -> dmu, dstd
__global__ void tanh_rsample_bwd_kernel(long long n, const float* __restrict__ a, const float* __restrict__ eps,
                                        const float* __restrict__ da, const float* __restrict__ dz,
                                        float* __restrict__ dmu, float* __restrict__ dsd, int apply_tanh) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float g = dz ? dz[i] : 0.f;
  if (da) g += apply_tanh ? da[i] * (1.f - a[i] * a[i]) : da[i];
  dmu[i] = g;
  dsd[i] = g * eps[i];
}

// log_prob with pre-tanh value z (from_value: z = atanh(clamp(value, +-0.999)), misc.py:297-300)
//   logp[r] = sum_d [ -(z-mu)^2/(2 std^2) - log std - 0.5 log 2pi ] - sum_d 2 (log2 - z - softplus(-2z))
// One warp per row; mu/std rows broadcast with period `bcast_rows` (sample_n).
__global__ void tanh_logprob_fwd_kernel(int rows, int L, int bcast_rows, const float* __restrict__ mu,
                                        const float* __restrict__ sd, const float* __restrict__ zin,
                                        int from_value, float* __restrict__ logp, float* __restrict__ gmu,
                                        float* __restrict__ gsd, float* __restrict__ gz) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const int pr = warp % bcast_rows;
  float acc = 0.f;
  for (int c = lane; c < L; c += 32) {
    const long long i = (long long)warp * L + c, j = (long long)pr * L + c;
    float z = zin[i];
    if (from_value) {
      const float v = fminf(fmaxf(z, -0.999f), 0.999f);
      z = 0.5f * logf(fmaxf(1.f + v, 1e-6f) / fmaxf(1.f - v, 1e-6f));
    }
    const float m = mu[j], s = sd[j];
    const float t = (z - m) / s;
    acc += -0.5f * t * t - logf(s) - 0.9189385332046727f
           - 2.f * (0.6931471805599453f - z - softplus_acc(-2.f * z));
    if (gmu) {
      gmu[i] = t / s;
      gsd[i] = (t * t - 1.f) / s;
      gz[i] = -t / s + 2.f * tanhf(z);
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) logp[warp] = acc;
}

// out[i] = x[i] * (*s) * c
__global__ void scale_by_device_scalar_kernel(long long n, const float* __restrict__ x, const float* __restrict__ s,
                                              float c, float* __restrict__ out) {
  const float k = (s ? *s : 1.f) * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    out[i] = x[i] * k;
}

static inline int nb(long long n, int t = 256) { return (int)((n + t - 1) / t); }

}  // namespace tacorl

using namespace tacorl;

extern "C" {

int tacorl_dlm_nll(int rows, int act_dims, const float* logits, long long ld, const float* actions,
                   long long lda, int num_classes, float act_min, float act_max, float gripper_alpha,
                   float* row_loss, float* loss_out, float* dlogits, long long ldd, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TACORL_REQUIRE(logits && actions && row_loss && loss_out, "dlm_nll: null pointer");
  TACORL_REQUIRE(rows > 0 && act_dims > 0, "dlm_nll: empty input");
  TACORL_REQUIRE(num_classes >= 2, "dlm_nll: num_classes must be >= 2 (got %d)", num_classes);
  const float half_bin = (act_max - act_min) / 2.f / (float)(num_classes - 1);
  const float log_half_classes = logf((float)(num_classes - 1) / 2.f);
  dlm_nll_kernel<<<nb((long long)rows * act_dims, 128), 128, 0, st>>>(rows, act_dims, logits, ld, actions, lda,
                                                                     half_bin, log_half_classes, act_min, act_max, gripper_alpha,
                                                                     row_loss, dlogits, ldd);
  TACORL_LAUNCH_CHECK();
  return colsum_f32(rows * (act_dims + 1), 1, row_loss, 1, loss_out, 0, st);
}

int tacorl_dlm_sample(int rows, int act_dims, const float* logits, long long ld, const float* u1,
                      const float* u2, const float* actions, long long lda, float grip_lo, float grip_hi,
                      float* pred, float* hit, float* acc_out, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TACORL_REQUIRE(logits && u1 && u2 && pred, "dlm_sample: null pointer");
  TACORL_REQUIRE(rows > 0, "dlm_sample: empty input");
  dlm_sample_kernel<<<nb((long long)rows * act_dims, 128), 128, 0, st>>>(rows, act_dims, logits, ld, u1, u2,
                                                                        actions, lda, grip_lo, grip_hi, pred, hit);
  TACORL_LAUNCH_CHECK();
  if (hit && acc_out && actions) {
    int rc = colsum_f32(rows, 1, hit, 1, acc_out, 0, st);
    if (rc) return rc;
    scale_by_device_scalar_kernel<<<1, 32, 0, st>>>(1, acc_out, nullptr, 1.f / (float)rows, acc_out);
    TACORL_LAUNCH_CHECK();
  }
  return 0;
}

int tacorl_gauss_head_fwd(int rows, int L, const float* raw, float* mean, float* stdv, void* stream) {
  if (rows * L == 0) return 0;
  gauss_head_fwd_kernel<<<nb((long long)rows * L), 256, 0, (cudaStream_t)stream>>>(rows, L, raw, mean, stdv);
  TACORL_LAUNCH_CHECK();
  return 0;
}
int tacorl_gauss_head_bwd(int rows, int L, const float* raw, const float* stdv, const float* dmean,
                          const float* dstd, float* draw, void* stream) {
  if (rows * L == 0) return 0;
  gauss_head_bwd_kernel<<<nb((long long)rows * L), 256, 0, (cudaStream_t)stream>>>(rows, L, raw, stdv, dmean, dstd, draw);
  TACORL_LAUNCH_CHECK();
  return 0;
}
int tacorl_softplus_head_fwd(int rows, int L, const float* raw, float min_std, float* mean, float* stdv,
                             void* stream) {
  if (rows * L == 0) return 0;
  softplus_head_fwd_kernel<<<nb((long long)rows * L), 256, 0, (cudaStream_t)stream>>>(rows, L, raw, min_std, mean, stdv);
  TACORL_LAUNCH_CHECK();
  return 0;
}
int tacorl_softplus_head_bwd(int rows, int L, const float* raw, const float* dmean, const float* dstd,
                             float* draw, void* stream) {
  if (rows * L == 0) return 0;
  softplus_head_bwd_kernel<<<nb((long long)rows * L), 256, 0, (cudaStream_t)stream>>>(rows, L, raw, dmean, dstd, draw);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_kl_balanced(int B, int L, const float* mu_q, const float* sd_q, const float* mu_p,
                       const float* sd_p, float kl_alpha, int balancing, float* kl_out, float* dmu_q,
                       float* dsd_q, float* dmu_p, float* dsd_p, void* stream) {
  TACORL_REQUIRE(B > 0 && L > 0, "kl_balanced: empty input");
  // value = w_p*KL + w_q*KL with (w_p, w_q) = (alpha, 1-alpha); without balancing both paths carry the
  // full gradient of a single KL term: value weight 1, gradient weights (1, 1).
  float w_p = balancing ? kl_alpha : 1.f, w_q = balancing ? 1.f - kl_alpha : 1.f;
  kl_balanced_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(B, L, mu_q, sd_q, mu_p, sd_p, w_p, w_q, kl_out, dmu_q,
                                                         dsd_q, dmu_p, dsd_p);
  TACORL_LAUNCH_CHECK();
  if (!balancing) {  // undo the (w_p + w_q) = 2 factor on the value
    scale_by_device_scalar_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(1, kl_out, nullptr, 0.5f, kl_out);
    TACORL_LAUNCH_CHECK();
  }
  return 0;
}

int tacorl_tanh_rsample_fwd(long long n, long long bcast, const float* mu, const float* sd, const float* eps,
                            float* a, float* z, int apply_tanh, void* stream) {
  if (n == 0) return 0;
  TACORL_REQUIRE(bcast > 0 && n % bcast == 0, "tanh_rsample_fwd: bad broadcast period");
  tanh_rsample_fwd_kernel<<<nb(n), 256, 0, (cudaStream_t)stream>>>(n, mu, sd, eps, bcast, a, z, apply_tanh);
  TACORL_LAUNCH_CHECK();
  return 0;
}
int tacorl_tanh_rsample_bwd(long long n, const float* a, const float* eps, const float* da, const float* dz,
                            float* dmu, float* dsd, int apply_tanh, void* stream) {
  if (n == 0) return 0;
  tanh_rsample_bwd_kernel<<<nb(n), 256, 0, (cudaStream_t)stream>>>(n, a, eps, da, dz, dmu, dsd, apply_tanh);
  TACORL_LAUNCH_CHECK();
  return 0;
}
int tacorl_tanh_logprob(int rows, int L, int bcast_rows, const float* mu, const float* sd, const float* z,
                        int from_value, float* logp, float* gmu, float* gsd, float* gz, void* stream) {
  if (rows == 0) return 0;
  TACORL_REQUIRE(bcast_rows > 0 && rows % bcast_rows == 0, "tanh_logprob: bad broadcast period");
  tanh_logprob_fwd_kernel<<<nb((long long)rows * 32, 128), 128, 0, (cudaStream_t)stream>>>(
      rows, L, bcast_rows, mu, sd, z, from_value, logp, gmu, gsd, gz);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_scale(long long n, const float* x, const float* dev_scalar, float c, float* out, void* stream) {
  if (n == 0) return 0;
  scale_by_device_scalar_kernel<<<(int)min((long long)1184, (n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      n, x, dev_scalar, c, out);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

// out[r][c] = x[r][c] * s[r] * k   (chain rule through per-row scalars such as log-probs)
namespace tacorl {
__global__ void rowscale_kernel(long long rows, int L, const float* __restrict__ x, const float* __restrict__ s,
                                float k, float* __restrict__ out, int accumulate) {
  const long long total = rows * L;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i] * s[i / L] * k;
    out[i] = accumulate ? out[i] + v : v;
  }
}
}  // namespace tacorl

extern "C" int tacorl_rowscale(long long rows, int L, const float* x, const float* row_scalars, float k,
                               float* out, int accumulate, void* stream) {
  if (rows * L == 0) return 0;
  tacorl::rowscale_kernel<<<(int)min((long long)1184, (rows * L + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      rows, L, x, row_scalars, k, out, accumulate);
  TACORL_LAUNCH_CHECK();
  return 0;
}
