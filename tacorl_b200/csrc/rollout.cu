// One control step of the action decoder for a batch of independent environments (tacorl_b200/rollout.py,
// DESIGN.md section 16): the two ReLU-RNN layers, the four heads and the discretised-logistic-mixture sample, in three
// graph-capturable launches of one kernel:
//   layer 0   hn0 = relu([plan | emb] W_ih0^T + h0 W_hh0^T + b_ih0 + b_hh0)      (h0 = 0 on a restarting row)
//   layer 1   hn1 = relu(hn0 W_ih1^T + h1 W_hh1^T + b_ih1 + b_hh1)                 (+ copies hn0 into hidden[0])
//   heads     logits = hn1 [W_prob; W_mean; W_log_scale; W_gripper]^T + b          (+ copies hn1 into hidden[1]); the
//             last CTA to finish draws the Philox uniforms, samples every row and advances the step counters.
// Each launch is a small-batch "decode" GEMV: a CTA owns kWarps output columns for ALL rows, so every weight is read
// once per step whatever the batch; the rows' inputs are staged through shared memory in 256-wide K chunks.  A warp owns
// one column; lane l accumulates k = chunk + 128 h + 4 l + q (h < 2, q < 4) in that order, chunk after chunk, and the
// 32 lane partials are summed by a fixed shuffle-down tree.  Nothing in that order depends on the number of rows or on
// any other row, so a row's result is bit-identical alone or in a batch of 64.
// tacorl_rollout_policy_sample draws the policy's own samples (a sampled latent plan, the flat-CQL actor's TanhNormal
// arm and GumbelSoftmax gripper) from the same counter-based stream, in one launch.
#include "common.cuh"
#include "internal.h"
#include "philox.cuh"
#include "dlm_sample.cuh"
#include "gripper.cuh"
#include "../../include/tacorl_b200.h"
#include <cuda_bf16.h>

namespace tacorl {

constexpr int kWarps = 16;           // output columns per CTA
constexpr int kChunk = 256;          // K chunk staged per pass
constexpr int kMaxRows = 64;
constexpr int kActDims = 6;          // continuous action dimensions (the seventh is the gripper)
constexpr int kHeadCols = 3 * kActDims * kMix + 2;

struct Seg {                          // one input segment: rows of A (n x K) against a K-slice of the weights
  const float* A = nullptr; long long lda = 0; int K = 0;
  int masked = 0;                     // restarting rows read zeros (h = 0)
};
struct Group {                        // a run of output columns sharing weight / bias tensors
  int cols = 0;
  const float* W[3] = {nullptr, nullptr, nullptr};
  const __nv_bfloat16* Wb[3] = {nullptr, nullptr, nullptr};   // bf16 operand copies (same layout) or null
  long long ldw[3] = {0, 0, 0};
  const float* b0 = nullptr; const float* b1 = nullptr;
};
struct GemvArgs {
  int n = 0, N = 0, n_seg = 0, n_grp = 0, relu = 0;
  Seg seg[3];
  Group grp[4];
  const int* restart = nullptr;
  float* out = nullptr; long long ldo = 0;
  // a copy of `n x cols` floats (src -> dst, rows of ld) done on the side by every CTA
  const float* copy_src = nullptr; float* copy_dst = nullptr; int copy_cols = 0;
  // heads only: the last CTA samples
  unsigned* done = nullptr;
  float* actions = nullptr;
  const int* env_id = nullptr; long long* t = nullptr;
  unsigned k0 = 0, k1 = 0;
  float grip_lo = -1.f, grip_hi = 1.f;
};

__device__ __forceinline__ float rne(float v) { return __bfloat162float(__float2bfloat16(v)); }

// uniform i of a row: word i mod 4 of draw i div 4 with counter (lo32(t), hi32(t), env_id, draw), as (w >> 8) 2^-24
__device__ __forceinline__ float rollout_uniform(unsigned long long t, unsigned env, int i, unsigned k0, unsigned k1) {
  const U4 r = philox4x32_10(U4{(unsigned)t, (unsigned)(t >> 32), env, (unsigned)(i >> 2)}, k0, k1);
  const unsigned w = (i & 3) == 0 ? r.x : (i & 3) == 1 ? r.y : (i & 3) == 2 ? r.z : r.w;
  return __fmul_rn((float)(w >> 8), 5.9604644775390625e-08f);
}

template <int NR, bool BF>
__global__ void __launch_bounds__(kWarps * 32) rollout_gemv_kernel(const GemvArgs a) {
  extern __shared__ float4 smem4[];
  float (*sx)[kChunk] = reinterpret_cast<float (*)[kChunk]>(smem4);   // [NR][kChunk]
  __shared__ unsigned s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = blockIdx.x * kWarps + warp;
  const int n = a.n;
  // side copy (grid-stride; nothing in this launch reads the destination)
  if (a.copy_dst) {
    const long long total = (long long)n * a.copy_cols;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
      a.copy_dst[i] = a.copy_src[i];
  }
  // the column's weight group
  int g = 0, jl = j;
  while (g < a.n_grp - 1 && jl >= a.grp[g].cols) { jl -= a.grp[g].cols; ++g; }
  const Group& G = a.grp[g];
  const float bias = j < a.N ? G.b0[jl] + (G.b1 ? G.b1[jl] : 0.f) : 0.f;
  float acc[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) acc[r] = 0.f;
  for (int s = 0; s < a.n_seg; ++s) {
    const Seg S = a.seg[s];
    const float* Wf = G.W[s] + (long long)jl * G.ldw[s];
    const __nv_bfloat16* Wb = G.Wb[s] ? G.Wb[s] + (long long)jl * G.ldw[s] : nullptr;
    for (int kc = 0; kc < S.K; kc += kChunk) {
      __syncthreads();
      for (int i = threadIdx.x; i < n * (kChunk / 4); i += blockDim.x) {
        const int r = i / (kChunk / 4), k = kc + 4 * (i % (kChunk / 4));
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < S.K && !(S.masked && a.restart[r])) v = *(const float4*)(S.A + r * S.lda + k);
        if (BF) { v.x = rne(v.x); v.y = rne(v.y); v.z = rne(v.z); v.w = rne(v.w); }
        *(float4*)&sx[r][k - kc] = v;
      }
      __syncthreads();
      if (j >= a.N) continue;
      float w[8];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = kc + 128 * h + 4 * lane;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < S.K) {
          if (Wb) {
            const uint2 raw = *(const uint2*)(Wb + k);
            const __nv_bfloat162 lo = *(const __nv_bfloat162*)&raw.x, hi = *(const __nv_bfloat162*)&raw.y;
            v = make_float4(__low2float(lo), __high2float(lo), __low2float(hi), __high2float(hi));
          } else {
            v = *(const float4*)(Wf + k);
            if (BF) { v.x = rne(v.x); v.y = rne(v.y); v.z = rne(v.z); v.w = rne(v.w); }
          }
        }
        w[4 * h] = v.x; w[4 * h + 1] = v.y; w[4 * h + 2] = v.z; w[4 * h + 3] = v.w;
      }
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        if (r < n) {
          const float4 x0 = *(const float4*)&sx[r][4 * lane], x1 = *(const float4*)&sx[r][128 + 4 * lane];
          float c = acc[r];
          c = fmaf(x0.x, w[0], c); c = fmaf(x0.y, w[1], c); c = fmaf(x0.z, w[2], c); c = fmaf(x0.w, w[3], c);
          c = fmaf(x1.x, w[4], c); c = fmaf(x1.y, w[5], c); c = fmaf(x1.z, w[6], c); c = fmaf(x1.w, w[7], c);
          acc[r] = c;
        }
      }
    }
  }
  if (j < a.N) {
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      if (r < n) {
        float v = acc[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) {
          v += bias;
          a.out[r * a.ldo + j] = a.relu ? fmaxf(v, 0.f) : v;
        }
      }
    }
  }
  if (!a.done) return;
  // heads: the last CTA to finish reads every row's logits and samples
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(a.done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int i = threadIdx.x; i < n * kActDims; i += blockDim.x) {
    const int r = i / kActDims, d = i % kActDims;
    const float* L = a.out + r * a.ldo;
    // dimension d's [prob 10 | mean 10 | log_scale 10] and the gripper pair, laid out as a one-dimension logits row
    // (read through L2: other CTAs wrote them)
    float lg[3 * kMix + 2];
    for (int k = 0; k < kMix; ++k) {
      lg[k] = __ldcg(L + d * kMix + k);
      lg[kMix + k] = __ldcg(L + kActDims * kMix + d * kMix + k);
      lg[2 * kMix + k] = __ldcg(L + 2 * kActDims * kMix + d * kMix + k);
    }
    lg[3 * kMix] = __ldcg(L + 3 * kActDims * kMix);
    lg[3 * kMix + 1] = __ldcg(L + 3 * kActDims * kMix + 1);
    const unsigned long long t = (unsigned long long)a.t[r];
    const unsigned env = (unsigned)a.env_id[r];
    const float u2 = rollout_uniform(t, env, kActDims * kMix + d, a.k0, a.k1);
    a.actions[r * (kActDims + 1) + d] =
        dlm_sample_dim(lg, 1, 0, [&](int k) { return rollout_uniform(t, env, d * kMix + k, a.k0, a.k1); }, u2);
    if (d == 0) a.actions[r * (kActDims + 1) + kActDims] = dlm_gripper(lg, 1, a.grip_lo, a.grip_hi);
  }
  __syncthreads();
  for (int r = threadIdx.x; r < n; r += blockDim.x) a.t[r] += 1;
  if (threadIdx.x == 0) *a.done = 0u;       // ready for the next step (and the next graph replay)
}

template <int NR, bool BF>
static int launch_gemv_nr(const GemvArgs& a, cudaStream_t st) {
  constexpr int smem = NR * kChunk * 4;
  // set on every call: the attribute is per device (a function attribute, not a stream operation: allowed while capturing)
  TACORL_CHECK_CUDA(cudaFuncSetAttribute(rollout_gemv_kernel<NR, BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  rollout_gemv_kernel<NR, BF><<<cdiv(a.N, kWarps), kWarps * 32, smem, st>>>(a);
  TACORL_LAUNCH_CHECK();
  return 0;
}

static int launch_gemv(const GemvArgs& a, int prec, cudaStream_t st) {
  const bool bf = prec == PREC_BF16;
  if (a.n <= 8) return bf ? launch_gemv_nr<8, true>(a, st) : launch_gemv_nr<8, false>(a, st);
  return bf ? launch_gemv_nr<kMaxRows, true>(a, st) : launch_gemv_nr<kMaxRows, false>(a, st);
}

// The policy's own draws (sampled plans, the flat-CQL actor) start at draw 32: the decoder step above uses draws 0..16
// of the same counter, so both can sample in one step with the same t and still read disjoint noise.
constexpr int kPolicyDraw0 = 32;

// Row r, continuous dimension d < A: words 0 / 1 of draw 32 + d are u_a / u_b, z = sqrt(-2 ln(1 - u_a)) cos(2 pi u_b)
// and out = tanh(mean + std z) (TanhNormal.sample()).  Gripper (logits given): words 0 / 1 of draw 32 + A are u_0 / u_1
// and out[A] = 2 argmax_c(normalised logit_c - log(-log(u_c))) - 1 (GumbelSoftmax.sample(), as gripper_gumbel_kernel
// computes it unclamped: u = 0 scores -inf, ties go to class 0).  One CTA, so that the step counters are advanced
// after every element has read them; each element is computed on its own, so a row's output does not depend on n.
__global__ void __launch_bounds__(256) rollout_policy_sample_kernel(
    int n, int A, const float* __restrict__ mean, const float* __restrict__ stdv, const float* __restrict__ grip,
    const int* __restrict__ mask, unsigned k0, unsigned k1, const int* __restrict__ env_id, long long* t, int advance_t,
    float* __restrict__ out, long long ldo) {
  const int per_row = A + (grip ? 1 : 0);
  for (int i = threadIdx.x; i < n * per_row; i += blockDim.x) {
    const int r = i / per_row, d = i % per_row;
    if (mask && mask[r] == 0) continue;
    const unsigned long long tt = (unsigned long long)t[r];
    const U4 w = philox4x32_10(U4{(unsigned)tt, (unsigned)(tt >> 32), (unsigned)env_id[r], (unsigned)(kPolicyDraw0 + d)},
                               k0, k1);
    const float ua = __fmul_rn((float)(w.x >> 8), 5.9604644775390625e-08f);
    const float ub = __fmul_rn((float)(w.y >> 8), 5.9604644775390625e-08f);
    if (d < A) {
      const float z = sqrtf(-2.f * logf(1.f - ua)) * cosf(6.28318530717958647692f * ub);
      out[r * ldo + d] = tanhf(fmaf(stdv[r * A + d], z, mean[r * A + d]));
    } else {
      float n0, n1;
      gr_normalise(grip[2 * r], grip[2 * r + 1], n0, n1);
      const float s0 = n0 - logf(-logf(ua)), s1 = n1 - logf(-logf(ub));
      out[r * ldo + A] = s1 > s0 ? 1.f : -1.f;
    }
  }
  if (!advance_t) return;
  __syncthreads();
  for (int r = threadIdx.x; r < n; r += blockDim.x) t[r] += 1;
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }
static bool aligned8(const void* p) { return ((uintptr_t)p & 7) == 0; }

}  // namespace tacorl

using namespace tacorl;

extern "C" {

size_t tacorl_rollout_ws_bytes(int n, int H) {
  return ((size_t)2 * n * H + (size_t)n * kHeadCols) * 4 + 256;
}

int tacorl_rollout_decoder_step(int n, int P, int E, int H, const float* plan, const float* emb, float* hidden,
                                const int* restart, const float* const* w, const void* const* w_bf16,
                                unsigned long long seed, const int* env_id, long long* t, float grip_lo, float grip_hi,
                                float* actions, float* logits, void* ws, size_t ws_bytes, int prec, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TACORL_REQUIRE(prec == PREC_F32 || prec == PREC_BF16, "rollout_decoder_step: unknown precision %d", prec);
  TACORL_REQUIRE(n >= 1 && n <= kMaxRows, "rollout_decoder_step: n = %d environments (1..%d)", n, kMaxRows);
  TACORL_REQUIRE(P > 0 && E > 0 && P % 4 == 0 && E % 4 == 0 && H > 0 && H % 8 == 0,
                 "rollout_decoder_step: plan %d / embedding %d must be multiples of 4, hidden %d of 8", P, E, H);
  TACORL_REQUIRE(plan && emb && hidden && restart && w && env_id && t && actions && ws, "rollout_decoder_step: null pointer");
  for (int i = 0; i < 16; ++i) TACORL_REQUIRE(w[i] && aligned16(w[i]), "rollout_decoder_step: weight %d null or not 16-byte aligned", i);
  TACORL_REQUIRE(aligned16(plan) && aligned16(emb) && aligned16(hidden) && aligned16(ws) && (!logits || aligned16(logits)),
                 "rollout_decoder_step: activations must be 16-byte aligned");
  TACORL_REQUIRE(ws_bytes >= tacorl_rollout_ws_bytes(n, H), "rollout_decoder_step: workspace too small");
  // bf16 operand copies, used by PREC_BF16 only: W_ih0, W_hh0, W_ih1, W_hh1, prob, mean, log_scale, gripper
  const __nv_bfloat16* wb[8] = {};
  if (prec == PREC_BF16 && w_bf16)
    for (int i = 0; i < 8; ++i) {
      wb[i] = (const __nv_bfloat16*)w_bf16[i];
      TACORL_REQUIRE(!wb[i] || aligned8(wb[i]), "rollout_decoder_step: bf16 weight %d not 8-byte aligned", i);
    }
  const int I = P + E;
  float* hn = (float*)ws;                               // (2, n, H) new hidden states
  float* lg_ws = hn + (size_t)2 * n * H;                // (n, 182) logits when the caller keeps none
  unsigned* done = (unsigned*)(((uintptr_t)(lg_ws + (size_t)n * kHeadCols) + 127) & ~(uintptr_t)127);
  int rc;
  GemvArgs a;
  a.n = n; a.restart = restart;
  // layer 0
  a.N = H; a.relu = 1; a.n_seg = 3; a.n_grp = 1;
  a.seg[0] = Seg{plan, P, P, 0}; a.seg[1] = Seg{emb, E, E, 0}; a.seg[2] = Seg{hidden, H, H, 1};
  Group& g0 = a.grp[0];
  g0.cols = H; g0.b0 = w[2]; g0.b1 = w[3];
  g0.W[0] = w[0]; g0.W[1] = w[0] + P; g0.W[2] = w[1];
  g0.Wb[0] = wb[0]; g0.Wb[1] = wb[0] ? wb[0] + P : nullptr; g0.Wb[2] = wb[1];
  g0.ldw[0] = I; g0.ldw[1] = I; g0.ldw[2] = H;
  a.out = hn; a.ldo = H;
  if ((rc = launch_gemv(a, prec, st))) return rc;
  // layer 1 (hidden[0] is no longer read: it takes hn0)
  a.n_seg = 2;
  a.seg[0] = Seg{hn, H, H, 0}; a.seg[1] = Seg{hidden + (size_t)n * H, H, H, 1};
  g0.b0 = w[6]; g0.b1 = w[7];
  g0.W[0] = w[4]; g0.W[1] = w[5]; g0.W[2] = nullptr;
  g0.Wb[0] = wb[2]; g0.Wb[1] = wb[3]; g0.Wb[2] = nullptr;
  g0.ldw[0] = H; g0.ldw[1] = H;
  a.out = hn + (size_t)n * H;
  a.copy_src = hn; a.copy_dst = hidden; a.copy_cols = H;
  if ((rc = launch_gemv(a, prec, st))) return rc;
  // heads + sample (hidden[1] is no longer read: it takes hn1)
  a.N = kHeadCols; a.relu = 0; a.n_seg = 1; a.n_grp = 4;
  a.seg[0] = Seg{hn + (size_t)n * H, H, H, 0};
  for (int h = 0; h < 4; ++h) {
    Group& g = a.grp[h];
    g = Group{};
    g.cols = h < 3 ? kActDims * kMix : 2;
    g.W[0] = w[8 + 2 * h]; g.b0 = w[9 + 2 * h]; g.Wb[0] = wb[4 + h]; g.ldw[0] = H;
  }
  a.out = logits ? logits : lg_ws; a.ldo = kHeadCols;
  a.copy_src = hn + (size_t)n * H; a.copy_dst = hidden + (size_t)n * H;
  a.done = done; a.actions = actions; a.env_id = env_id; a.t = t;
  a.k0 = (unsigned)seed; a.k1 = (unsigned)(seed >> 32);
  a.grip_lo = grip_lo; a.grip_hi = grip_hi;
  return launch_gemv(a, prec, st);
}

int tacorl_rollout_policy_sample(int n, int A, const float* mean, const float* std, const float* grip_logits,
                                 const int* mask, unsigned long long seed, const int* env_id, long long* t, int advance_t,
                                 float* out, long long ldo, void* stream) {
  TACORL_REQUIRE(n >= 1 && n <= kMaxRows, "rollout_policy_sample: n = %d rows (1..%d)", n, kMaxRows);
  TACORL_REQUIRE(A >= 1, "rollout_policy_sample: A = %d continuous dimensions", A);
  TACORL_REQUIRE(ldo >= A + (grip_logits ? 1 : 0), "rollout_policy_sample: output row stride %lld < %d", ldo,
                 A + (grip_logits ? 1 : 0));
  TACORL_REQUIRE(mean && std && env_id && t && out, "rollout_policy_sample: null pointer");
  rollout_policy_sample_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(n, A, mean, std, grip_logits, mask, (unsigned)seed,
                                                                    (unsigned)(seed >> 32), env_id, t, advance_t, out, ldo);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
