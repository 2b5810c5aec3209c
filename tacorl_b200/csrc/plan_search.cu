// Critic-guided plan search of the rollout policy (tacorl_b200/rollout.py PlanSearch, DESIGN.md section 16.2): a
// cross-entropy-method search over the pre-tanh latent plan z of each replanning environment, every candidate scored by
// min(Q1, Q2) of TACO-RL's twin critics.  One iteration is
//   tacorl_plan_search_sample_l0   candidates z = mu + sigma eps (Philox draws 256 + (k K + c) P + d of the row's
//                                  counter) and layer 0 of both critics, h0 = silu(u[env] + W0[:, D:] tanh z), where
//                                  u = W0[:, :D] e + b0 is computed once per environment and broadcast to its K candidates
//   tacorl_plan_search_hidden      hidden layers 1..L-1 of both critics: bias + SiLU GEMMs (tcgen05 in bf16 mode, FFMA
//                                  in fp32 mode) with split-K pinned to 1
//   tacorl_plan_search_select      the output layer of both critics, s = min(Q1, Q2), the E elites, the refit of
//                                  (mu, sigma) and the best candidate so far; after the last iteration it writes the plan
// Every output element is summed in an order fixed by its own row: a row's candidates, scores and plan are
// bit-identical alone or among 64 rows, at any position.
#include "common.cuh"
#include "internal.h"
#include "philox.cuh"
#include "../../include/tacorl_b200.h"
#include <cuda_bf16.h>

namespace tacorl {

constexpr int kPsDraw0 = 256;         // first Philox draw of the search (decoder: 0..16, policy sampler: 32..)
constexpr int kPsTile = 32;           // candidates per sample_l0 CTA
constexpr int kPsThreads = 256;
constexpr int kPsMaxP = 64;
constexpr int kPsMaxK = 512;

__device__ __forceinline__ float ps_silu(float v) { return v / (1.f + __expf(-v)); }

// grid (K / 32, n): CTA (tile, i) draws candidates 32 tile .. 32 tile + 31 of environment i and runs layer 0 of both
// critics on them.  u_j = W0_j[:, :D] e_j + b0_j is summed by one thread per output column in ascending d (the
// observation part, then the goal part), and the action part is added to it in ascending p.
__global__ void __launch_bounds__(kPsThreads) plan_search_sample_l0_kernel(
    int K, int P, int Do, int Dg, int H, int k, const float* __restrict__ mu, const float* __restrict__ sigma,
    const float* __restrict__ eo1, const float* __restrict__ eg1, const float* __restrict__ W1, const float* __restrict__ b1,
    const float* __restrict__ eo2, const float* __restrict__ eg2, const float* __restrict__ W2, const float* __restrict__ b2,
    unsigned k0, unsigned k1, const int* __restrict__ env_id, const long long* __restrict__ t, float* __restrict__ z,
    float* __restrict__ u_out, float* __restrict__ h1, __nv_bfloat16* __restrict__ h1b, float* __restrict__ h2,
    __nv_bfloat16* __restrict__ h2b) {
  extern __shared__ float ps_smem[];
  float* su = ps_smem;                        // [H] u of the current critic
  float* sa = su + H;                         // [32][P] tanh z
  const int i = blockIdx.y, c0 = blockIdx.x * kPsTile;
  const int D = Do + Dg, ldw = D + P;
  const unsigned long long tt = (unsigned long long)t[i];
  const unsigned env = (unsigned)env_id[i];
  for (int e = threadIdx.x; e < kPsTile * P; e += blockDim.x) {
    const int cl = e / P, d = e % P, c = c0 + cl;
    const float m = mu[(long long)i * P + d];
    float zz = m;
    const unsigned draw = (unsigned)(kPsDraw0 + ((long long)k * K + c) * P + d);
    const U4 w = philox4x32_10(U4{(unsigned)tt, (unsigned)(tt >> 32), env, draw}, k0, k1);
    const float ua = __fmul_rn((float)(w.x >> 8), 5.9604644775390625e-08f);
    const float ub = __fmul_rn((float)(w.y >> 8), 5.9604644775390625e-08f);
    if (!(k == 0 && c == 0)) {                // candidate (0, 0) is the actor's deterministic plan
      const float eps = sqrtf(-2.f * logf(1.f - ua)) * cosf(6.28318530717958647692f * ub);
      zz = fmaf(sigma[(long long)i * P + d], eps, m);
    }
    const long long row = (long long)i * K + c;
    z[row * P + d] = zz;
    if (u_out) { u_out[(row * P + d) * 2] = ua; u_out[(row * P + d) * 2 + 1] = ub; }
    sa[cl * P + d] = tanhf(zz);
  }
  for (int j = 0; j < 2; ++j) {
    const float* eo = j ? eo2 : eo1;
    const float* eg = j ? eg2 : eg1;
    const float* W = j ? W2 : W1;
    const float* b = j ? b2 : b1;
    float* h = j ? h2 : h1;
    __nv_bfloat16* hb = j ? h2b : h1b;
    __syncthreads();                          // sa written / su of the previous critic read
    for (int col = threadIdx.x; col < H; col += blockDim.x) {
      const float* wr = W + (long long)col * ldw;
      float acc = b[col];
      for (int d = 0; d < Do; ++d) acc = fmaf(wr[d], eo[(long long)i * Do + d], acc);
      for (int d = 0; d < Dg; ++d) acc = fmaf(wr[Do + d], eg[(long long)i * Dg + d], acc);
      su[col] = acc;
    }
    __syncthreads();
    for (int col = threadIdx.x; col < H; col += blockDim.x) {
      const float* wa = W + (long long)col * ldw + D;
      float acc[kPsTile];
      const float u = su[col];
#pragma unroll
      for (int cl = 0; cl < kPsTile; ++cl) acc[cl] = u;
      for (int p = 0; p < P; ++p) {
        const float w = wa[p];
#pragma unroll
        for (int cl = 0; cl < kPsTile; ++cl) acc[cl] = fmaf(w, sa[cl * P + p], acc[cl]);
      }
#pragma unroll
      for (int cl = 0; cl < kPsTile; ++cl) {
        const long long o = ((long long)i * K + c0 + cl) * H + col;
        const float v = ps_silu(acc[cl]);
        h[o] = v;
        if (hb) hb[o] = __float2bfloat16(v);
      }
    }
  }
}

// One CTA per environment.  Scores: warp w takes candidates w, w + 8, ...; lane l sums h = l, l + 32, ... in ascending
// order and a fixed shuffle-down tree adds the 32 partials.  Elites: a candidate's rank is the number of candidates with
// a higher score or an equal score and a lower index; ranks below E are elites.  Refit: one thread per dimension sums
// the elites in ascending c, mean first, then the squared deviations (population std), all in plain fp32 adds and
// multiplies (no contraction), so an fp32 restatement reproduces them bit for bit.
__global__ void __launch_bounds__(kPsThreads) plan_search_select_kernel(
    int K, int P, int H, int E, int k, int last, float min_std, const float* __restrict__ z,
    const float* __restrict__ h1, const float* __restrict__ w1, const float* __restrict__ b1,
    const float* __restrict__ h2, const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ scores,
    float* __restrict__ mu, float* __restrict__ sigma, float* __restrict__ best_z, float* __restrict__ best_s,
    const int* __restrict__ restart, float* __restrict__ plan, float* __restrict__ plan_value) {
  __shared__ float ss[kPsMaxK];
  __shared__ unsigned char elite[kPsMaxK];
  __shared__ int s_top;
  const int i = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int c = warp; c < K; c += nw) {
    const long long row = (long long)i * K + c;
    float q[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float* h = (j ? h2 : h1) + row * H;
      const float* w = j ? w2 : w1;
      float acc = 0.f;
      for (int x = lane; x < H; x += 32) acc = fmaf(w[x], h[x], acc);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
      q[j] = acc + (j ? b2[0] : b1[0]);
    }
    if (lane == 0) {
      const float s = (isnan(q[0]) || isnan(q[1])) ? -INFINITY : fminf(q[0], q[1]);
      ss[c] = s;
      scores[row] = s;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    const float s = ss[c];
    int rank = 0;
    for (int x = 0; x < K; ++x) {
      const float o = ss[x];
      rank += (o > s) || (o == s && x < c);
    }
    elite[c] = rank < E;
    if (rank == 0) s_top = c;
  }
  __syncthreads();
  const int top = s_top;
  const float top_s = ss[top];
  // best so far: strictly better than every earlier iteration's best (ties keep the earliest (k, c))
  const bool better = k == 0 || top_s > best_s[i];
  for (int d = threadIdx.x; d < P; d += blockDim.x) {
    const float* zi = z + (long long)i * K * P + d;
    float sum = 0.f;
    for (int c = 0; c < K; ++c)
      if (elite[c]) sum = __fadd_rn(sum, zi[(long long)c * P]);
    const float m = __fdiv_rn(sum, (float)E);
    float sq = 0.f;
    for (int c = 0; c < K; ++c)
      if (elite[c]) {
        const float dv = __fsub_rn(zi[(long long)c * P], m);
        sq = __fadd_rn(sq, __fmul_rn(dv, dv));
      }
    const float sd = __fsqrt_rn(__fdiv_rn(sq, (float)E));
    mu[(long long)i * P + d] = m;
    sigma[(long long)i * P + d] = fmaxf(sd, min_std);
    if (better) best_z[(long long)i * P + d] = zi[(long long)top * P];
  }
  __syncthreads();                             // every thread has read best_s[i]
  if (threadIdx.x == 0 && better) best_s[i] = top_s;
  if (!last || (restart && restart[i] == 0)) return;
  __syncthreads();
  for (int d = threadIdx.x; d < P; d += blockDim.x) plan[(long long)i * P + d] = tanhf(best_z[(long long)i * P + d]);
  if (threadIdx.x == 0) plan_value[i] = best_s[i];
}

struct PsLayout {
  float* h[2][2];                   // [critic][slot] fp32 (rows, H)
  __nv_bfloat16* hb[2][2];          // bf16 twins
  __nv_bfloat16* wcast;             // (H, H) bf16 staging of a weight without a caller copy
  size_t bytes;
};

static PsLayout ps_layout(void* ws, int n, int K, int H) {
  PsLayout l;
  Arena a(ws, ~size_t(0) >> 1);
  const size_t rows = (size_t)n * K;
  for (int j = 0; j < 2; ++j)
    for (int s = 0; s < 2; ++s) l.h[j][s] = a.take<float>(rows * H);
  for (int j = 0; j < 2; ++j)
    for (int s = 0; s < 2; ++s) l.hb[j][s] = a.take<__nv_bfloat16>(rows * H);
  l.wcast = a.take<__nv_bfloat16>((size_t)H * H);
  l.bytes = a.off;
  return l;
}

static bool ps_aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

static int ps_check(int n, int K, int P, int H, const char* who) {
  TACORL_REQUIRE(n >= 1 && n <= 64, "%s: n = %d environments (1..64)", who, n);
  TACORL_REQUIRE(K >= 32 && K <= kPsMaxK && K % 32 == 0, "%s: K = %d samples (a multiple of 32 in 32..%d)", who, K,
                 kPsMaxK);
  TACORL_REQUIRE(P >= 1 && P <= kPsMaxP, "%s: plan dimension %d (1..%d)", who, P, kPsMaxP);
  TACORL_REQUIRE(H >= 32 && H <= 1024 && H % 32 == 0, "%s: critic hidden width %d (a multiple of 32 in 32..1024)", who,
                 H);
  return 0;
}

}  // namespace tacorl

using namespace tacorl;

extern "C" {

size_t tacorl_plan_search_ws_bytes(int n, int K, int P, int H) {
  (void)P;
  return ps_layout(nullptr, n, K, H).bytes + 256;
}

int tacorl_plan_search_sample_l0(int n, int K, int P, int Do, int Dg, int H, int k, const float* mu, const float* sigma,
                                 const float* eo1, const float* eg1, const float* W0_1, const float* b0_1,
                                 const float* eo2, const float* eg2, const float* W0_2, const float* b0_2,
                                 unsigned long long seed, const int* env_id, const long long* t, float* z,
                                 float* u_out, void* ws, size_t ws_bytes, int prec, void* stream) {
  int rc;
  if ((rc = ps_check(n, K, P, H, "plan_search_sample_l0"))) return rc;
  TACORL_REQUIRE(prec == PREC_F32 || prec == PREC_BF16, "plan_search_sample_l0: unknown precision %d", prec);
  TACORL_REQUIRE(Do >= 1 && Dg >= 0 && k >= 0, "plan_search_sample_l0: widths %d / %d, iteration %d", Do, Dg, k);
  TACORL_REQUIRE(mu && sigma && eo1 && eo2 && (Dg == 0 || (eg1 && eg2)) && W0_1 && b0_1 && W0_2 && b0_2 && env_id && t &&
                 z && ws, "plan_search_sample_l0: null pointer");
  TACORL_REQUIRE(ws_bytes >= tacorl_plan_search_ws_bytes(n, K, P, H) && ps_aligned16(ws),
                 "plan_search_sample_l0: workspace too small or not 16-byte aligned");
  const PsLayout l = ps_layout(ws, n, K, H);
  const bool bf = prec == PREC_BF16;
  const size_t smem = ((size_t)H + (size_t)kPsTile * P) * sizeof(float);
  plan_search_sample_l0_kernel<<<dim3(K / kPsTile, n), kPsThreads, smem, (cudaStream_t)stream>>>(
      K, P, Do, Dg, H, k, mu, sigma, eo1, eg1, W0_1, b0_1, eo2, eg2, W0_2, b0_2, (unsigned)seed, (unsigned)(seed >> 32),
      env_id, t, z, u_out, l.h[0][0], bf ? l.hb[0][0] : nullptr, l.h[1][0], bf ? l.hb[1][0] : nullptr);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_plan_search_hidden(int n, int K, int H, int layer, const float* W1, const void* W1_bf16, const float* b1,
                              const float* W2, const void* W2_bf16, const float* b2, void* ws, size_t ws_bytes, int prec,
                              void* stream) {
  int rc;
  if ((rc = ps_check(n, K, 1, H, "plan_search_hidden"))) return rc;
  TACORL_REQUIRE(prec == PREC_F32 || prec == PREC_BF16, "plan_search_hidden: unknown precision %d", prec);
  TACORL_REQUIRE(layer >= 1, "plan_search_hidden: layer %d (layer 0 is sample_l0's)", layer);
  TACORL_REQUIRE(W1 && b1 && W2 && b2 && ws, "plan_search_hidden: null pointer");
  TACORL_REQUIRE(ws_bytes >= tacorl_plan_search_ws_bytes(n, K, 1, H) && ps_aligned16(ws),
                 "plan_search_hidden: workspace too small or not 16-byte aligned");
  const PsLayout l = ps_layout(ws, n, K, H);
  cudaStream_t st = (cudaStream_t)stream;
  const int src = (layer - 1) & 1, dst = layer & 1;
  const int rows = n * K;
  for (int j = 0; j < 2; ++j) {
    const float* W = j ? W2 : W1;
    const float* b = j ? b2 : b1;
    if (prec == PREC_BF16) {
      const void* Wb = j ? W2_bf16 : W1_bf16;
      if (!Wb || !ps_aligned16(Wb)) {   // TMA reads 16-byte aligned rows: stage the weight
        if ((rc = cast_bf16_2d(W, H, H, H, l.wcast, H, st))) return rc;
        Wb = l.wcast;
      }
      TcArgs e;
      e.C = l.h[j][dst]; e.ldc = H; e.Cb = l.hb[j][dst]; e.ldcb = H; e.bias = b; e.act = ACT_SILU;
      e.split_k = 1;                  // "auto" may depend on the row count: a row's sum must not
      if ((rc = gemm_tc_bf16(l.hb[j][src], H, 0, Wb, H, 0, rows, H, H, e, nullptr, 0, st))) return rc;
    } else {
      GemmArgs g;
      g.transB = 1; g.M = rows; g.N = H; g.K = H;
      g.A = l.h[j][src]; g.lda = H; g.B = W; g.ldb = H; g.C = l.h[j][dst]; g.ldc = H; g.bias = b; g.act = ACT_SILU;
      g.split_k = 1;
      if ((rc = gemm_f32(g, nullptr, 0, st))) return rc;
    }
  }
  return 0;
}

int tacorl_plan_search_select(int n, int K, int P, int H, int L, int E, int k, int last, float min_std, const float* z,
                              const float* w_out1, const float* b_out1, const float* w_out2, const float* b_out2,
                              float* scores, float* mu, float* sigma, float* best_z, float* best_s, const int* restart,
                              float* plan, float* plan_value, const void* ws, size_t ws_bytes, void* stream) {
  int rc;
  if ((rc = ps_check(n, K, P, H, "plan_search_select"))) return rc;
  TACORL_REQUIRE(L >= 1 && E >= 1 && E <= K && k >= 0 && min_std > 0.f,
                 "plan_search_select: layers %d, elites %d of %d, iteration %d, min_std %g", L, E, K, k, min_std);
  TACORL_REQUIRE(z && w_out1 && b_out1 && w_out2 && b_out2 && scores && mu && sigma && best_z && best_s && ws &&
                 (!last || (plan && plan_value)), "plan_search_select: null pointer");
  TACORL_REQUIRE(ws_bytes >= tacorl_plan_search_ws_bytes(n, K, P, H) && ps_aligned16(ws),
                 "plan_search_select: workspace too small or not 16-byte aligned");
  const PsLayout l = ps_layout(const_cast<void*>(ws), n, K, H);
  const int s = (L - 1) & 1;
  plan_search_select_kernel<<<n, kPsThreads, 0, (cudaStream_t)stream>>>(
      K, P, H, E, k, last, min_std, z, l.h[0][s], w_out1, b_out1, l.h[1][s], w_out2, b_out2, scores, mu, sigma, best_z,
      best_s, restart, plan, plan_value);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
