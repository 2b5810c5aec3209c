// ReLU Elman RNN layer (one direction), forward and BPTT backward, time-major buffers.
// C-ABI: tacorl_rnn_layer_{fwd,bwd}.  Replaces nn.RNN(nonlinearity="relu") as used by the
// plan-recognition BiRNN (/root/reference/src/tacorl/networks/plan_encoders/
// plan_recognition_tanh_net.py:23-31, plan_recognition_net.py:27-35) and the action decoder
// (networks/action_decoders/rnn_models.py:5-16):
//     h_t = relu(W_ih x_t + b_ih + W_hh h_{t-1} + b_hh),  h_init = h0 or 0.
// `n_steps` < T runs only the first n_steps of the recurrence (reverse: starting at t = T-1);
// the BiRNN's last-layer reverse direction only needs one step because only out[:, -1] is
// consumed (plan_recognition_tanh_net.py:43; SURVEY.md §0 finding 7-ii).
// fp32 parity path: one input GEMM for all steps + one recurrent GEMM per step.
#include "common.cuh"
#include "internal.h"
#include "../../include/tacorl_b200.h"
#include <cuda_bf16.h>

namespace tacorl {

__global__ void vec_add_kernel(int n, const float* a, const float* b, float* o) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = a[i] + b[i];
}

// rows x H block with row stride ld: p = relu(p)  (+ optional bf16 copy with row pitch ldb)
__global__ void relu_rows_kernel(long long rows, int H, float* p, long long ld, __nv_bfloat16* pb, long long ldb) {
  const long long total = rows * H;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    float* q = p + (i / H) * ld + (i % H);
    const float v = fmaxf(*q, 0.f);
    *q = v;
    if (pb) pb[(i / H) * ldb + (i % H)] = __float2bfloat16(v);
  }
}

// d = (d + add?) * [out > 0]  (+ optional bf16 copy with row pitch lddb)
__global__ void mask_rows_kernel(long long rows, int H, float* d, long long ldd, const float* out,
                                 long long ldo, const float* add, long long lda, __nv_bfloat16* db, long long lddb) {
  const long long total = rows * H;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / H; const int c = (int)(i % H);
    float v = d[r * ldd + c];
    if (add) v += add[r * lda + c];
    v = out[r * ldo + c] > 0.f ? v : 0.f;
    d[r * ldd + c] = v;
    if (db) db[r * lddb + c] = __float2bfloat16(v);
  }
}

static inline int ew_blocks(long long n) { return (int)min((long long)1184, (n + 255) / 256); }

}  // namespace tacorl

using namespace tacorl;

extern "C" {

size_t tacorl_rnn_layer_ws_bytes(int T, int B, int I, int H) {
  // bias sum + split-K partials for the recurrent GEMM (<= 16 splits of BxH) and the weight grads;
  // bf16 path: staged copies of W_ih, W_hh, x, h / dpre
  const size_t mx = (size_t)(H > I ? H : I);
  size_t sk = (size_t)16 * B * H * 4;
  size_t wg = (size_t)4 * H * mx * 4;
  size_t bf = ((size_t)H * (I + 8) + (size_t)H * H + (size_t)T * B * (I + 8) + 2 * (size_t)T * B * H) * 2 + 8192;
  return (size_t)H * 4 + 4096 + (sk > wg ? sk : wg) + bf + (1 << 16);
}

static int rnn_fwd_f32(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                       const float* w_hh, const float* b_ih, const float* b_hh, const float* h0,
                       int reverse, int n_steps, float* out, long long ldo, const void*, const void*, void*, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  TACORL_REQUIRE(x && w_ih && w_hh && b_ih && b_hh && out && ws, "rnn_layer_fwd: null pointer");
  TACORL_REQUIRE(n_steps >= 1 && n_steps <= T, "rnn_layer_fwd: n_steps %d out of range (T=%d)", n_steps, T);
  if (B == 0) return 0;
  Arena ar(ws, ws_bytes);
  float* bsum = ar.take<float>(H);
  TACORL_REQUIRE(bsum, "rnn_layer_fwd: workspace too small");
  float* sk = (float*)(ar.base + ar.off);
  size_t sk_bytes = ar.left();
  vec_add_kernel<<<cdiv(H, 256), 256, 0, st>>>(H, b_ih, b_hh, bsum);
  TACORL_LAUNCH_CHECK();
  const int t_lo = reverse ? T - n_steps : 0;
  int rc;
  GemmArgs in;   // pre-activations of all steps: out[t] = x[t] W_ih^T + (b_ih + b_hh)
  in.transB = 1; in.M = n_steps * B; in.N = H; in.K = I;
  in.A = x + (long long)t_lo * B * ldx; in.lda = ldx; in.B = w_ih; in.ldb = I;
  in.C = out + (long long)t_lo * B * ldo; in.ldc = ldo; in.bias = bsum; in.split_k = 0;
  if ((rc = gemm_f32(in, sk, sk_bytes, st))) return rc;
  for (int s = 0; s < n_steps; ++s) {
    const int t = reverse ? T - 1 - s : s;
    float* ot = out + (long long)t * B * ldo;
    const float* hp; long long ldh;
    if (s == 0) { hp = h0; ldh = H; }
    else { hp = out + (long long)(reverse ? t + 1 : t - 1) * B * ldo; ldh = ldo; }
    if (!hp) {
      relu_rows_kernel<<<ew_blocks((long long)B * H), 256, 0, st>>>(B, H, ot, ldo, nullptr, 0);
      TACORL_LAUNCH_CHECK();
      continue;
    }
    GemmArgs r;
    r.transB = 1; r.M = B; r.N = H; r.K = H; r.A = hp; r.lda = ldh; r.B = w_hh; r.ldb = H;
    r.C = ot; r.ldc = ldo; r.beta = 1.f; r.act = ACT_RELU; r.split_k = 0;
    if ((rc = gemm_f32(r, sk, sk_bytes, st))) return rc;
  }
  return 0;
}

static int rnn_bwd_f32(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                       const float* w_hh, const float* h0, int reverse, int n_steps, const float* out,
                       long long ldo, float* dout, long long lddo, const float* dhn, float* dx,
                       long long lddx, int dx_accumulate, float* dw_ih, float* dw_hh, float* db_ih,
                       float* db_hh, int accumulate, float* dh0, const void*, const void*, const void*, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  TACORL_REQUIRE(x && w_ih && w_hh && out && dout && ws, "rnn_layer_bwd: null pointer");
  TACORL_REQUIRE(n_steps >= 1 && n_steps <= T, "rnn_layer_bwd: n_steps out of range");
  if (B == 0) return 0;
  float* sk = (float*)ws;
  size_t sk_bytes = ws_bytes;
  const float beta0 = accumulate ? 1.f : 0.f;
  const int t_lo = reverse ? T - n_steps : 0;
  int rc;
  // BPTT: walk the recurrence backwards; dout[t] becomes dpre[t] in place.
  for (int s = n_steps - 1; s >= 0; --s) {
    const int t = reverse ? T - 1 - s : s;
    float* dt = dout + (long long)t * B * lddo;
    const float* ot = out + (long long)t * B * ldo;
    mask_rows_kernel<<<ew_blocks((long long)B * H), 256, 0, st>>>(
        B, H, dt, lddo, ot, ldo, (s == n_steps - 1) ? dhn : nullptr, H, nullptr, 0);
    TACORL_LAUNCH_CHECK();
    if (s > 0) {  // dout[t_prev] += dpre[t] W_hh
      const int tp = reverse ? t + 1 : t - 1;
      GemmArgs c;
      c.M = B; c.N = H; c.K = H; c.A = dt; c.lda = lddo; c.B = w_hh; c.ldb = H;
      c.C = dout + (long long)tp * B * lddo; c.ldc = lddo; c.beta = 1.f; c.split_k = 0;
      if ((rc = gemm_f32(c, sk, sk_bytes, st))) return rc;
    } else if (dh0) {
      GemmArgs c;
      c.M = B; c.N = H; c.K = H; c.A = dt; c.lda = lddo; c.B = w_hh; c.ldb = H; c.C = dh0; c.ldc = H;
      c.split_k = 0;
      if ((rc = gemm_f32(c, sk, sk_bytes, st))) return rc;
    }
  }
  float* dpre = dout + (long long)t_lo * B * lddo;
  const long long rows = (long long)n_steps * B;
  // dW_hh (+)= sum_{s>=1} dpre[t(s)]^T h[t(s-1)]  (+ dpre[t(0)]^T h0)
  if (dw_hh) {
    bool wrote = false;
    if (n_steps > 1) {
      GemmArgs w;
      w.transA = 1; w.M = H; w.N = H; w.K = (n_steps - 1) * B;
      if (!reverse) { w.A = dpre + (long long)B * lddo; w.B = out; }
      else { w.A = dpre; w.B = out + (long long)(t_lo + 1) * B * ldo; }
      w.lda = lddo; w.ldb = ldo; w.C = dw_hh; w.ldc = H; w.beta = beta0; w.split_k = 0;
      if ((rc = gemm_f32(w, sk, sk_bytes, st))) return rc;
      wrote = true;
    }
    if (h0) {
      const int t0 = reverse ? T - 1 : 0;
      GemmArgs w;
      w.transA = 1; w.M = H; w.N = H; w.K = B; w.A = dout + (long long)t0 * B * lddo; w.lda = lddo;
      w.B = h0; w.ldb = H; w.C = dw_hh; w.ldc = H; w.beta = wrote ? 1.f : beta0; w.split_k = 0;
      if ((rc = gemm_f32(w, sk, sk_bytes, st))) return rc;
      wrote = true;
    }
    if (!wrote && !accumulate) TACORL_CHECK_CUDA(cudaMemsetAsync(dw_hh, 0, (size_t)H * H * 4, st));
  }
  if (dw_ih) {
    GemmArgs w;
    w.transA = 1; w.M = H; w.N = I; w.K = (int)rows; w.A = dpre; w.lda = lddo;
    w.B = x + (long long)t_lo * B * ldx; w.ldb = ldx; w.C = dw_ih; w.ldc = I; w.beta = beta0; w.split_k = 0;
    if ((rc = gemm_f32(w, sk, sk_bytes, st))) return rc;
  }
  // db_ih == db_hh == column sums of dpre: reduce once, reuse
  if (db_ih || db_hh) {
    float* first = db_ih ? db_ih : db_hh;
    if (!accumulate) {
      if ((rc = colsum2_f32((int)rows, H, dpre, lddo, first, 0, sk, sk_bytes, st))) return rc;
      if (db_ih && db_hh) TACORL_CHECK_CUDA(cudaMemcpyAsync(db_hh, db_ih, (size_t)H * 4, cudaMemcpyDeviceToDevice, st));
    } else {
      if (db_ih) if ((rc = colsum2_f32((int)rows, H, dpre, lddo, db_ih, 1, sk, sk_bytes, st))) return rc;
      if (db_hh) if ((rc = colsum2_f32((int)rows, H, dpre, lddo, db_hh, 1, sk, sk_bytes, st))) return rc;
    }
  }
  if (dx) {
    if (!dx_accumulate && n_steps < T) {
      // rows outside the active range receive no gradient
      const long long lo_rows = (long long)t_lo * B, hi_rows = (long long)(T - t_lo - n_steps) * B;
      if (lo_rows) TACORL_CHECK_CUDA(cudaMemset2DAsync(dx, lddx * 4, 0, (size_t)I * 4, lo_rows, st));
      if (hi_rows) TACORL_CHECK_CUDA(cudaMemset2DAsync(dx + (long long)(t_lo + n_steps) * B * lddx, lddx * 4, 0,
                                                       (size_t)I * 4, hi_rows, st));
    }
    GemmArgs d;
    d.M = (int)rows; d.N = I; d.K = H; d.A = dpre; d.lda = lddo; d.B = w_ih; d.ldb = I;
    d.C = dx + (long long)t_lo * B * lddx; d.ldc = lddx; d.beta = dx_accumulate ? 1.f : 0.f; d.split_k = 0;
    if ((rc = gemm_f32(d, sk, sk_bytes, st))) return rc;
  }
  return 0;
}


// ------------------------------------------------------------------------------------------ bf16 tensor-core path
// Weights are staged to bf16 once per call; h_t / dpre_t are written in fp32 (saved / accumulated) and as
// dense bf16 copies that feed the next step's tcgen05 GEMM.  No transposes: W_hh / W_ih / dpre / h / x are
// consumed in their stored orientation through K-major or MN-major UMMA descriptors.
static int rnn_fwd_bf16(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                        const float* w_hh, const float* b_ih, const float* b_hh, const float* h0,
                        int reverse, int n_steps, float* out, long long ldo, const void* w_ih_bf16,
                        const void* w_hh_bf16, void* h_bf16_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  const long long Ip = (I + 7) & ~7LL;
  // caller-maintained bf16 weight copies (tacorl_adam_step shadow) replace the per-call staging casts
  const bool wih_ready = w_ih_bf16 && Ip == I && ((uintptr_t)w_ih_bf16 & 15) == 0;
  const bool whh_ready = w_hh_bf16 && ((uintptr_t)w_hh_bf16 & 15) == 0;
  Arena ar(ws, ws_bytes);
  float* bsum = ar.take<float>(H);
  const __nv_bfloat16* wih = wih_ready ? (const __nv_bfloat16*)w_ih_bf16 : ar.take<__nv_bfloat16>((size_t)H * Ip);
  const __nv_bfloat16* whh = whh_ready ? (const __nv_bfloat16*)w_hh_bf16 : ar.take<__nv_bfloat16>((size_t)H * H);
  __nv_bfloat16* xb = ar.take<__nv_bfloat16>((size_t)n_steps * B * Ip);
  // the bf16 hidden states are the next step's operand; a caller that will run the backward pass keeps them
  // (h_bf16_out, dense [T][B][H]) so that BPTT does not have to re-cast the saved fp32 activations
  const bool hb_ext = h_bf16_out && ((uintptr_t)h_bf16_out & 15) == 0;
  __nv_bfloat16* hb = hb_ext ? (__nv_bfloat16*)h_bf16_out : ar.take<__nv_bfloat16>((size_t)T * B * H);
  __nv_bfloat16* h0b = h0 ? ar.take<__nv_bfloat16>((size_t)B * H) : nullptr;
  unsigned* flags = ar.take<unsigned>(64);
  TACORL_REQUIRE(bsum && wih && whh && xb && hb && (!h0 || h0b) && flags, "rnn_layer_fwd(bf16): workspace too small");
  TACORL_REQUIRE(H % 8 == 0, "rnn_layer_fwd(bf16): hidden size must be a multiple of 8");
  float* sk = (float*)(ar.base + ar.off);
  size_t sk_bytes = ar.left();
  const int t_lo = reverse ? T - n_steps : 0;
  int rc;
  vec_add_kernel<<<cdiv(H, 256), 256, 0, st>>>(H, b_ih, b_hh, bsum);
  TACORL_LAUNCH_CHECK();
  if (!wih_ready && (rc = cast_bf16_2d(w_ih, I, H, I, (void*)wih, Ip, st))) return rc;
  if (!whh_ready && (rc = cast_bf16_2d(w_hh, H, H, H, (void*)whh, H, st))) return rc;
  if ((rc = cast_bf16_2d(x + (long long)t_lo * B * ldx, ldx, (long long)n_steps * B, I, xb, Ip, st))) return rc;
  if (h0 && (rc = cast_bf16_2d(h0, H, B, H, h0b, H, st))) return rc;
  TcArgs in;
  in.C = out + (long long)t_lo * B * ldo; in.ldc = ldo; in.bias = bsum; in.split_k = 1;
  if ((rc = gemm_tc_bf16(xb, Ip, 0, wih, Ip, 0, n_steps * B, H, I, in, sk, sk_bytes, st))) return rc;
  for (int s = 0; s < n_steps; ++s) {
    const int t = reverse ? T - 1 - s : s;
    float* ot = out + (long long)t * B * ldo;
    __nv_bfloat16* hbt = hb + (long long)t * B * H;
    const __nv_bfloat16* hp = (s == 0) ? h0b : hb + (long long)(reverse ? t + 1 : t - 1) * B * H;
    if (!hp) {
      relu_rows_kernel<<<ew_blocks((long long)B * H), 256, 0, st>>>(B, H, ot, ldo, hbt, H);
      TACORL_LAUNCH_CHECK();
      continue;
    }
    if (s == 1 && flags) {   // steps 1 .. n_steps-1 in one persistent launch (weights resident in shared memory)
      rc = rnn_seq_tc(hb, T, whh, H, B, H, H, t, reverse ? -1 : 1, n_steps - 1, 1.f, out, ldo, (long long)B * ldo, nullptr, 0,
                      0, hb, ACT_RELU, flags, st);
      if (rc < 0) return rc;
      if (rc == 0) break;
    }
    TcArgs r;
    r.C = ot; r.ldc = ldo; r.beta = 1.f; r.act = ACT_RELU; r.Cb = hbt; r.ldcb = H; r.split_k = 0;
    if ((rc = gemm_tc_bf16(hp, H, 0, whh, H, 0, B, H, H, r, sk, sk_bytes, st))) return rc;
  }
  return 0;
}

static int rnn_bwd_bf16(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                        const float* w_hh, const float* h0, int reverse, int n_steps, const float* out,
                        long long ldo, float* dout, long long lddo, const float* dhn, float* dx,
                        long long lddx, int dx_accumulate, float* dw_ih, float* dw_hh, float* db_ih,
                        float* db_hh, int accumulate, float* dh0, const void* w_ih_bf16, const void* w_hh_t_bf16,
                        const void* h_bf16, void* ws, size_t ws_bytes, cudaStream_t st) {
  const long long Ip = (I + 7) & ~7LL;
  const bool wih_ready = w_ih_bf16 && Ip == I && ((uintptr_t)w_ih_bf16 & 15) == 0;
  const bool whht_ready = w_hh_t_bf16 && ((uintptr_t)w_hh_t_bf16 & 15) == 0;   // W_hh^T, prepared off the critical path
  const bool hb_ready = h_bf16 && ((uintptr_t)h_bf16 & 15) == 0;               // bf16 hidden states kept by the forward
  Arena ar(ws, ws_bytes);
  const __nv_bfloat16* wih = wih_ready ? (const __nv_bfloat16*)w_ih_bf16 : ar.take<__nv_bfloat16>((size_t)H * Ip);
  __nv_bfloat16* whh = whht_ready ? (__nv_bfloat16*)w_hh_t_bf16 : ar.take<__nv_bfloat16>((size_t)H * H);
  __nv_bfloat16* xb = ar.take<__nv_bfloat16>((size_t)n_steps * B * Ip);
  __nv_bfloat16* hb = hb_ready ? (__nv_bfloat16*)h_bf16 : ar.take<__nv_bfloat16>((size_t)T * B * H);
  __nv_bfloat16* db = ar.take<__nv_bfloat16>((size_t)T * B * H);
  __nv_bfloat16* h0b = h0 ? ar.take<__nv_bfloat16>((size_t)B * H) : nullptr;
  unsigned* flags = ar.take<unsigned>(64);
  TACORL_REQUIRE(wih && whh && xb && hb && db && (!h0 || h0b) && flags, "rnn_layer_bwd(bf16): workspace too small");
  float* sk = (float*)(ar.base + ar.off);
  size_t sk_bytes = ar.left();
  const float beta0 = accumulate ? 1.f : 0.f;
  const int t_lo = reverse ? T - n_steps : 0;
  const long long rows = (long long)n_steps * B;
  int rc;
  if (!wih_ready && (rc = cast_bf16_2d(w_ih, I, H, I, (void*)wih, Ip, st))) return rc;
  if (!whht_ready && (rc = cast_transpose_bf16(w_hh, H, H, H, whh, H, st))) return rc;   // W_hh^T: K-major B for the carry GEMM
  if ((rc = cast_bf16_2d(x + (long long)t_lo * B * ldx, ldx, rows, I, xb, Ip, st))) return rc;
  if (!hb_ready && (rc = cast_bf16_2d(out + (long long)t_lo * B * ldo, ldo, rows, H, hb + (long long)t_lo * B * H, H, st))) return rc;
  if (h0 && (rc = cast_bf16_2d(h0, H, B, H, h0b, H, st))) return rc;
  {  // last step of the recurrence: dpre = (dout (+ dhn)) * [h > 0]
    const int t = reverse ? T - n_steps : n_steps - 1;
    mask_rows_kernel<<<ew_blocks((long long)B * H), 256, 0, st>>>(
        B, H, dout + (long long)t * B * lddo, lddo, out + (long long)t * B * ldo, ldo, dhn, H, db + (long long)t * B * H, H);
    TACORL_LAUNCH_CHECK();
  }
  for (int s = n_steps - 1; s >= 0; --s) {
    const int t = reverse ? T - 1 - s : s;
    __nv_bfloat16* dbt = db + (long long)t * B * H;
    if (s == n_steps - 1 && s > 0) {   // the whole BPTT chain s = n_steps-1 .. 1 in one persistent launch
      const int tp = reverse ? t + 1 : t - 1;
      rc = rnn_seq_tc(db, T, whh, H, B, H, H, tp, reverse ? 1 : -1, n_steps - 1, 1.f, dout, lddo, (long long)B * lddo, out, ldo,
                      (long long)B * ldo, db, ACT_NONE, flags, st);
      if (rc < 0) return rc;
      if (rc == 0) { s = 1; continue; }   // resume at s = 0 (dh0)
    }
    if (s > 0) {   // dpre[t_prev] = (dout[t_prev] + dpre[t] W_hh) * [h[t_prev] > 0], one fused GEMM (+ bf16 copy)
      const int tp = reverse ? t + 1 : t - 1;
      TcArgs c;
      c.C = dout + (long long)tp * B * lddo; c.ldc = lddo; c.beta = 1.f; c.split_k = 0;
      c.gate = out + (long long)tp * B * ldo; c.ldgate = ldo;
      c.Cb = db + (long long)tp * B * H; c.ldcb = H;
      if ((rc = gemm_tc_bf16(dbt, H, 0, whh, H, 0, B, H, H, c, sk, sk_bytes, st))) return rc;
    } else if (dh0) {
      TcArgs c;
      c.C = dh0; c.ldc = H; c.split_k = 1;
      if ((rc = gemm_tc_bf16(dbt, H, 0, whh, H, 0, B, H, H, c, sk, sk_bytes, st))) return rc;
    }
  }
  float* dpre = dout + (long long)t_lo * B * lddo;
  const __nv_bfloat16* dpb = db + (long long)t_lo * B * H;
  if (dw_hh) {
    bool wrote = false;
    if (n_steps > 1) {   // dW_hh = dpre[pairs]^T h[prev]: both operands stored [K=rows][H]: MN-major
      const __nv_bfloat16 *a, *b;
      if (!reverse) { a = dpb + (long long)B * H; b = hb; }
      else { a = dpb; b = hb + (long long)(t_lo + 1) * B * H; }
      TcArgs w;
      w.C = dw_hh; w.ldc = H; w.beta = beta0; w.split_k = 0;
      if ((rc = gemm_tc_bf16(a, H, 1, b, H, 1, H, H, (n_steps - 1) * B, w, sk, sk_bytes, st))) return rc;
      wrote = true;
    }
    if (h0) {
      const int t0 = reverse ? T - 1 : 0;
      TcArgs w;
      w.C = dw_hh; w.ldc = H; w.beta = wrote ? 1.f : beta0; w.split_k = 0;
      if ((rc = gemm_tc_bf16(db + (long long)t0 * B * H, H, 1, h0b, H, 1, H, H, B, w, sk, sk_bytes, st))) return rc;
      wrote = true;
    }
    if (!wrote && !accumulate) TACORL_CHECK_CUDA(cudaMemsetAsync(dw_hh, 0, (size_t)H * H * 4, st));
  }
  if (dw_ih) {
    TcArgs w;
    w.C = dw_ih; w.ldc = I; w.beta = beta0; w.split_k = 0;
    if ((rc = gemm_tc_bf16(dpb, H, 1, xb, Ip, 1, H, I, (int)rows, w, sk, sk_bytes, st))) return rc;
  }
  // db_ih == db_hh == column sums of dpre: reduce once, reuse
  if (db_ih || db_hh) {
    float* first = db_ih ? db_ih : db_hh;
    if (!accumulate) {
      if ((rc = colsum2_f32((int)rows, H, dpre, lddo, first, 0, sk, sk_bytes, st))) return rc;
      if (db_ih && db_hh) TACORL_CHECK_CUDA(cudaMemcpyAsync(db_hh, db_ih, (size_t)H * 4, cudaMemcpyDeviceToDevice, st));
    } else {
      if (db_ih) if ((rc = colsum2_f32((int)rows, H, dpre, lddo, db_ih, 1, sk, sk_bytes, st))) return rc;
      if (db_hh) if ((rc = colsum2_f32((int)rows, H, dpre, lddo, db_hh, 1, sk, sk_bytes, st))) return rc;
    }
  }
  if (dx) {
    if (!dx_accumulate && n_steps < T) {
      const long long lo_rows = (long long)t_lo * B, hi_rows = (long long)(T - t_lo - n_steps) * B;
      if (lo_rows) TACORL_CHECK_CUDA(cudaMemset2DAsync(dx, lddx * 4, 0, (size_t)I * 4, lo_rows, st));
      if (hi_rows) TACORL_CHECK_CUDA(cudaMemset2DAsync(dx + (long long)(t_lo + n_steps) * B * lddx, lddx * 4, 0,
                                                       (size_t)I * 4, hi_rows, st));
    }
    TcArgs d;   // dx = dpre W_ih  (B operand = W_ih as stored [K=H][N=I]: MN-major)
    d.C = dx + (long long)t_lo * B * lddx; d.ldc = lddx; d.beta = dx_accumulate ? 1.f : 0.f; d.split_k = 1;
    if ((rc = gemm_tc_bf16(dpb, H, 0, wih, Ip, 1, (int)rows, I, H, d, sk, sk_bytes, st))) return rc;
  }
  return 0;
}


// ------------------------------------------------------------------------------------------ whole layer, both directions
// bf16 tensor-core path of one (bi)directional layer in one call: the two directions' recurrences run side by side in
// ONE persistent launch (rnn_wave_kernel, batch <= 64), the hidden states / pre-activation gradients have bf16 twins in
// the layer's own (T, B, D*H) layout (written by the recurrence kernels), so the next layer's input projection, the BPTT
// and the weight-gradient GEMMs read them in place: no staging casts, no per-direction streams, no concat.
struct Layer2Ws {
  float* bsum[2] = {nullptr, nullptr};
  const __nv_bfloat16* wih[2] = {nullptr, nullptr};
  const __nv_bfloat16* whh[2] = {nullptr, nullptr};
  const __nv_bfloat16* xb = nullptr; long long ldxb = 0;
  unsigned* flags = nullptr;
  float* sk = nullptr; size_t sk_bytes = 0;
};

static int layer2_fwd_bf16(int T, int B, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                           long long ldxb, const float* const* w, const void* const* w_bf16, const int* n_steps,
                           float* out, long long ldo, void* out_bf16, void* ws, size_t ws_bytes, cudaStream_t st) {
  TACORL_REQUIRE(x && w && n_steps && out && out_bf16 && ws, "rnn_layer2_fwd: null pointer");
  TACORL_REQUIRE(D == 1 || D == 2, "rnn_layer2_fwd: D must be 1 or 2");
  TACORL_REQUIRE(H % 8 == 0 && ldo % 8 == 0 && ((uintptr_t)out_bf16 & 15) == 0,
                 "rnn_layer2_fwd: hidden size / output pitch must be multiples of 8 and the bf16 twin 16-byte aligned");
  for (int d = 0; d < D; ++d)
    TACORL_REQUIRE(n_steps[d] >= 1 && n_steps[d] <= T, "rnn_layer2_fwd: n_steps[%d] = %d out of range (T=%d)", d, n_steps[d], T);
  if (B == 0) return 0;
  const long long Ip = (I + 7) & ~7LL;
  Arena ar(ws, ws_bytes);
  Layer2Ws L;
  int rc;
  for (int d = 0; d < D; ++d) {
    L.bsum[d] = ar.take<float>(H);
    const void* tih = w_bf16 ? w_bf16[2 * d] : nullptr;
    const void* thh = w_bf16 ? w_bf16[2 * d + 1] : nullptr;
    const bool ih_ready = tih && Ip == I && ((uintptr_t)tih & 15) == 0, hh_ready = thh && ((uintptr_t)thh & 15) == 0;
    __nv_bfloat16* cih = ih_ready ? nullptr : ar.take<__nv_bfloat16>((size_t)H * Ip);
    __nv_bfloat16* chh = hh_ready ? nullptr : ar.take<__nv_bfloat16>((size_t)H * H);
    TACORL_REQUIRE(L.bsum[d] && (ih_ready || cih) && (hh_ready || chh), "rnn_layer2_fwd: workspace too small");
    if (!ih_ready && (rc = cast_bf16_2d(w[4 * d], I, H, I, cih, Ip, st))) return rc;
    if (!hh_ready && (rc = cast_bf16_2d(w[4 * d + 1], H, H, H, chh, H, st))) return rc;
    L.wih[d] = ih_ready ? (const __nv_bfloat16*)tih : cih;
    L.whh[d] = hh_ready ? (const __nv_bfloat16*)thh : chh;
    vec_add_kernel<<<cdiv(H, 256), 256, 0, st>>>(H, w[4 * d + 2], w[4 * d + 3], L.bsum[d]);
    TACORL_LAUNCH_CHECK();
  }
  const bool x_ready = x_bf16 && ldxb % 8 == 0 && ldxb >= I && ((uintptr_t)x_bf16 & 15) == 0 && (I % 8 == 0);
  if (x_ready) { L.xb = (const __nv_bfloat16*)x_bf16; L.ldxb = ldxb; }
  else {
    __nv_bfloat16* xc = ar.take<__nv_bfloat16>((size_t)T * B * Ip);
    TACORL_REQUIRE(xc, "rnn_layer2_fwd: workspace too small");
    if ((rc = cast_bf16_2d(x, ldx, (long long)T * B, I, xc, Ip, st))) return rc;
    L.xb = xc; L.ldxb = Ip;
  }
  L.flags = ar.take<unsigned>(128);
  TACORL_REQUIRE(L.flags, "rnn_layer2_fwd: workspace too small");
  L.sk = (float*)(ar.base + ar.off); L.sk_bytes = ar.left();
  __nv_bfloat16* outb = (__nv_bfloat16*)out_bf16;
  WaveLaneHost lanes[2];
  int n_lanes = 0;
  for (int d = 0; d < D; ++d) {
    const int n = n_steps[d], t_lo = d ? T - n : 0, t0 = d ? T - 1 : 0;
    TcArgs in;   // pre-activations of the active steps: out[t, :, dH:(d+1)H] = x[t] W_ih^T + (b_ih + b_hh)
    in.C = out + (long long)t_lo * B * ldo + (long long)d * H; in.ldc = ldo; in.bias = L.bsum[d];
    in.split_k = n * B <= 128 ? 0 : 1;      // a single step (the top layer's reverse direction): the cluster split-K kernel
    if ((rc = gemm_tc_bf16(L.xb + (long long)t_lo * B * L.ldxb, L.ldxb, 0, L.wih[d], Ip, 0, n * B, H, I, in, L.sk, L.sk_bytes, st)))
      return rc;
    // first step: h_init = 0
    relu_rows_kernel<<<ew_blocks((long long)B * H), 256, 0, st>>>(B, H, out + (long long)t0 * B * ldo + (long long)d * H, ldo,
                                                                 outb + (long long)t0 * B * ldo + (long long)d * H, ldo);
    TACORL_LAUNCH_CHECK();
    if (n > 1) {
      WaveLaneHost& h = lanes[n_lanes];
      h.Ab = outb + (long long)d * H; h.lda = ldo; h.a_ts = (long long)B * ldo;
      h.W = L.whh[d]; h.ldw = H;
      h.tau0 = d ? T - 2 : 1; h.dtau = d ? -1 : 1; h.n_steps = n - 1; h.beta = 1.f;
      h.C = out + (long long)d * H; h.ldc = ldo; h.c_ts = (long long)B * ldo;
      h.Cb = outb + (long long)d * H; h.ldcb = ldo; h.cb_ts = (long long)B * ldo;
      h.act = ACT_RELU; h.flags = L.flags + 64 * n_lanes;
      ++n_lanes;
    }
  }
  if (n_lanes == 0) return 0;
  rc = rnn_wave_tc(lanes, n_lanes, T, B, H, H, st);
  if (rc <= 0) return rc;
  for (int l = 0; l < n_lanes; ++l) {          // shapes the two-lane kernel does not cover
    const WaveLaneHost& h = lanes[l];
    rc = 1;
    if (h.lda == H)                              // dense hidden states (D == 1): the 8-way persistent kernel, batch <= 128
      rc = rnn_seq_tc(h.Ab, T, h.W, H, B, H, H, h.tau0, h.dtau, h.n_steps, 1.f, h.C, h.ldc, h.c_ts, nullptr, 0, 0, h.Cb,
                      ACT_RELU, h.flags, st);
    if (rc < 0) return rc;
    if (rc == 0) continue;
    for (int s = 0; s < h.n_steps; ++s) {        // step by step
      const int tau = h.tau0 + s * h.dtau;
      TcArgs r;
      r.C = h.C + (long long)tau * h.c_ts; r.ldc = h.ldc; r.beta = 1.f; r.act = ACT_RELU;
      r.Cb = (__nv_bfloat16*)h.Cb + (long long)tau * h.cb_ts; r.ldcb = h.ldcb; r.split_k = 0;
      if ((rc = gemm_tc_bf16((const __nv_bfloat16*)h.Ab + (long long)(tau - h.dtau) * h.a_ts, h.lda, 0, h.W, H, 0, B, H, H, r,
                             L.sk, L.sk_bytes, st)))
        return rc;
    }
  }
  return 0;
}

// Weight gradients of one layer2 backward, once its recurrence has written dpre (fp32 in dout, bf16 twin in dpre_bf16):
// dW_hh = dpre[pairs]^T h[prev], dW_ih = dpre^T x, db_ih = db_hh = column sums of dpre.  Nothing on the dependent chain
// (the next layer's BPTT) reads them, so tacorl_rnn_layer2_wgrad issues them on a second stream beside that chain; the
// one-call backward runs the same code on its own stream.  max_ctas caps the GEMMs' persistent grids (TcArgs::max_ctas).
static int layer2_wgrad_bf16(int T, int B, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                             long long ldxb, const int* n_steps, const void* out_bf16, long long ldo, const float* dout,
                             long long lddo, const void* dpre_bf16, float* const* dw, void* ws, size_t ws_bytes,
                             int max_ctas, cudaStream_t st) {
  const long long Ip = (I + 7) & ~7LL;
  Arena ar(ws, ws_bytes);
  int rc;
  bool need_x = false;
  for (int d = 0; d < D; ++d) need_x = need_x || dw[4 * d];
  const __nv_bfloat16* xb = nullptr; long long ldb_x = 0;
  const bool x_ready = x_bf16 && ldxb % 8 == 0 && ldxb >= I && ((uintptr_t)x_bf16 & 15) == 0 && (I % 8 == 0);
  if (x_ready) { xb = (const __nv_bfloat16*)x_bf16; ldb_x = ldxb; }
  else if (need_x) {
    __nv_bfloat16* xc = ar.take<__nv_bfloat16>((size_t)T * B * Ip);
    TACORL_REQUIRE(xc, "rnn_layer2_bwd: workspace too small");
    if ((rc = cast_bf16_2d(x, ldx, (long long)T * B, I, xc, Ip, st))) return rc;
    xb = xc; ldb_x = Ip;
  }
  float* sk = (float*)(ar.base + ar.off);
  const size_t sk_bytes = ar.left();
  const __nv_bfloat16* hb = (const __nv_bfloat16*)out_bf16;
  const __nv_bfloat16* dpb = (const __nv_bfloat16*)dpre_bf16;
  for (int d = 0; d < D; ++d) {
    const int n = n_steps[d], t_lo = d ? T - n : 0;
    const long long col = (long long)d * H, rows = (long long)n * B;
    const float* dpre = dout + (long long)t_lo * B * lddo + col;
    const __nv_bfloat16* dp = dpb + (long long)t_lo * B * lddo + col;
    float *dw_ih = dw[4 * d], *dw_hh = dw[4 * d + 1], *db_ih = dw[4 * d + 2], *db_hh = dw[4 * d + 3];
    if (dw_hh) {
      if (n > 1) {   // dW_hh = dpre[pairs]^T h[prev]: both operands stored [K = rows][H]: MN-major
        const __nv_bfloat16 *a, *b;
        if (d == 0) { a = dp + (long long)B * lddo; b = hb + col; }
        else { a = dp; b = hb + (long long)(t_lo + 1) * B * ldo + col; }
        TcArgs g;
        g.C = dw_hh; g.ldc = H; g.split_k = 0; g.max_ctas = max_ctas;
        if ((rc = gemm_tc_bf16(a, lddo, 1, b, ldo, 1, H, H, (n - 1) * B, g, sk, sk_bytes, st))) return rc;
      } else {
        TACORL_CHECK_CUDA(cudaMemsetAsync(dw_hh, 0, (size_t)H * H * 4, st));
      }
    }
    if (dw_ih) {
      TcArgs g;
      g.C = dw_ih; g.ldc = I; g.split_k = 0; g.max_ctas = max_ctas;
      if ((rc = gemm_tc_bf16(dp, lddo, 1, xb + (long long)t_lo * B * ldb_x, ldb_x, 1, H, I, (int)rows, g, sk, sk_bytes, st))) return rc;
    }
    if (db_ih || db_hh) {   // db_ih == db_hh == column sums of dpre: reduce once, reuse
      float* first = db_ih ? db_ih : db_hh;
      if ((rc = colsum2_f32((int)rows, H, dpre, lddo, first, 0, sk, sk_bytes, st))) return rc;
      if (db_ih && db_hh) TACORL_CHECK_CUDA(cudaMemcpyAsync(db_hh, db_ih, (size_t)H * 4, cudaMemcpyDeviceToDevice, st));
    }
  }
  return 0;
}

static int layer2_bwd_bf16(int T, int B, int Bg, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                           long long ldxb, const float* const* w, const void* const* w_bf16, const int* n_steps,
                           const float* out, long long ldo, const void* out_bf16, float* dout, long long lddo,
                           void* dpre_bf16, float* dx, long long lddx, float* const* dw, void* ws, size_t ws_bytes,
                           cudaStream_t st) {
  TACORL_REQUIRE(x && w && n_steps && out && out_bf16 && dout && dpre_bf16 && dw && ws, "rnn_layer2_bwd: null pointer");
  TACORL_REQUIRE(D == 1 || D == 2, "rnn_layer2_bwd: D must be 1 or 2");
  TACORL_REQUIRE(H % 8 == 0 && ldo % 8 == 0 && lddo % 8 == 0 && ((uintptr_t)out_bf16 & 15) == 0 && ((uintptr_t)dpre_bf16 & 15) == 0,
                 "rnn_layer2_bwd: pitches must be multiples of 8 and the bf16 twins 16-byte aligned");
  TACORL_REQUIRE(n_steps[0] == T, "rnn_layer2_bwd: the forward direction must cover every step");
  TACORL_REQUIRE(Bg >= 0 && Bg <= B, "rnn_layer2_bwd: grad_rows %d out of range (B=%d)", Bg, B);
  if (B == 0) return 0;
  if (Bg == 0) Bg = B;
  const long long Ip = (I + 7) & ~7LL;
  Arena ar(ws, ws_bytes);
  int rc;
  const __nv_bfloat16* wih[2] = {nullptr, nullptr};
  const __nv_bfloat16* whht[2] = {nullptr, nullptr};
  for (int d = 0; d < D; ++d) {
    TACORL_REQUIRE(n_steps[d] >= 1 && n_steps[d] <= T, "rnn_layer2_bwd: n_steps out of range");
    const void* tih = w_bf16 ? w_bf16[2 * d] : nullptr;
    const void* tht = w_bf16 ? w_bf16[2 * d + 1] : nullptr;       // W_hh^T, prepared off the critical path
    const bool ih_ready = tih && Ip == I && ((uintptr_t)tih & 15) == 0, ht_ready = tht && ((uintptr_t)tht & 15) == 0;
    __nv_bfloat16* cih = ih_ready ? nullptr : ar.take<__nv_bfloat16>((size_t)H * Ip);
    __nv_bfloat16* cht = ht_ready ? nullptr : ar.take<__nv_bfloat16>((size_t)H * H);
    TACORL_REQUIRE((ih_ready || cih) && (ht_ready || cht), "rnn_layer2_bwd: workspace too small");
    if (!ih_ready && (rc = cast_bf16_2d(w[2 * d], I, H, I, cih, Ip, st))) return rc;
    if (!ht_ready && (rc = cast_transpose_bf16(w[2 * d + 1], H, H, H, cht, H, st))) return rc;
    wih[d] = ih_ready ? (const __nv_bfloat16*)tih : cih;
    whht[d] = ht_ready ? (const __nv_bfloat16*)tht : cht;
  }
  unsigned* flags = ar.take<unsigned>(128);
  TACORL_REQUIRE(flags, "rnn_layer2_bwd: workspace too small");
  float* sk = (float*)(ar.base + ar.off);
  const size_t sk_bytes = ar.left();
  __nv_bfloat16* dpb = (__nv_bfloat16*)dpre_bf16;
  WaveLaneHost lanes[2];
  int n_lanes = 0;
  for (int d = 0; d < D; ++d) {
    const int n = n_steps[d];
    const int t_last = d ? T - n : n - 1;     // last step of the recurrence: dpre = dout * [h > 0]
    const long long col = (long long)d * H;
    mask_rows_kernel<<<ew_blocks((long long)Bg * H), 256, 0, st>>>(
        Bg, H, dout + (long long)t_last * B * lddo + col, lddo, out + (long long)t_last * B * ldo + col, ldo, nullptr, 0,
        dpb + (long long)t_last * B * lddo + col, lddo);
    TACORL_LAUNCH_CHECK();
    if (n > 1) {   // dpre[t_prev] = (dout[t_prev] + dpre[t] W_hh) * [h[t_prev] > 0] down the whole chain
      WaveLaneHost& h = lanes[n_lanes];
      h.Ab = dpb + col; h.lda = lddo; h.a_ts = (long long)B * lddo;
      h.W = whht[d]; h.ldw = H;
      h.tau0 = d ? T - n + 1 : n - 2; h.dtau = d ? 1 : -1; h.n_steps = n - 1; h.beta = 1.f;
      h.C = dout + col; h.ldc = lddo; h.c_ts = (long long)B * lddo;
      h.gate = out + col; h.ldgate = ldo; h.gate_ts = (long long)B * ldo;
      h.Cb = dpb + col; h.ldcb = lddo; h.cb_ts = (long long)B * lddo;
      h.act = ACT_NONE; h.flags = flags + 64 * n_lanes;
      ++n_lanes;
    }
  }
  if (n_lanes > 0) {
    rc = rnn_wave_tc(lanes, n_lanes, T, Bg, H, H, st);   // (rows >= Bg of a time step carry no gradient: they stay zero)
    if (rc < 0) return rc;
    if (rc > 0) {
      for (int l = 0; l < n_lanes; ++l) {
        const WaveLaneHost& h = lanes[l];
        rc = 1;
        if (h.lda == H && h.ldgate == H && Bg == B)
          rc = rnn_seq_tc(h.Ab, T, h.W, H, B, H, H, h.tau0, h.dtau, h.n_steps, 1.f, h.C, h.ldc, h.c_ts, h.gate, h.ldgate,
                          h.gate_ts, h.Cb, ACT_NONE, h.flags, st);
        if (rc < 0) return rc;
        if (rc == 0) continue;
        for (int s = 0; s < h.n_steps; ++s) {
          const int tau = h.tau0 + s * h.dtau;
          TcArgs c;
          c.C = h.C + (long long)tau * h.c_ts; c.ldc = h.ldc; c.beta = 1.f; c.split_k = 0;
          c.gate = h.gate + (long long)tau * h.gate_ts; c.ldgate = h.ldgate;
          c.Cb = (__nv_bfloat16*)h.Cb + (long long)tau * h.cb_ts; c.ldcb = h.ldcb;
          if ((rc = gemm_tc_bf16((const __nv_bfloat16*)h.Ab + (long long)(tau - h.dtau) * h.a_ts, h.lda, 0, h.W, H, 0, Bg, H, H, c,
                                 sk, sk_bytes, st)))
            return rc;
        }
      }
    }
  }
  if ((rc = layer2_wgrad_bf16(T, B, I, H, D, x, ldx, x_bf16, ldxb, n_steps, out_bf16, ldo, dout, lddo, dpre_bf16, dw, sk,
                              sk_bytes, 0, st)))
    return rc;
  if (dx) {   // dx (+)= dpre_d W_ih_d  (B operand = W_ih as stored [K = H][N = I]: MN-major)
    for (int d = 0; d < D; ++d) {
      const int n = n_steps[d], t_lo = d ? T - n : 0;
      TcArgs g;
      g.C = dx + (long long)t_lo * B * lddx; g.ldc = lddx; g.beta = d ? 1.f : 0.f; g.split_k = 1;
      if ((rc = gemm_tc_bf16(dpb + (long long)t_lo * B * lddo + (long long)d * H, lddo, 0, wih[d], Ip, 1, n * B, I, H, g, sk,
                             sk_bytes, st)))
        return rc;
    }
  }
  return 0;
}

int tacorl_rnn_layer_fwd(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                         const float* w_hh, const float* b_ih, const float* b_hh, const float* h0,
                         int reverse, int n_steps, float* out, long long ldo, const void* w_ih_bf16,
                         const void* w_hh_bf16, void* h_bf16_out, void* ws, size_t ws_bytes, int prec, void* stream) {
  TACORL_REQUIRE(prec == PREC_F32 || prec == PREC_BF16, "rnn_layer_fwd: unknown precision %d", prec);
  auto fn = prec == PREC_BF16 ? rnn_fwd_bf16 : rnn_fwd_f32;
  return fn(T, B, I, H, x, ldx, w_ih, w_hh, b_ih, b_hh, h0, reverse, n_steps, out, ldo, w_ih_bf16, w_hh_bf16, h_bf16_out,
            ws, ws_bytes, (cudaStream_t)stream);
}

int tacorl_rnn_layer_bwd(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                         const float* w_hh, const float* h0, int reverse, int n_steps, const float* out,
                         long long ldo, float* dout, long long lddo, const float* dhn, float* dx,
                         long long lddx, int dx_accumulate, float* dw_ih, float* dw_hh, float* db_ih,
                         float* db_hh, int accumulate, float* dh0, const void* w_ih_bf16, const void* w_hh_t_bf16,
                         const void* h_bf16, void* ws, size_t ws_bytes, int prec, void* stream) {
  TACORL_REQUIRE(prec == PREC_F32 || prec == PREC_BF16, "rnn_layer_bwd: unknown precision %d", prec);
  auto fn = prec == PREC_BF16 ? rnn_bwd_bf16 : rnn_bwd_f32;
  return fn(T, B, I, H, x, ldx, w_ih, w_hh, h0, reverse, n_steps, out, ldo, dout, lddo, dhn, dx, lddx,
            dx_accumulate, dw_ih, dw_hh, db_ih, db_hh, accumulate, dh0, w_ih_bf16, w_hh_t_bf16, h_bf16, ws, ws_bytes,
            (cudaStream_t)stream);
}

size_t tacorl_rnn_layer2_ws_bytes(int T, int B, int I, int H, int D) {
  return (size_t)D * tacorl_rnn_layer_ws_bytes(T, B, I, H) + 8192;
}

int tacorl_rnn_layer2_fwd(int T, int B, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                          long long ldxb, const float* const* w, const void* const* w_bf16, const int* n_steps,
                          float* out, long long ldo, void* out_bf16, void* ws, size_t ws_bytes, void* stream) {
  return layer2_fwd_bf16(T, B, I, H, D, x, ldx, x_bf16, ldxb, w, w_bf16, n_steps, out, ldo, out_bf16, ws, ws_bytes,
                         (cudaStream_t)stream);
}

int tacorl_rnn_layer2_bwd(int T, int B, int grad_rows, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                          long long ldxb, const float* const* w, const void* const* w_bf16, const int* n_steps,
                          const float* out, long long ldo, const void* out_bf16, float* dout, long long lddo,
                          void* dpre_bf16, float* dx, long long lddx, float* const* dw, void* ws, size_t ws_bytes,
                          void* stream) {
  return layer2_bwd_bf16(T, B, grad_rows, I, H, D, x, ldx, x_bf16, ldxb, w, w_bf16, n_steps, out, ldo, out_bf16, dout, lddo, dpre_bf16,
                         dx, lddx, dw, ws, ws_bytes, (cudaStream_t)stream);
}

int tacorl_rnn_layer2_wgrad(int T, int B, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                            long long ldxb, const int* n_steps, const void* out_bf16, long long ldo, const float* dout,
                            long long lddo, const void* dpre_bf16, float* const* dw, void* ws, size_t ws_bytes,
                            int max_ctas, void* stream) {
  TACORL_REQUIRE(x && n_steps && out_bf16 && dout && dpre_bf16 && dw && ws, "rnn_layer2_wgrad: null pointer");
  TACORL_REQUIRE(D == 1 || D == 2, "rnn_layer2_wgrad: D must be 1 or 2");
  TACORL_REQUIRE(H % 8 == 0 && ldo % 8 == 0 && lddo % 8 == 0 && ((uintptr_t)out_bf16 & 15) == 0 && ((uintptr_t)dpre_bf16 & 15) == 0,
                 "rnn_layer2_wgrad: pitches must be multiples of 8 and the bf16 twins 16-byte aligned");
  TACORL_REQUIRE(n_steps[0] == T, "rnn_layer2_wgrad: the forward direction must cover every step");
  TACORL_REQUIRE(max_ctas >= 0, "rnn_layer2_wgrad: max_ctas must be >= 0");
  for (int d = 0; d < D; ++d)
    TACORL_REQUIRE(n_steps[d] >= 1 && n_steps[d] <= T, "rnn_layer2_wgrad: n_steps out of range");
  if (B == 0) return 0;
  return layer2_wgrad_bf16(T, B, I, H, D, x, ldx, x_bf16, ldxb, n_steps, out_bf16, ldo, dout, lddo, dpre_bf16, dw, ws,
                           ws_bytes, max_ctas, (cudaStream_t)stream);
}

int tacorl_cast_transpose_bf16(const float* src, int rows, int cols, void* dst, void* stream) {
  TACORL_REQUIRE(src && dst, "cast_transpose_bf16: null pointer");
  return cast_transpose_bf16(src, cols, rows, cols, dst, rows, (cudaStream_t)stream);
}

}  // extern "C"
