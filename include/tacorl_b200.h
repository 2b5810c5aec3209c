/*
 * tacorl_b200 — C ABI of the B200-native (sm_100a) PlayLMP / TACO-RL training hot path.
 *
 * The reference (ErickRosete/tacorl) is pure Python over torch.nn; it has no FFI.  Its plug-in
 * boundary for this path is the Hydra `_target_` class paths + nn.Module method signatures
 * (SURVEY.md §8b).  The Python mirror of those classes lives in `tacorl_b200/networks`,
 * `tacorl_b200/modules`; every one of their tensor contractions / reductions calls one of the
 * entry points below through ctypes (tacorl_b200/_lib.py).  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - all pointers are DEVICE pointers to fp32 unless stated; no allocation happens inside: scratch
 *     comes from the caller's `ws` (size from the matching *_ws_bytes query);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return 0 on success, <0 on error with a message in tacorl_last_error() (thread-local);
 *   - random numbers are inputs (the host draws them with the reference's torch calls, in the
 *     reference's order — SURVEY.md Appendix C);
 *   - `prec`: TACORL_PREC_F32 = full-fp32 SIMT (parity path), TACORL_PREC_BF16 = bf16 tcgen05
 *     tensor-core operands with fp32 accumulation (performance path).
 *   - file:line citations are into /root/reference/src/tacorl/.
 */
#ifndef TACORL_B200_H_
#define TACORL_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TACORL_B200_ABI_VERSION 7

#define TACORL_PREC_F32 0
#define TACORL_PREC_BF16 1

#define TACORL_ACT_NONE 0
#define TACORL_ACT_RELU 1
#define TACORL_ACT_SILU 2

const char* tacorl_last_error(void);
int tacorl_abi_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py reports the delta) */
unsigned long long tacorl_launch_count(void);

/* Leave n SMs out of the grids of the persistent one-CTA-per-SM kernels (convolutions, weight gradients) so that a
 * concurrently running collective (NCCL all-reduce of the previous gradient slice) finds free SMs; returns the CTA count
 * those kernels now launch.  Default 0 (env TACORL_SM_RESERVE). */
int tacorl_set_sm_reserve(int n);

/* ---- dense layers -------------------------------------------------------------------------
 * C[M,N] = act(alpha * op(A)[M,K] op(B)[K,N] + beta * C + bias[N]); row-major with leading dims.
 * transA: A stored [K,M]; transB: B stored [N,K] (a torch Linear weight).  Cpre (optional) receives
 * the pre-activation.  Replaces every nn.Linear / F.linear on the path: encoder.py:398-403,
 * goal_encoder.py:18-24, actor.py:252-266, critic.py:92-97, action_decoder_logistic.py:289-293,
 * plan_recognition_tanh_net.py:44-45 — and the autograd GEMMs behind them. */
int tacorl_gemm(int transA, int transB, int M, int N, int K, float alpha, const float* A, long long lda,
                const float* B, long long ldb, float beta, float* C, long long ldc, const float* bias, int act,
                float* Cpre, long long ldpre, void* ws, size_t ws_bytes, int prec, void* stream);
/* Same, with optional dense bf16 copies of the operands as stored (A_bf16: rows x cols of A with pitch = cols, likewise
 * B_bf16).  PREC_BF16 uses them instead of staging a cast of the fp32 operand each call: the weights' copies are kept
 * current by tacorl_adam_step (shadow_bf16).  Ignored for PREC_F32 or when the pitch is not a multiple of 8. */
int tacorl_gemm_ex(int transA, int transB, int M, int N, int K, float alpha, const float* A, long long lda,
                   const float* B, long long ldb, float beta, float* C, long long ldc, const float* bias, int act,
                   float* Cpre, long long ldpre, const void* A_bf16, const void* B_bf16, void* ws, size_t ws_bytes,
                   int prec, void* stream);
/* out[n] (+)= sum_m X[m*ldx+n]  (bias gradients) */
int tacorl_colsum(int M, int N, const float* X, long long ldx, float* out, int accumulate, void* stream);
/* dZ = dY * act'(.)   relu: pass the post-activation, silu: pass the pre-activation */
int tacorl_act_bwd(int act, long long n, const float* dY, const float* y_or_pre, float* dZ, void* stream);
/* out = x * (*dev_scalar or 1) * c */
int tacorl_scale(long long n, const float* x, const float* dev_scalar, float c, float* out, void* stream);
/* out[r][c] (+)= x[r][c] * row_scalars[r] * k */
int tacorl_rowscale(long long rows, int L, const float* x, const float* row_scalars, float k, float* out,
                    int accumulate, void* stream);

/* ---- LMP vision encoder: encoder.py:369-419 (LMPVisionEncoder), utils.py:39-76 (SpatialSoftArgmax)
 * x: (N,3,H,W) NCHW; x_dtype 0 = fp32 (already normalised, the reference's batch contract) or 1 = uint8 raw frames
 * normalised on the fly as v = u8 * x_scale + x_shift (ScaleImageTensor + Normalize of utils/transforms.py:87-101 /
 * config rl_train.yaml:2-14 fused into the first load; SURVEY.md §8f row 1).  params/grads: 11 pointers in state_dict order
 *   model.0.{weight,bias}, model.2.{weight,bias}, model.4.{weight,bias}, model.6.temperature,
 *   fc_layers.0.{weight,bias}, fc_layers.3.{weight,bias}          (SURVEY.md Appendix B)
 * Saved for backward (caller-owned; pass NULL for y1,y2[,y3,feat,smax,ssum,h4] in inference):
 *   y1 (N,H1,W1,32), y2 (N,H2,W2,64) post-ReLU NHWC (fp32 for PREC_F32, bf16 for PREC_BF16),
 *   y3 (N,H3,W3,64) post-ReLU NHWC fp32; feat (N,128);
 *   smax, ssum (N,64) softmax statistics; h4 (N,hidden).   emb: (N,latent).
 *   xs (PREC_BF16 only, optional): the (N,H1+1,W1+1,64) bf16 space-to-depth copy of the normalised image that conv1
 *   consumes; when the forward call stores it and the backward call receives it, the backward pass does not touch x. */
size_t tacorl_lmp_encoder_ws_bytes(int N, int H, int W, int hidden, int latent, int backward);
int tacorl_lmp_encoder_fwd(const void* x, int x_dtype, float x_scale, float x_shift, int N, int H, int W,
                           const float* const* params, int hidden,
                           int latent, float* y1, float* y2, float* y3, float* feat, float* smax,
                           float* ssum, float* h4, float* emb, void* xs, void* ws, size_t ws_bytes, int prec,
                           void* stream);
int tacorl_lmp_encoder_bwd(const void* x, int x_dtype, float x_scale, float x_shift, int N, int H, int W,
                           const float* const* params, int hidden,
                           int latent, const float* y1, const float* y2, const float* y3,
                           const float* feat, const float* smax, const float* ssum, const float* h4,
                           const float* d_emb, float* const* grads, int accumulate, const void* xs, void* ws,
                           size_t ws_bytes, int prec, void* stream);

/* Diagnostic hook for the implicit-GEMM convolution kernels behind tacorl_lmp_encoder_* (PREC_BF16):
 * runs ONE op on fp32 NHWC inputs staged to bf16.  op 1/2/3: conv1/2/3 forward (in0 = image NCHW | y1 | y2);
 * 4/5: conv3/conv2 data gradient (in0 = dY, in1 = saved activation gating the result);
 * 6/7/8: conv3/conv2/conv1 weight gradient (in0 = dY, in1 = y2 | y1 | image) -> torch (oc,c,ky,kx) layout.
 * H, W are the IMAGE dims the layer geometry derives from (encoder.py:369-390). */
int tacorl_conv_tc_debug(int op, const float* in0, const float* in1, const float* Wt, const float* bias, int N,
                         int H, int W, float* out, void* ws, size_t ws_bytes, void* stream);

/* Diagnostic hook for the bf16 tcgen05 GEMM family behind tacorl_gemm* (PREC_BF16): runs the run-time dispatch on bf16
 * operands already on the device, with no 2^24-multiply-add fp32 cut-off.  A: a_mn ? stored [K][M] : [M][K] (pitch lda),
 * B: b_mn ? stored [K][N] : [N][K] (pitch ldb), both 16-byte aligned with 16-byte multiple pitches.  Epilogue per output
 * element: pre = alpha * A.B + beta * C + bias -> Cpre; act; 0 where gate <= 0; -> C (may be NULL) and bf16 Cb (may be
 * NULL).  split_k: 0 = automatic, else the K splits asked for (cut down to what ws holds).  ws: split-K partials.
 * route (host int[4]): {0 = tiled kernel, 1 = skinny cluster kernel; tiled BN or skinny NT; z-slices (tiled: K splits
 * used, skinny: K slabs per cluster); CTAs launched}. */
int tacorl_gemm_tc_debug(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, int M, int N,
                         int K, float alpha, float beta, float* C, long long ldc, void* Cb, long long ldcb,
                         const float* bias, int act, float* Cpre, long long ldpre, int split_k, const float* gate,
                         long long ldgate, void* ws, size_t ws_bytes, int* route, void* stream);

/* ---- ReLU RNN layer, one direction, time-major (T*B rows): nn.RNN(nonlinearity="relu") at
 * rnn_models.py:5-16 (decoder) and plan_recognition_tanh_net.py:23-31 / plan_recognition_net.py:27-35
 * (BiRNN).  h0 may be NULL (zeros).  reverse: recurrence runs t = T-1 .. T-n_steps.
 * bwd: `dout` (dL/dout) is overwritten with dL/dpre; dx rows outside the active range are zeroed
 * unless dx_accumulate.  Any of dx/dw_ih/dw_hh/db_ih/db_hh/dh0/dhn may be NULL. */
size_t tacorl_rnn_layer_ws_bytes(int T, int B, int I, int H);
/* bf16 path: steps 1..n_steps-1 of a layer run in ONE persistent launch (weights resident in shared memory, steps
 * chained by device-side arrival counters); set TACORL_RNN_SEQ=0 to launch step by step instead (bit-identical
 * results).  A persistent launch occupies 120 of the 148 SMs and spin-waits on its peer clusters; the library chains
 * such launches through an event so that two of them never run concurrently, whatever streams they are on.  Returns how many spin-waits ever gave up (0 in a healthy process;
 * synchronises the device). */
unsigned tacorl_rnn_seq_timeouts(void);
/* persistent launches at run time: 0 = off (step-by-step launches), 1 = on, 2 = on with the two lanes of a
 * bidirectional layer launched one after the other (diagnostic: bit-identical to 1); returns the previous setting */
int tacorl_rnn_seq_enable(int on);
/* bf16 path, optional (NULL = stage internally): w_*_bf16 dense bf16 copies of the weights (tacorl_adam_step keeps
 * them current); h_bf16_out: (T, B, H) bf16 buffer that receives the hidden states the tensor cores consumed — hand
 * it back to the backward call as h_bf16 and BPTT skips re-casting the saved fp32 activations; w_hh_t_bf16: W_hh^T
 * as bf16 (tacorl_cast_transpose_bf16), which the caller can prepare off the critical path. */
int tacorl_rnn_layer_fwd(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                         const float* w_hh, const float* b_ih, const float* b_hh, const float* h0,
                         int reverse, int n_steps, float* out, long long ldo, const void* w_ih_bf16,
                         const void* w_hh_bf16, void* h_bf16_out, void* ws, size_t ws_bytes, int prec, void* stream);
int tacorl_rnn_layer_bwd(int T, int B, int I, int H, const float* x, long long ldx, const float* w_ih,
                         const float* w_hh, const float* h0, int reverse, int n_steps, const float* out,
                         long long ldo, float* dout, long long lddo, const float* dhn, float* dx,
                         long long lddx, int dx_accumulate, float* dw_ih, float* dw_hh, float* db_ih,
                         float* db_hh, int accumulate, float* dh0, const void* w_ih_bf16, const void* w_hh_t_bf16,
                         const void* h_bf16, void* ws, size_t ws_bytes, int prec, void* stream);
/* ---- a whole (bi)directional layer in one call, bf16 tensor-core path (replaces nn.RNN's per-layer work at
 * plan_recognition_tanh_net.py:23-46 (bidirectional, D = 2) and rnn_models.py:5-16 (decoder, D = 1), h_init = 0).
 * The recurrences of the two directions run side by side in ONE persistent launch (rnn_wave_kernel: 4-CTA clusters split
 * K, 64 CTAs per direction, weights resident in shared memory, steps chained by device-side arrival counters; batch
 * <= 64; larger batches use the 8-way kernel above or per-step launches).  Layouts: out / dout fp32 (T, B, D*H),
 * direction d owns columns [d*H, (d+1)*H); out_bf16 / dpre_bf16 are bf16 twins in the SAME layout, written by the
 * recurrence kernels: the next layer's input projection (x_bf16 of the next call), BPTT and the weight-gradient GEMMs
 * read them in place, so no staging cast is launched.
 *   w      : fwd [4*D] = w_ih, w_hh, b_ih, b_hh of the forward direction, then of the reverse one;
 *            bwd [2*D] = w_ih, w_hh per direction.
 *   w_bf16 : [2*D] per direction: bf16 twin of w_ih, and of w_hh (fwd) / of W_hh^T (bwd); entries may be NULL.
 *   n_steps: [D] steps each direction runs (reverse: t = T-1 .. T-n); bwd needs n_steps[0] == T.
 *   dw     : [4*D] dw_ih, dw_hh, db_ih, db_hh per direction (entries may be NULL); dx: (T, B, I) or NULL.
 *   grad_rows: 0 or B = every batch row; 0 < grad_rows < B: only the first grad_rows rows of each time step carry a
 *            gradient (rows behind them in dout AND dpre_bf16 must be zero on entry): BPTT runs on those rows alone. */
size_t tacorl_rnn_layer2_ws_bytes(int T, int B, int I, int H, int D);
int tacorl_rnn_layer2_fwd(int T, int B, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                          long long ldxb, const float* const* w, const void* const* w_bf16, const int* n_steps,
                          float* out, long long ldo, void* out_bf16, void* ws, size_t ws_bytes, void* stream);
int tacorl_rnn_layer2_bwd(int T, int B, int grad_rows, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                          long long ldxb, const float* const* w, const void* const* w_bf16, const int* n_steps,
                          const float* out, long long ldo, const void* out_bf16, float* dout, long long lddo,
                          void* dpre_bf16, float* dx, long long lddx, float* const* dw, void* ws, size_t ws_bytes,
                          void* stream);
/* The weight-gradient half of tacorl_rnn_layer2_bwd (dW_hh, dW_ih and the bias sums into dw), for a call of it made with
 * every dw entry NULL once that call's recurrence has finished: dout / dpre_bf16 hold dpre.  Nothing on the dependent
 * chain reads these gradients, so this may run on a second stream beside the next layer's backward, with its own
 * workspace (tacorl_rnn_layer2_ws_bytes) and max_ctas > 0 capping the GEMMs' persistent grids to the SMs the
 * concurrent recurrence leaves free (148 - 64 per lane); 0 = every SM.  The results do not depend on max_ctas. */
int tacorl_rnn_layer2_wgrad(int T, int B, int I, int H, int D, const float* x, long long ldx, const void* x_bf16,
                            long long ldxb, const int* n_steps, const void* out_bf16, long long ldo, const float* dout,
                            long long lddo, const void* dpre_bf16, float* const* dw, void* ws, size_t ws_bytes,
                            int max_ctas, void* stream);
/* dst (cols x rows, bf16, dense) = transpose of src (rows x cols, fp32, dense) */
int tacorl_cast_transpose_bf16(const float* src, int rows, int cols, void* dst, void* stream);

/* ---- action decoder losses: action_decoder_logistic.py:184-235 (_logistic_loss), :114-133 (_loss),
 * :238-266 (_sample).  logits row = [prob A*10 | mean A*10 | log_scale A*10 | gripper 2].
 * dlm_nll writes the mean loss to loss_out[0], per-term losses to row_loss (rows*(A+1)) and, if
 * dlogits != NULL, dLoss/dlogits.  dlm_sample: u1 (rows,A,10), u2 (rows,A) ~ U[0,1); pred (rows,A+1);
 * hit/acc_out optional gripper accuracy (play_lmp_for_rl.py:165-176). */
int tacorl_dlm_nll(int rows, int act_dims, const float* logits, long long ld, const float* actions,
                   long long lda, int num_classes, float act_min, float act_max, float gripper_alpha,
                   float* row_loss, float* loss_out, float* dlogits, long long ldd, void* stream);
int tacorl_dlm_sample(int rows, int act_dims, const float* logits, long long ld, const float* u1,
                      const float* u2, const float* actions, long long lda, float grip_lo, float grip_hi,
                      float* pred, float* hit, float* acc_out, void* stream);

/* ---- distribution heads.  raw: (rows, 2L) = [mean | log_std or var].
 * gauss_head: actor.py:259-266 (clamp +-9, exp(clamp(-5,2)));
 * softplus_head: plan_recognition_tanh_net.py:44-46 (softplus + min_std). */
int tacorl_gauss_head_fwd(int rows, int L, const float* raw, float* mean, float* stdv, void* stream);
int tacorl_gauss_head_bwd(int rows, int L, const float* raw, const float* stdv, const float* dmean,
                          const float* dstd, float* draw, void* stream);
int tacorl_softplus_head_fwd(int rows, int L, const float* raw, float min_std, float* mean, float* stdv,
                             void* stream);
int tacorl_softplus_head_bwd(int rows, int L, const float* raw, const float* dmean, const float* dstd,
                             float* draw, void* stream);
/* ---- discrete open/close gripper head of the flat-CQL baseline: GumbelSoftmax of utils/distributions.py:15-58 as used
 * by Actor.get_actions / sample_n_with_log_prob / log_prob (actor.py:66-156).  logits: (rows0, 2); u: (rows, 2) uniforms
 * (row r reads logits row r % rows0: the n sampled copies of sample_n share the logits); index: class id 0 / 1 as float,
 * action = 2 * index - 1.  clamp_u = 1: the rsample path (torch clamp_probs), 0: GumbelSoftmax.sample. */
int tacorl_gripper_gumbel(int rows, int rows0, const float* logits, const float* u, int clamp_u, float* index,
                          float* action, void* stream);
/* logp[r] = log_softmax(logits[r % rows0])[index[r]]  (GumbelSoftmax.log_prob of a class index, :50-58) */
int tacorl_gripper_logprob(int rows, int rows0, const float* logits, const float* index, float* logp, void* stream);
int tacorl_gripper_logprob_bwd(int rows, const float* logits, const float* index, const float* dlogp, float* dlogits,
                               void* stream);
/* balanced KL of the underlying Normals, play_lmp_for_rl.py:259-285; grads are d kl / d(.) */
int tacorl_kl_balanced(int B, int L, const float* mu_q, const float* sd_q, const float* mu_p,
                       const float* sd_p, float kl_alpha, int balancing, float* kl_out, float* dmu_q,
                       float* dsd_q, float* dmu_p, float* dsd_p, void* stream);
/* TanhNormal, utils/distributions.py:61-153.  rsample: a = tanh(mu + std*eps) (mu/std broadcast with
 * period `bcast` elements for sample_n); logprob: (rows) with optional gradient outputs. */
int tacorl_tanh_rsample_fwd(long long n, long long bcast, const float* mu, const float* sd, const float* eps,
                            float* a, float* z, int apply_tanh, void* stream);
int tacorl_tanh_rsample_bwd(long long n, const float* a, const float* eps, const float* da, const float* dz,
                            float* dmu, float* dsd, int apply_tanh, void* stream);
int tacorl_tanh_logprob(int rows, int L, int bcast_rows, const float* mu, const float* sd, const float* z,
                        int from_value, float* logp, float* gmu, float* gsd, float* gz, void* stream);

/* ---- transformer plan recogniser pieces: plan_recognition_transformer.py:70-105 (+ torch's
 * nn.TransformerEncoderLayer: post-norm, ReLU, eps 1e-5, (T,B,D) layout).  Linear layers use tacorl_gemm.
 * Dropout masks are pre-scaled keep masks (or NULL).  attn: T <= 32, head_dim <= 16; qkv (T,B,3D) = [q|k|v],
 * P (B*heads,T,T) = saved softmax.  add_ln: y = LayerNorm(x + r*mask); bwd ACCUMULATES dw/db (zero them first). */
int tacorl_posemb_fwd(int B, int T, int D0, int D, const float* emb, const float* pos, const float* mask, float* x,
                      void* stream);
int tacorl_posemb_bwd(int B, int T, int D0, int D, const float* dx, const float* mask, float* demb, float* dpos,
                      void* stream);
int tacorl_attn_fwd(int B, int T, int D, int heads, const float* qkv, const float* amask, float* P, float* out,
                    void* stream);
int tacorl_attn_bwd(int B, int T, int D, int heads, const float* qkv, const float* amask, const float* P,
                    const float* dout, float* dqkv, void* stream);
int tacorl_add_ln_fwd(int rows, int D, const float* x, const float* r, const float* mask, const float* w,
                      const float* b, float eps, float* y, float* xhat, float* rstd, void* stream);
int tacorl_add_ln_bwd(int rows, int D, const float* dy, const float* xhat, const float* rstd, const float* w,
                      const float* mask, float* dx, float* dr, float* dw, float* db, void* stream);
int tacorl_mean_t_fwd(int B, int T, int C, const float* x, float* y, void* stream);
int tacorl_mean_t_bwd(int B, int T, int C, const float* dy, float* dx, void* stream);
int tacorl_mul(long long n, const float* a, const float* b, float* out, void* stream);

/* ---- CQL losses, cql_offline_lightning.py:284-406, 439-468.
 * q*_all: [data (B) | rand (n,B) | curr (n,B) | next (n,B)].  scalars[14]:
 *  0 bellman_q1, 1 bellman_q2, 2 conservative_q1, 3 conservative_q2, 4 alpha_prime, 5 alpha_prime_loss,
 *  6 q1_loss, 7 q2_loss, 8 q1_data, 9 q1_random, 10 q1_policy, 11 q2_data, 12 q2_random, 13 q2_policy */
#define TACORL_CQL_NUM_SCALARS 14
int tacorl_cql_critic_loss(int B, int n, const float* q1_all, const float* q2_all, const float* lp_curr,
                           const float* lp_next, const float* tq1, const float* tq2, const float* reward,
                           const float* done, const float* log_alpha_prime, float rand_density, float discount,
                           float reward_scale, float gap, float conservative_weight, float temp,
                           int with_lagrange, float* scalars, float* dq1_all, float* dq2_all,
                           float* d_log_alpha_prime, void* stream);
/* mode 0: alpha loss; 1: actor loss, BC epochs (a = log-prob of data action);
 * 2: actor loss, Q epochs (a,b = Q1,Q2 at the policy action).  out[0]=loss, out[1]=alpha (modes 1,2) */
int tacorl_cql_actor_loss(int mode, int B, const float* log_pi, const float* a, const float* b,
                          const float* log_alpha, float target_entropy, float* out, float* d_log_alpha,
                          float* d_log_pi, float* da, float* db, void* stream);

/* ---- data-parallel gradient exchange (SURVEY 8(b): dp_allreduce_{init,enqueue,wait}); replaces Lightning's DDP over
 * gloo (config/trainer/default.yaml:1-4, scripts/train.py:73-75).  One communicator per process (one process per GPU).
 * unique_id: rank 0 fills 128 bytes that the host broadcasts to the other ranks by any means; init: every rank.
 * enqueue: in-place sum over the ranks of buf[0..n) (dtype 0 = fp32, 1 = bf16), ordered after everything queued on
 * `stream`, executed on the library's own communication stream (returns at once; capturable in a CUDA graph);
 * wait: `stream` waits for every exchange enqueued so far.  NCCL is dlopen()ed (TACORL_NCCL_LIB overrides the path). */
int tacorl_dp_unique_id(void* id128);
int tacorl_dp_allreduce_init(const void* id128, int rank, int world);
int tacorl_dp_allreduce_enqueue(void* buf, long long n, int dtype, void* stream);
int tacorl_dp_allreduce_wait(void* stream);
int tacorl_dp_allreduce_destroy(void);

/* ---- device-side input pipeline (SURVEY 8f-1): the per-sample work of the reference's DataLoader workers on uint8
 * frames resident in HBM.  Random quantities are inputs (drawn by the host in the reference's order).
 * window_gather_u8: out[b][t] = store[start[b] + min(t, window[b]-1)] (pad_sequence by repetition,
 *   play_dataset.py:282-330), each frame shifted by (shift[b][t] - pad) pixels with edge clamping = RandomShiftsAug
 *   (utils/transforms.py:265-299: replicate-pad by `pad`, integer shift in [0, 2 pad]); shift NULL = no augmentation.
 * actions_gather_pad: same windows over a (frames, A) fp32 store; zero_pad = 1: steps past the window are zero except
 *   the last channel, which repeats (the "rel" action modalities, play_dataset.py:291-301).
 * color_jitter_u8: ScaleImageTensor (u8/255) -> torchvision ColorJitter ops in the per-frame order `order` (three op
 *   ids packed 4 bits each, first op lowest: 0 brightness, 1 contrast, 3 hue, 0xF none) with per-frame factors
 *   (brightness, contrast, hue) -> Normalize(mean, std): utils/transforms.py:87-101, 302-330.  order NULL = no jitter.
 *   mean_ws: N floats of scratch. */
int tacorl_window_gather_u8(const unsigned char* store, long long frames, int C, int H, int W, const int* start,
                            const int* window, const int* shift, int pad, int B, int T, unsigned char* out, void* stream);
int tacorl_actions_gather_pad(const float* store, long long frames, int A, const int* start, const int* window, int B,
                              int T, int zero_pad, float* out, void* stream);
int tacorl_color_jitter_u8(const unsigned char* x, long long N, int H, int W, const int* order, const float* factors,
                           float norm_mean, float norm_std, float* mean_ws, float* out, void* stream);

/* ---- HBM-resident replay (tacorl_b200/replay.py; sampling rules: DESIGN.md section 13).  A step's batch is drawn and
 * assembled on the device by two graph-capturable launches; nothing is allocated and nothing crosses PCIe.
 * replay_sample: ONE CTA.  Reads *step_dev, draws with Philox4x32-10 (key = (lo32(seed), hi32(seed) ^ rank * 0x9E3779B9),
 *   counter = (lo32(step), hi32(step), sample, draw id)), writes the tables and stores *step_dev + 1.
 *   kind 0 PlayLMP, 1 TACO-RL, 2 flat CQL.  valid: start frames (kinds 0/1: >= min_window frames left in the episode;
 *   kind 2: frames with a successor in their episode), n_valid entries.  geom_thr: n_geom non-decreasing thresholds of
 *   Geometric(p) on {1, 2, ...}: thr[k] = floor(2^32 P(d <= k + 1)).  neg_thr: TACO-RL negative goal iff u < neg_thr.
 *   tab  (4, B) int32: start | window | goal | disp  (kind 2: frame i | 1 | goal | reward);
 *   out64 (3, B) int64: idx | window_size | disp     (kind 2: rewards | terminals | goal);
 *   shift (n_mod, B, n_slots, 2) int32 in [0, 2 pad], or NULL for no RandomShiftsAug.
 *   jitter (optional, NULL = none): ColorJitter of every output frame: jit_order (n_mod, B, n_slots) int32 packed op
 *   order as tacorl_color_jitter_u8 takes it (a uniform order of the ops enabled in jitter->ops, bit 0 brightness,
 *   1 contrast, 3 hue), jit_factors (n_mod, B, n_slots, 3) fp32 = lo[i] + span[i] * (u >> 8) * 2^-24 per enabled op
 *   (1, 1, 0 for disabled ones).  Negative goal iff u < neg_thr (neg_thr = 2^32: always).
 *   Every index table must hold only in-range frame ids: the host validates them before upload.
 * replay_gather: ONE launch for every image output of the batch plus the action rows.  images[i].out is
 *   (B, T, 3, H, W) for TACORL_REPLAY_WINDOW (pad_sequence by repetition), else (B, 3, H, W) with the frame
 *   start (OBS), start + 1 (NEXT) or goal (GOAL) of `tab`; each frame is shifted by its slot shift_slot (+ t) of the
 *   modality's shift table (NULL = none), like tacorl_window_gather_u8.
 * replay_color_jitter: ScaleImageTensor -> ColorJitter -> Normalize of B x nf uint8 frames (the uint8 output of a
 *   gather) into fp32, frame (b, t) taking entry b * n_slots + slot0 + t of the sampler's jitter tables of its modality.
 *   mean_ws: B * nf floats.  Two launches (contrast mean, apply), the kernels of tacorl_color_jitter_u8.  act_out: (B, T, A) rows of act_store windowed
 *   like tacorl_actions_gather_pad (act_role WINDOW) or (B, A) (act_role OBS); NULL = no actions. */
#define TACORL_REPLAY_MAX_IMAGES 8
#define TACORL_REPLAY_WINDOW 0
#define TACORL_REPLAY_OBS 1
#define TACORL_REPLAY_NEXT 2
#define TACORL_REPLAY_GOAL 3
typedef struct tacorl_replay_image {
  const unsigned char* store;   /* (frames, 3, H, W) uint8 */
  unsigned char* out;
  const int* shift;             /* (B, n_slots, 2) shift table of this modality, or NULL */
  int H; int W;                 /* W % 4 == 0 */
  int role;                     /* TACORL_REPLAY_* */
  int shift_slot; int n_slots;
} tacorl_replay_image;
typedef struct tacorl_replay_jitter {
  int ops;                      /* bit 0 brightness, bit 1 contrast, bit 3 hue */
  float lo[3]; float span[3];   /* factor ranges of brightness, contrast, hue */
} tacorl_replay_jitter;
int tacorl_replay_sample(int kind, int B, int min_window, int max_window, int n_mod, int n_slots, int pad,
                         unsigned long long neg_thr, unsigned long long seed, int rank, long long* step_dev,
                         const int* ep_end, long long frames, const int* valid, long long n_valid,
                         const unsigned* geom_thr, int n_geom, int* tab, int* shift, long long* out64,
                         const tacorl_replay_jitter* jitter, int* jit_order, float* jit_factors, void* stream);
int tacorl_replay_gather(int B, int T, int pad, const int* tab, int n_images, const tacorl_replay_image* images,
                         const float* act_store, int A, int act_role, int zero_pad, float* act_out, void* stream);
int tacorl_replay_color_jitter(const unsigned char* x, int B, int nf, int H, int W, const int* order,
                               const float* factors, int n_slots, int slot0, float norm_mean, float norm_std,
                               float* mean_ws, float* out, void* stream);

/* ---- validation sweeps of an HBM-resident split (tacorl_b200/replay.py mode="sweep"; rules: DESIGN.md section 14).
 * replay_sweep: replay_sample's kernel in sweep mode.  *cursor_dev is an item cursor: row b < n of the B-row tables
 *   takes item i = (cursor + b) mod n_valid, start valid[i], and draws its window / goal / disp / CQL goal with the laws
 *   of replay_sample from counter (lo32(i), hi32(i), 0, draw id); then *cursor_dev += n.  No shift and no jitter.
 * replay_gather_rows: replay_gather over rows [0, n) of the B-row tables (images[i].out and act_out: prefixes of the
 *   B-row buffers).  replay_gather is replay_gather_rows with n = B.
 * metrics_accumulate: ONE launch, one thread per slot: acc[i] += n * (double)*value[i] for i < k, acc[k] += n.
 *   The struct travels by value, so a call needs no host-to-device copy. */
#define TACORL_METRICS_MAX 32
typedef struct tacorl_metrics {
  const float* value[TACORL_METRICS_MAX];   /* device fp32 scalars */
  int k;                                    /* number of metrics */
  int n;                                    /* items of the batch */
} tacorl_metrics;
int tacorl_replay_sweep(int kind, int B, int n, int min_window, int max_window, unsigned long long neg_thr,
                        unsigned long long seed, int rank, long long* cursor_dev, const int* ep_end, long long frames,
                        const int* valid, long long n_valid, const unsigned* geom_thr, int n_geom, int* tab,
                        long long* out64, void* stream);
int tacorl_replay_gather_rows(int B, int n, int T, int pad, const int* tab, int n_images,
                              const tacorl_replay_image* images, const float* act_store, int A, int act_role,
                              int zero_pad, float* act_out, void* stream);
int tacorl_metrics_accumulate(const tacorl_metrics* m, double* acc, void* stream);

/* ---- per-step training metrics (tacorl_b200/runtime.py TrainMetricsRecorder; DESIGN.md section 15).
 * metrics_record: ONE launch, one CTA of 32 threads, graph-capturable.  slot = *step_dev % ring_rows; thread i writes
 *   *value[i] to ring[slot * 32 + i] and adds it to the fp64 sum acc[i] and 1 to the count acc[32 + i].  A NULL
 *   value[i] (a key not logged in this mode) and every slot i >= k write NaN to the ring and leave acc alone.  Then
 *   *step_dev += 1.  m->n is not read.  ring: ring_rows x 32 fp32; acc: 64 fp64. */
int tacorl_metrics_record(const tacorl_metrics* m, float* ring, int ring_rows, long long* step_dev, double* acc,
                          void* stream);

/* ---- fused small-MLP chains (fp32): a whole Linear -> act -> Linear ... stack in ONE launch, forward or backward.
 * Replaces the per-layer launches behind VisualGoalEncoder.forward (goal_encoder.py:29-33), MLPPolicy.forward
 * (actor.py:252-270: 3 x Linear+SiLU, then fc_mean | fc_log_std as ONE layer of two weight segments) and
 * MLPQNetwork.forward (critic.py:92-97).  <= 4 layers, widths <= 256 and multiples of 4 (the last layer's output width
 * is free), the last layer has no activation.  The input may be the concatenation of two tensors along the feature
 * dim (state | goal, embedding | action): no torch.cat.  z: (rows, sum of the hidden widths) receives the
 * pre-activations of layers 0 .. L-2 (the backward pass's saved tensors).  bwd: dW / db per segment may be NULL
 * (gradient w.r.t. the input only); dx0 / dx1 may be NULL. */
/* OR-ed into tacorl_mlp_layer.act of a ReLU layer: z receives relu(z) instead of the pre-activation (the backward pass
 * reads the same buffer: relu'(z) and relu(z) are the same functions of either; LMPVisionEncoder's saved h4) */
#define TACORL_MLP_SAVE_ACTIVATED 0x100
typedef struct tacorl_mlp_layer {
  const float* W0; const float* b0; int n0;     /* first weight segment: (n0, in) row-major, bias (n0) or NULL */
  const float* W1; const float* b1; int n1;     /* optional second segment stacked behind it (n1 = 0: none) */
  const float* W2; const float* b2; int n2;     /* optional third segment (n2 = 0: none; needs n1 > 0):
                                                 * fc_mean | fc_log_std | gripper_action of a discrete-gripper MLPPolicy */
  int in; int act;                              /* input width; activation on the output (TACORL_ACT_*) */
  float* dW0; float* db0; float* dW1; float* db1; float* dW2; float* db2;   /* backward outputs */
} tacorl_mlp_layer;
size_t tacorl_mlp_chain_ws_bytes(int L, int rows, const tacorl_mlp_layer* layers);
int tacorl_mlp_chain_fwd(int L, int rows, const tacorl_mlp_layer* layers, const float* x0, int xin0, long long ldx0,
                         const float* x1, int xin1, long long ldx1, float* z, long long ldz, float* out, long long ldo,
                         void* stream);
int tacorl_mlp_chain_bwd(int L, int rows, const tacorl_mlp_layer* layers, const float* x0, int xin0, long long ldx0,
                         const float* x1, int xin1, long long ldx1, const float* z, long long ldz, const float* d_out,
                         long long lddo, float* dx0, long long lddx0, float* dx1, long long lddx1, void* ws,
                         size_t ws_bytes, void* stream);

/* ---- optimiser side: Adam (play_lmp_for_rl.py:362-368, cql_offline_lightning.py:553-574) fused with
 * clip_grad_norm_ (:522-537) over flat buffers; Polyak (:229-232); sum of squares (ws >= 592 floats) */
/* step: host-side step count (>=1) used for the bias corrections, OR step_dev != NULL: a device int that the
 * call increments and reads (so a captured CUDA graph replays with the right bias correction). */
int tacorl_adam_step(long long n, float* p, const float* g, float* m, float* v, float lr, float beta1,
                     float beta2, float eps, int step, int* step_dev, float grad_scale, const float* sqnorm,
                     float max_norm, void* shadow_bf16, void* stream);
/* One optimiser step applied slice by slice (a slice whose gradient is final early -- everything behind the vision
 * encoders -- is updated on a side stream while the encoder backward still runs): every slice of the step reads the same
 * device step count; only the FIRST call of a step passes increment_step = 1.  background = 1: launch a small grid
 * (one CTA per SM) that shares the SMs with whatever else is running instead of filling them. */
int tacorl_adam_step_range(long long n, float* p, const float* g, float* m, float* v, float lr, float beta1,
                           float beta2, float eps, int step, int* step_dev, int increment_step, int background,
                           float grad_scale, const float* sqnorm, float max_norm, void* shadow_bf16, void* stream);

/* ---- batched rollout: one control step of ActionDecoderLogistic.act (action_decoder_logistic.py:116-122) for n
 * independent environments, 1 <= n <= 64 (tacorl_b200/rollout.py, DESIGN.md section 16).  Three graph-capturable
 * launches (layer 0, layer 1, heads + sample); no allocation, no host synchronisation.
 *   plan (n, P), emb (n, E): the decoder input [plan | emb], fp32, P and E multiples of 4;
 *   hidden (2, n, H): the recurrent state, read and updated in place; H a multiple of 8;
 *   restart (n) int32: a non-zero row starts from h = 0 (clear_hidden_state()); the call does not clear it;
 *   w: 16 fp32 tensors, rnn.{weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0, weight_ih_l1, weight_hh_l1, bias_ih_l1,
 *      bias_hh_l1}, {prob_fc, mean_fc, log_scale_fc, gripper_fc}.{weight, bias}, 16-byte aligned;
 *   w_bf16: NULL or 8 bf16 operand copies (entries may be NULL) of weight_ih_l0, weight_hh_l0, weight_ih_l1,
 *      weight_hh_l1, prob_fc, mean_fc, log_scale_fc, gripper_fc weights; PREC_BF16 reads them instead of rounding the
 *      fp32 weights itself (the same values);
 *   noise: counter-based Philox4x32-10 with key (lo32(seed), hi32(seed)); row r's uniform i < 66 is word i mod 4 of
 *      the draw with counter (lo32(t[r]), hi32(t[r]), env_id[r], i div 4), as (w >> 8) 2^-24; i < 60 is u1[i / 10][i %
 *      10], i >= 60 is u2[i - 60]; then tacorl_dlm_sample's transforms.  t (n) int64 is incremented by the call;
 *   actions (n, 7); logits: NULL or (n, 182) [prob 60 | mean 60 | log_scale 60 | gripper 2];
 *   ws: tacorl_rollout_ws_bytes(n, H) bytes, ZERO-FILLED before its first use (it holds a completion counter that
 *      every call leaves at zero).  Calls that share a ws must be stream-ordered.
 *   prec: PREC_F32 = fp32 FFMA; PREC_BF16 = operands rounded to bf16 (nearest even), fp32 accumulation.
 * Every output element is reduced in an order that depends neither on n nor on the other rows: a row's hidden state,
 * logits and action are bit-identical whether it runs alone or in a batch. */
size_t tacorl_rollout_ws_bytes(int n, int H);
int tacorl_rollout_decoder_step(int n, int P, int E, int H, const float* plan, const float* emb, float* hidden,
                                const int* restart, const float* const* w, const void* const* w_bf16,
                                unsigned long long seed, const int* env_id, long long* t, float grip_lo, float grip_hi,
                                float* actions, float* logits, void* ws, size_t ws_bytes, int prec, void* stream);
/* ---- the rollout policy's own sampling (sampled latent plans, the flat-CQL actor), one graph-capturable launch for n
 * rows, 1 <= n <= 64; fp32 arithmetic in both precision modes.  mean, std (n, A): ops.gauss_head's output; grip_logits:
 * NULL or (n, 2); mask: NULL or (n) int32, rows whose mask is 0 are not written.  Draw j of row r is the Philox4x32-10
 * block with key (lo32(seed), hi32(seed)) and counter (lo32(t[r]), hi32(t[r]), env_id[r], j); its words 0 and 1 give
 * u_a = (w0 >> 8) 2^-24 and u_b = (w1 >> 8) 2^-24.  Dimension d < A uses draw 32 + d:
 * out[r][d] = tanh(mean + std sqrt(-2 ln(1 - u_a)) cos(2 pi u_b)).  The gripper uses draw 32 + A:
 * out[r][A] = 2 argmax_c(normalised logit_c - log(-log(u_c))) - 1 with u_0 = u_a, u_1 = u_b (ties -> class 0).
 * (Draws 0..16 are tacorl_rollout_decoder_step's.)  advance_t = 1: every row's t is incremented after sampling.
 * out has row stride ldo floats.  Each row is computed on its own: bit-identical alone or among 64 rows. */
int tacorl_rollout_policy_sample(int n, int A, const float* mean, const float* std, const float* grip_logits,
                                 const int* mask, unsigned long long seed, const int* env_id, long long* t, int advance_t,
                                 float* out, long long ldo, void* stream);
int tacorl_polyak_update(long long n, float* target, const float* source, float tau, void* stream);
int tacorl_sqnorm(long long n, const float* x, float* out, float* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TACORL_B200_H_ */
