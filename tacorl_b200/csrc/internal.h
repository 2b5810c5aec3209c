// Internal (non-ABI) declarations shared between the .cu translation units.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace tacorl {

const char* last_error();
unsigned long long launch_count();

int colsum_tall_f32(long long M, int N, const float* X, float* out, int accumulate, float* ws,
                    size_t ws_bytes, cudaStream_t st);

int im2col_f32(const float* x, long long sn, long long sc, long long sh, long long sw, int C, int KH,
               int KW, int stride, int OH, int OW, int nframes, float* col, cudaStream_t st, int korder);
int colsum_tall_bf16(long long M, int N, const void* X, float* out, int accumulate, float* ws, size_t ws_bytes,
                     cudaStream_t st);
int col2im_f32(const float* dcol, int C, int H, int W, int KH, int KW, int stride, int OH, int OW,
               int nframes, const float* ymask, float* dx, cudaStream_t st);
int permute_conv_weight_f32(const float* src, float* dst, int OC, int C, int KH, int KW, int dir,
                            cudaStream_t st);
int softargmax_fwd_f32(const float* y, int N, int OH, int OW, int C, const float* temperature,
                       float* feat, float* smax, float* ssum, cudaStream_t st);
int softargmax_bwd_f32(const float* y, int N, int OH, int OW, int C, const float* temperature,
                       const float* feat, const float* smax, const float* ssum, const float* dfeat,
                       float* dy, float* dtau_part, cudaStream_t st);

// CTAs a persistent one-CTA-per-SM kernel launches: 148 minus the SMs left free for concurrently running collectives
// (tacorl_set_sm_reserve / TACORL_SM_RESERVE).  A statically scheduled 148-CTA kernel whose last CTAs cannot be placed
// because NCCL holds their SMs takes up to twice as long; leaving those SMs out of the grid costs only their share.
int persistent_ctas();
void set_sm_reserve(int n);

// ---- TMA tensor maps of the tensor-core kernels (gemm_tc.cu)
// Encodes a bf16 tensor map of `rank` dimensions: dims[0] is contiguous, byte_strides[i] is the stride of dimension
// i + 1, box is the tile one TMA load copies.  No interleave, 256-byte L2 promotion, elements outside the tensor read as
// zero.  On failure the library error names `what` (kernel and operand) and the shape; the caller checks alignment.
bool tmap_encoder_available();
int encode_tmap_bf16(CUtensorMap* tm, const char* what, int rank, const void* base, const cuuint64_t* dims,
                     const cuuint64_t* byte_strides, const cuuint32_t* box,
                     CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B);

// ---- bf16 tcgen05 GEMM (gemm_tc.cu)
struct TcArgs {
  float alpha = 1.f, beta = 0.f;
  float* C = nullptr; long long ldc = 0;          // fp32 output
  void* Cb = nullptr; long long ldcb = 0;         // optional bf16 copy of the output
  const float* bias = nullptr;
  int act = ACT_NONE;
  float* Cpre = nullptr; long long ldpre = 0;
  int split_k = 0;                                // 0 = auto
  const float* gate = nullptr; long long ldgate = 0;   // optional ReLU gate applied to the output
};
// bf16 operands in place: a_mn/b_mn = operand stored [K][rows] (rows contiguous) instead of [rows][K].
// route (optional, host int[4]) receives the kernel that ran: {0 = tiled, 1 = skinny cluster; tiled BN or skinny NT;
// z-slices (tiled: K splits used, skinny: the cluster's K slabs); CTAs launched}.
int gemm_tc_bf16(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, int M, int N,
                 int K, const TcArgs& e, float* ws, size_t ws_bytes, cudaStream_t st, int* route = nullptr);
// persistent recurrence (gemm_tc.cu): returns 1 if unsupported (caller launches step by step); flags: >= 16 unsigned
int rnn_seq_tc(const void* Ab, int T, const void* W, long long ldw, int M, int N, int K, int tau0, int dtau, int n_steps,
               float beta, float* C, long long ldc, long long c_ts, const float* gate, long long ldgate, long long gate_ts,
               void* Cb, int act, unsigned* flags, cudaStream_t st);
// two-lane persistent recurrence (gemm_tc.cu, rnn_wave_kernel): batch rows <= 64, 1 or 2 independent recurrences in one
// launch.  Ab: bf16 [T][M][K] with row pitch lda and time stride a_ts (elements); Cb receives the bf16 results (row pitch
// ldcb, time stride cb_ts) and is normally the same tensor as Ab.  flags: >= 16 unsigned per lane.
struct WaveLaneHost {
  const void* Ab = nullptr; long long lda = 0, a_ts = 0;
  const void* W = nullptr; long long ldw = 0;
  int tau0 = 0, dtau = 1, n_steps = 0;
  float beta = 1.f;
  float* C = nullptr; long long ldc = 0, c_ts = 0;
  const float* gate = nullptr; long long ldgate = 0, gate_ts = 0;
  void* Cb = nullptr; long long ldcb = 0, cb_ts = 0;
  int act = ACT_NONE;
  unsigned* flags = nullptr;
};
int rnn_wave_tc(const WaveLaneHost* lanes, int n_lanes, int T, int M, int N, int K, cudaStream_t st);
unsigned rnn_seq_timeouts();
bool rnn_seq_enabled();
void rnn_seq_set_enabled(int on);
int rnn_seq_mode();
int cast_bf16_2d(const float* src, long long lds, long long rows, int cols, void* dst, long long ldd, cudaStream_t st);
int cast_transpose_bf16(const float* src, long long lds, int rows, int cols, void* dst, long long ldd, cudaStream_t st);
int gemm_tc_from_f32(const GemmArgs& g, float* ws, size_t ws_bytes, cudaStream_t st);
// precision dispatch used by the composite ops
static inline int gemm_any(int prec, const GemmArgs& g, float* ws, size_t ws_bytes, cudaStream_t st) {
  return prec == PREC_BF16 ? gemm_tc_from_f32(g, ws, ws_bytes, st) : gemm_f32(g, ws, ws_bytes, st);
}

// ---- implicit-GEMM convolutions (conv_tc.cu); all activations NHWC bf16
int conv_tc_pack(int mode, const float* W, void* Wp, cudaStream_t st);
bool conv_lin_conv1_wgrad_ok(int Wp);
int conv_lin_conv1_wgrad(const void* dy1p, const void* xs, int N, int Hp, int Wp, float beta, float* dW, float* db,
                         float* ws, size_t ws_bytes, cudaStream_t st);
bool conv_lin_conv3_wgrad_ok(int W2);
int conv_lin_conv3_wgrad(const void* dy3p, const void* y2b, int N, int H2, int W2, float beta, float* dW, float* db,
                         float* ws, size_t ws_bytes, cudaStream_t st);
int conv_tc_pack_multi(int n, const int* modes, const float* const* Ws, void* const* Wps, cudaStream_t st);
int conv_tc_s2d(const float* x, int N, int H, int W, int SH, int SW, void* xs, cudaStream_t st);
int conv_tc_s2d_u8(const unsigned char* x, int N, int H, int W, int SH, int SW, float scale, float shift, void* xs,
                   cudaStream_t st);
int u8_to_f32_normalized(long long n, const unsigned char* x, float scale, float shift, float* out, cudaStream_t st);
int conv_tc_conv1_fwd(const void* xs, int N, int H1, int W1, const void* wp, const float* bias, void* y1b, cudaStream_t st);
int conv_tc_conv2_fwd(const void* y1b, int N, int H1, int W1, int H2, int W2, const void* wp, const float* bias,
                      void* y2b, cudaStream_t st);
int conv_tc_conv3_fwd(const void* y2b, int N, int H2, int W2, int H3, int W3, const void* wp, const float* bias,
                      float* y3, cudaStream_t st);
// linear-shift forms (input window loaded once per tile, taps = shifted UMMA descriptors)
int conv_lin_conv1_fwd(const void* xs, int N, int H1, int W1, const void* wp, const float* bias, void* y1b, cudaStream_t st);
int conv_lin_conv3_fwd(const void* y2b, int N, int H2, int W2, int H3, int W3, const void* wp, const float* bias,
                       float* y3, cudaStream_t st);
int conv_dgrad2_fused(const void* dy2b, int N, int H1, int W1, int H2, int W2, const void* wp5, const void* y1b, void* dy1b,
                      int out_pad, cudaStream_t st);
int conv_tc_conv3_dgrad(const void* dy3b, int N, int H2, int W2, int H3, int W3, const void* wp, const void* y2b,
                        void* dy2b, cudaStream_t st);
int conv_tc_conv2_dgrad(const void* dy2b, int N, int H1, int W1, int H2, int W2, const void* wp_classes,
                        const void* y1b, void* dy1b, cudaStream_t st);
int softargmax_bwd_bf16out(const float* y, int N, int OH, int OW, int C, const float* temperature, const float* feat,
                           const float* smax, const float* ssum, const float* dfeat, void* dy_bf16, float* dtau_part,
                           int pad_h, int pad_w, cudaStream_t st);
int conv_tc_wgrad(int layer, const void* dyb, const void* src, int N, int SH, int SW, int RA, int RB, float beta,
                  float* dW, float* db, float* ws, size_t ws_bytes, cudaStream_t st);

// simple bump allocator over a caller-provided workspace (256-byte aligned slices)
struct Arena {
  char* base; size_t cap; size_t off = 0;
  Arena(void* p, size_t n) : base((char*)p), cap(n) {}
  template <typename T> T* take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    if (off + bytes > cap) return nullptr;
    T* r = (T*)(base + off);
    off += bytes;
    return r;
  }
  size_t left() const { return cap - off; }
};

}  // namespace tacorl
