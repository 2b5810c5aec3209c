// Device-side input pipeline (SURVEY.md section 8f-1): what the reference's CPU DataLoader workers do per training
// sample, as streaming kernels over uint8 frames that are already resident in HBM.
//   window gather + pad_sequence   /root/reference/src/tacorl/datamodule/dataset/play_dataset.py:115-169, 282-330
//   RandomShiftsAug                utils/transforms.py:265-299  (replicate-pad by `pad`, shift by an integer in [0, 2 pad])
//   ScaleImageTensor               utils/transforms.py:87-101   (u8 / 255)
//   ColorTransform                 utils/transforms.py:302-330  (torchvision ColorJitter: brightness / contrast / hue in
//                                                                a random order per image)
//   Normalize(mean, std)           config/datamodule/transform_manager/transforms/rl_train.yaml:12-14
// All random quantities (window starts / sizes, shifts, jitter factors, op order) are inputs, drawn by the host in the
// reference's order, like every other noise tensor of this library.
#include "common.cuh"
#include "internal.h"
#include "../../include/tacorl_b200.h"

namespace tacorl {

// batch[b][t] = store[start[b] + min(t, window[b] - 1)] shifted by (sx, sy) - pad with edge clamping.
// One thread = 16 consecutive bytes of an output row (W % 16 == 0) or one byte.
__global__ void window_gather_u8_kernel(const unsigned char* __restrict__ store, long long frames, int C, int H, int W,
                                        const int* __restrict__ start, const int* __restrict__ window,
                                        const int* __restrict__ shift, int pad, int B, int T,
                                        unsigned char* __restrict__ out) {
  const long long plane = (long long)H * W;
  const long long total = (long long)B * T * C * plane;
  for (long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 4; i < total;
       i += (long long)gridDim.x * blockDim.x * 4) {
    long long r = i;
    const int x = (int)(r % W); r /= W;
    const int y = (int)(r % H); r /= H;
    const int c = (int)(r % C); r /= C;
    const int t = (int)(r % T);
    const int b = (int)(r / T);
    const int w = window ? window[b] : T;
    long long f = (long long)start[b] + min(t, max(w, 1) - 1);
    f = min(max(f, 0LL), frames - 1);
    const unsigned char* src = store + (f * C + c) * plane;
    int sx = 0, sy = 0;
    if (shift) { sx = shift[((long long)b * T + t) * 2] - pad; sy = shift[((long long)b * T + t) * 2 + 1] - pad; }
    const int yy = min(max(y + sy, 0), H - 1);
    unsigned char v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = src[(long long)yy * W + min(max(x + j + sx, 0), W - 1)];
    if (x + 3 < W && ((i & 3) == 0)) *reinterpret_cast<uchar4*>(out + i) = make_uchar4(v[0], v[1], v[2], v[3]);
    else
      for (int j = 0; j < 4 && x + j < W; ++j) out[i + j] = v[j];
  }
}

// "rel" action modalities: steps >= window are zero except the last channel (gripper), which repeats the last valid
// step (play_dataset.py:291-301); other vector modalities repeat the last valid step entirely (zero_pad = 0).
__global__ void actions_gather_pad_kernel(const float* __restrict__ store, long long frames, int A,
                                          const int* __restrict__ start, const int* __restrict__ window, int B, int T,
                                          int zero_pad, float* __restrict__ out) {
  const int total = B * T * A;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int a = i % A, t = (i / A) % T, b = i / (A * T);
  const int w = max(window ? window[b] : T, 1);
  const long long f = min(max((long long)start[b] + min(t, w - 1), 0LL), frames - 1);
  float v = store[f * A + a];
  if (zero_pad && t >= w && a < A - 1) v = 0.f;
  out[i] = v;
}

// ---- torchvision colour ops on float RGB in [0, 1] (torchvision/transforms/_functional_tensor.py)
__device__ __forceinline__ float cj_clamp01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }
__device__ __forceinline__ float cj_gray(float r, float g, float b) { return 0.2989f * r + 0.587f * g + 0.114f * b; }
__device__ __forceinline__ void cj_hue(float& r, float& g, float& b, float hf) {
  const float maxc = fmaxf(r, fmaxf(g, b)), minc = fminf(r, fminf(g, b));
  const bool eqc = maxc == minc;
  const float cr = maxc - minc;
  const float s = cr / (eqc ? 1.f : maxc);
  const float div = eqc ? 1.f : cr;
  const float rc = (maxc - r) / div, gc = (maxc - g) / div, bc = (maxc - b) / div;
  const float hr = (maxc == r) ? (bc - gc) : 0.f;
  const float hg = ((maxc == g) && (maxc != r)) ? (2.f + rc - bc) : 0.f;
  const float hb = ((maxc != g) && (maxc != r)) ? (4.f + gc - rc) : 0.f;
  float h = fmodf((hr + hg + hb) / 6.f + 1.f, 1.f);
  h = h + hf;
  h = h - floorf(h);                                   // python's % 1.0 for floats
  const float v = maxc;
  const float h6 = h * 6.f;
  const float fi = floorf(h6);
  const float f = h6 - fi;
  int i = ((int)fi) % 6;
  if (i < 0) i += 6;
  const float p = cj_clamp01(v * (1.f - s)), q = cj_clamp01(v * (1.f - f * s)), t = cj_clamp01(v * (1.f - (1.f - f) * s));
  switch (i) {
    case 0: r = v; g = t; b = p; break;
    case 1: r = q; g = v; b = p; break;
    case 2: r = p; g = v; b = t; break;
    case 3: r = p; g = q; b = v; break;
    case 4: r = t; g = p; b = v; break;
    default: r = v; g = p; b = q; break;
  }
}
// ops of one frame in ColorJitter's order: order = three op ids (0 brightness, 1 contrast, 3 hue) packed 4 bits each,
// first op in the low bits; 0xF = no op.  `upto_contrast`: stop before the contrast op (pre-pass computing its mean).
__device__ __forceinline__ void cj_apply(float& r, float& g, float& b, int order, float fb, float fc, float fh, float mean,
                                         bool upto_contrast) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int op = (order >> (4 * k)) & 0xF;
    if (op == 0) { r = cj_clamp01(r * fb); g = cj_clamp01(g * fb); b = cj_clamp01(b * fb); }
    else if (op == 1) {
      if (upto_contrast) return;
      r = cj_clamp01(fc * r + (1.f - fc) * mean); g = cj_clamp01(fc * g + (1.f - fc) * mean); b = cj_clamp01(fc * b + (1.f - fc) * mean);
    } else if (op == 3) cj_hue(r, g, b, fh);
  }
}

// Frame n of the batch reads its op order / factors at entry (n / nf) * n_slots + slot0 + n % nf of the tables: frames
// come in groups of nf (a window), each group's parameters in a row of n_slots entries (tacorl_replay_color_jitter).
// nf = n_slots = 1, slot0 = 0: entry n.
__device__ __forceinline__ long long cj_entry(long long n, int nf, int n_slots, int slot0) {
  return (n / nf) * n_slots + slot0 + n % nf;
}

// pre-pass: mean over the frame of the grayscale of the image as it is when the contrast op runs
__global__ void color_jitter_mean_kernel(const unsigned char* __restrict__ x, int H, int W, const int* __restrict__ order,
                                         const float* __restrict__ factors, int nf, int n_slots, int slot0,
                                         float* __restrict__ mean) {
  __shared__ float red[32];
  const int n = blockIdx.x;
  const long long plane = (long long)H * W;
  const unsigned char* xp = x + (long long)n * 3 * plane;
  const long long q = cj_entry(n, nf, n_slots, slot0);
  const int ord = order[q];
  const float fb = factors[q * 3], fc = factors[q * 3 + 1], fh = factors[q * 3 + 2];
  float s = 0.f;
  for (long long p = threadIdx.x; p < plane; p += blockDim.x) {
    float r = xp[p] * (1.f / 255.f), g = xp[plane + p] * (1.f / 255.f), b = xp[2 * plane + p] * (1.f / 255.f);
    cj_apply(r, g, b, ord, fb, fc, fh, 0.f, true);
    s += cj_gray(r, g, b);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) mean[n] = t / (float)plane;
  }
}

__global__ void color_jitter_kernel(const unsigned char* __restrict__ x, long long N, int H, int W,
                                    const int* __restrict__ order, const float* __restrict__ factors, int nf,
                                    int n_slots, int slot0, const float* __restrict__ mean, float norm_mean,
                                    float norm_std, float* __restrict__ out) {
  const long long plane = (long long)H * W, total = N * plane;
  const float inv_std = 1.f / norm_std;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / plane, p = i - n * plane;
    const unsigned char* xp = x + n * 3 * plane;
    float r = xp[p] * (1.f / 255.f), g = xp[plane + p] * (1.f / 255.f), b = xp[2 * plane + p] * (1.f / 255.f);
    if (order) {
      const long long q = cj_entry(n, nf, n_slots, slot0);
      cj_apply(r, g, b, order[q], factors[q * 3], factors[q * 3 + 1], factors[q * 3 + 2], mean[n], false);
    }
    float* op = out + n * 3 * plane;
    op[p] = (r - norm_mean) * inv_std; op[plane + p] = (g - norm_mean) * inv_std; op[2 * plane + p] = (b - norm_mean) * inv_std;
  }
}

}  // namespace tacorl

using namespace tacorl;

extern "C" {

int tacorl_window_gather_u8(const unsigned char* store, long long frames, int C, int H, int W, const int* start,
                            const int* window, const int* shift, int pad, int B, int T, unsigned char* out, void* stream) {
  TACORL_REQUIRE(store && start && out && frames > 0, "window_gather_u8: null pointer / empty store");
  TACORL_REQUIRE(W % 4 == 0 && ((uintptr_t)out & 3) == 0, "window_gather_u8: image width must be a multiple of 4");
  const long long total = (long long)B * T * C * H * W;
  if (total == 0) return 0;
  const long long threads = total / 4;
  window_gather_u8_kernel<<<(int)min((long long)148 * 16, (threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      store, frames, C, H, W, start, window, shift, pad, B, T, out);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_actions_gather_pad(const float* store, long long frames, int A, const int* start, const int* window, int B,
                              int T, int zero_pad, float* out, void* stream) {
  TACORL_REQUIRE(store && start && out && frames > 0, "actions_gather_pad: null pointer / empty store");
  const int total = B * T * A;
  if (total == 0) return 0;
  actions_gather_pad_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(store, frames, A, start, window, B, T,
                                                                              zero_pad, out);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_color_jitter_u8(const unsigned char* x, long long N, int H, int W, const int* order, const float* factors,
                           float norm_mean, float norm_std, float* mean_ws, float* out, void* stream) {
  TACORL_REQUIRE(x && out, "color_jitter_u8: null pointer");
  TACORL_REQUIRE(!order || (factors && mean_ws), "color_jitter_u8: factors / workspace missing");
  TACORL_REQUIRE(norm_std != 0.f, "color_jitter_u8: std must not be zero");
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (order) {
    color_jitter_mean_kernel<<<(int)N, 256, 0, st>>>(x, H, W, order, factors, 1, 1, 0, mean_ws);
    TACORL_LAUNCH_CHECK();
  }
  const long long total = N * H * W;
  color_jitter_kernel<<<(int)min((long long)148 * 16, (total + 255) / 256), 256, 0, st>>>(x, N, H, W, order, factors, 1, 1, 0,
                                                                                        mean_ws, norm_mean, norm_std, out);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_replay_color_jitter(const unsigned char* x, int B, int nf, int H, int W, const int* order,
                               const float* factors, int n_slots, int slot0, float norm_mean, float norm_std,
                               float* mean_ws, float* out, void* stream) {
  TACORL_REQUIRE(x && order && factors && mean_ws && out, "replay_color_jitter: null pointer");
  TACORL_REQUIRE(norm_std != 0.f, "replay_color_jitter: std must not be zero");
  TACORL_REQUIRE(nf > 0 && slot0 >= 0 && slot0 + nf <= n_slots, "replay_color_jitter: slots %d + %d > %d", slot0, nf,
                 n_slots);
  const long long N = (long long)B * nf;
  if (N == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  color_jitter_mean_kernel<<<(int)N, 256, 0, st>>>(x, H, W, order, factors, nf, n_slots, slot0, mean_ws);
  TACORL_LAUNCH_CHECK();
  const long long total = N * H * W;
  color_jitter_kernel<<<(int)min((long long)148 * 16, (total + 255) / 256), 256, 0, st>>>(
      x, N, H, W, order, factors, nf, n_slots, slot0, mean_ws, norm_mean, norm_std, out);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
