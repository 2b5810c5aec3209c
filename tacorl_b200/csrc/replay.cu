// HBM-resident replay: every training step draws its own batch on the device and assembles it from uint8 frame stores
// that were uploaded once (tacorl_b200/replay.py, DESIGN.md section 13).  Two launches per step, both graph-capturable:
//   replay_sample_kernel   one CTA: reads the device step counter, draws every random quantity of the batch with
//                          counter-based Philox4x32-10 (key = seed with the rank folded in, counter = (step, sample, draw
//                          id)), writes int32 index tables and the int64 batch scalars, then advances the counter;
//                          in sweep mode (DESIGN.md section 14) it reads an item cursor instead, takes rows [0, n) from
//                          the items cursor .. cursor + n - 1 of the start table in order, draws with counter = (item, 0,
//                          draw id) and advances the cursor by n;
//   replay_gather_kernel   one block per output image plane (every modality and role of the batch in one grid, driven by
//                          a small descriptor array) plus one block per sample for the action rows.
// The gather keeps window_gather_u8_kernel's semantics (data_pipeline.cu): pad_sequence by repetition of the last frame,
// RandomShiftsAug as an integer shift with edge clamping, and pad_rel_actions for the action rows.
#include "common.cuh"
#include "internal.h"
#include "../../include/tacorl_b200.h"

namespace tacorl {

// ---- Philox4x32-10 (Salmon et al., SC'11); oracle/replay_oracle.py restates it in numpy
struct U4 { unsigned x, y, z, w; };

__device__ __forceinline__ U4 philox4x32_10(U4 c, unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c;
}

// uniform integer on [0, n): (uint64(u) * n) >> 32
__device__ __forceinline__ long long uniform_below(unsigned u, long long n) {
  return (long long)(((unsigned long long)u * (unsigned long long)n) >> 32);
}

// Geometric law on {1, 2, ...} by inverse CDF: thr[k] = floor(2^32 * P(d <= k + 1)); d = 1 + #{k : thr[k] <= u}
// (thr is non-decreasing, so this is the first k with u < thr[k], plus one).
__device__ __forceinline__ int geometric(unsigned u, const unsigned* __restrict__ thr, int n) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (thr[mid] <= u) lo = mid + 1; else hi = mid;
  }
  return lo + 1;
}

enum { KIND_PLAY_LMP = 0, KIND_TACORL = 1, KIND_CQL = 2 };
enum { DRAW_SAMPLE = 0, DRAW_NEG_GOAL = 1, DRAW_SHIFT0 = 2 };

// uniform float on [lo, lo + span): lo + span * (u >> 8) * 2^-24, every operation rounded once (no FMA contraction), so
// numpy's float32 arithmetic reproduces it bit for bit
__device__ __forceinline__ float uniform_float(unsigned u, float lo, float span) {
  return __fadd_rn(lo, __fmul_rn(span, __fmul_rn((float)(u >> 8), 5.9604644775390625e-08f)));
}

// the 6 orders of ColorJitter's enabled ops (0 brightness, 1 contrast, 3 hue)
__constant__ int kJitterPerms[6][3] = {{0, 1, 3}, {0, 3, 1}, {1, 0, 3}, {1, 3, 0}, {3, 0, 1}, {3, 1, 0}};

struct JitterParams { int ops; float lo[3], span[3]; };

// rows: rows [0, rows) of the B-row tables are written (rows = B when training).  sweep: *step_dev is an item cursor;
// row b takes item (cursor + b) mod n_valid of the start table and draws with counter (lo32(item), hi32(item), 0, draw
// id); the cursor advances by rows.  Otherwise row b draws its start with counter (lo32(step), hi32(step), b, draw id)
// and the step advances by one.
__global__ void replay_sample_kernel(int kind, int B, int rows, int sweep, int min_window, int max_window, int n_mod,
                                     int n_slots, int pad, unsigned long long neg_thr, unsigned k0, unsigned k1,
                                     long long* __restrict__ step_dev,
                                     const int* __restrict__ ep_end, long long frames, const int* __restrict__ valid,
                                     long long n_valid, const unsigned* __restrict__ geom_thr, int n_geom,
                                     int* __restrict__ tab, int* __restrict__ shift, long long* __restrict__ out64,
                                     JitterParams jit, int* __restrict__ jorder, float* __restrict__ jfac) {
  __shared__ unsigned long long s_step;
  if (threadIdx.x == 0) s_step = (unsigned long long)*step_dev;
  __syncthreads();
  const unsigned c0 = (unsigned)s_step, c1 = (unsigned)(s_step >> 32);
  int* t_start = tab;
  int* t_window = tab + B;
  int* t_goal = tab + 2 * B;
  int* t_disp = tab + 3 * B;
  for (int b = threadIdx.x; b < rows; b += blockDim.x) {
    const unsigned long long item = sweep ? (s_step + b) % (unsigned long long)n_valid : 0ull;
    const U4 ctr = sweep ? U4{(unsigned)item, (unsigned)(item >> 32), 0u, 0u} : U4{c0, c1, (unsigned)b, 0u};
    const U4 r = philox4x32_10(U4{ctr.x, ctr.y, ctr.z, DRAW_SAMPLE}, k0, k1);
    const int s = valid[sweep ? (long long)item : uniform_below(r.x, n_valid)];
    const int end = ep_end[s];
    if (kind == KIND_CQL) {
      // transition (s, s + 1); goal = min(s + k, ep_end[s]), k ~ Geometric; reward = terminal = [goal is the successor]
      const int k = geometric(r.w, geom_thr, n_geom);
      const int goal = (int)min((long long)s + k, (long long)end);
      const int hit = goal == s + 1;
      t_start[b] = s; t_window[b] = 1; t_goal[b] = goal; t_disp[b] = hit;
      out64[b] = hit; out64[B + b] = hit; out64[2 * B + b] = goal;
      continue;
    }
    const int wmax = min(max_window, end - s + 1);
    const int w = min_window + (int)uniform_below(r.y, wmax - min_window + 1);
    int goal = s + w - 1, disp = 1;
    if (kind == KIND_TACORL) {
      if ((unsigned long long)r.z < neg_thr) {
        const U4 g = philox4x32_10(U4{ctr.x, ctr.y, ctr.z, DRAW_NEG_GOAL}, k0, k1);
        goal = (int)uniform_below(g.x, frames);
        disp = -1;
      } else {
        const int d = geometric(r.w, geom_thr, n_geom);
        const int last = s + w - 1;
        goal = (int)min((long long)last + d - 1, (long long)end);
        disp = goal - last + 1;
      }
    }
    t_start[b] = s; t_window[b] = w; t_goal[b] = goal; t_disp[b] = disp;
    out64[b] = s; out64[B + b] = w; out64[2 * B + b] = disp;
  }
  if (shift != nullptr) {
    // one draw per (modality, output frame slot): x then y, each uniform on [0, 2 pad]
    const long long n = (long long)n_mod * B * n_slots;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
      const int j = (int)(i % n_slots);
      const int b = (int)((i / n_slots) % B);
      const int m = (int)(i / ((long long)n_slots * B));
      const U4 r = philox4x32_10(U4{c0, c1, (unsigned)b, (unsigned)(DRAW_SHIFT0 + m * n_slots + j)}, k0, k1);
      shift[2 * i] = (int)uniform_below(r.x, 2 * pad + 1);
      shift[2 * i + 1] = (int)uniform_below(r.y, 2 * pad + 1);
    }
  }
  if (jorder != nullptr) {
    // one draw per (modality, output frame slot) after the shift draws: op order, brightness, contrast, hue factors
    const long long n = (long long)n_mod * B * n_slots;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
      const int j = (int)(i % n_slots);
      const int b = (int)((i / n_slots) % B);
      const int m = (int)(i / ((long long)n_slots * B));
      const unsigned draw = (unsigned)(DRAW_SHIFT0 + n_mod * n_slots + m * n_slots + j);
      const U4 r = philox4x32_10(U4{c0, c1, (unsigned)b, draw}, k0, k1);
      const int* perm = kJitterPerms[uniform_below(r.x, 6)];
      int code = 0, k = 0;
      for (int q = 0; q < 3; ++q)
        if ((jit.ops >> perm[q]) & 1) code |= perm[q] << (4 * k++);
      for (; k < 3; ++k) code |= 0xF << (4 * k);
      jorder[i] = code;
      jfac[3 * i] = (jit.ops & 1) ? uniform_float(r.y, jit.lo[0], jit.span[0]) : 1.f;
      jfac[3 * i + 1] = (jit.ops & 2) ? uniform_float(r.z, jit.lo[1], jit.span[1]) : 1.f;
      jfac[3 * i + 2] = (jit.ops & 8) ? uniform_float(r.w, jit.lo[2], jit.span[2]) : 0.f;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *step_dev = (long long)(s_step + (sweep ? (unsigned long long)rows : 1ull));
}

// acc[i] += n * value[i] for i < k, acc[k] += n: one thread per slot, so every sum is taken in a fixed order
__global__ void metrics_accumulate_kernel(const __grid_constant__ tacorl_metrics m, double* __restrict__ acc) {
  const int i = threadIdx.x;
  if (i < m.k) acc[i] += (double)m.n * (double)*m.value[i];
  else if (i == m.k) acc[i] += (double)m.n;
}

// one training step's scalars into row (*step_dev % ring_rows) of the ring; acc[i] += value, acc[32 + i] += 1 for every
// logged key.  32 threads always write the whole row (NaN for a null or unused slot), so a graph captured before a
// later mode added a column leaves no stale entry behind.  One launch per step: every sum is taken in step order.
__global__ void metrics_record_kernel(const __grid_constant__ tacorl_metrics m, float* __restrict__ ring, int ring_rows,
                                      long long* __restrict__ step_dev, double* __restrict__ acc) {
  const int i = threadIdx.x;
  const long long slot = *step_dev % ring_rows;
  const float* p = i < m.k ? m.value[i] : nullptr;
  float v = __int_as_float(0x7fc00000);
  if (p) {
    v = *p;
    acc[i] += (double)v;
    acc[TACORL_METRICS_MAX + i] += 1.0;
  }
  ring[slot * TACORL_METRICS_MAX + i] = v;
  __syncthreads();
  if (i == 0) *step_dev += 1;
}

constexpr int kMaxImages = TACORL_REPLAY_MAX_IMAGES;

struct GatherImage {
  const unsigned char* store;
  unsigned char* out;
  const int* shift;
  int H, W, role, nf, shift_slot, n_slots;
  int plane0;                      // first block of this output
};
struct GatherArgs {
  GatherImage img[kMaxImages];
  int n_img, n_planes;
  int B, T, pad;
  const int* tab;
  const float* act_store;
  float* act_out;
  int A, act_role, zero_pad;
};

__device__ __forceinline__ long long source_frame(int role, const int* tab, int B, int b, int t) {
  const int s = tab[b];
  switch (role) {
    case TACORL_REPLAY_WINDOW: return (long long)s + min(t, max(tab[B + b], 1) - 1);
    case TACORL_REPLAY_NEXT: return (long long)s + 1;
    case TACORL_REPLAY_GOAL: return tab[2 * B + b];
    default: return s;
  }
}

__global__ void __launch_bounds__(256) replay_gather_kernel(const __grid_constant__ GatherArgs a) {
  const int blk = blockIdx.x;
  if (blk >= a.n_planes) {                    // action rows of sample b
    const int b = blk - a.n_planes;
    const int nf = a.act_role == TACORL_REPLAY_WINDOW ? a.T : 1;
    const int w = max(a.tab[a.B + b], 1);
    for (int i = threadIdx.x; i < nf * a.A; i += blockDim.x) {
      const int t = i / a.A, c = i - t * a.A;
      const long long f = source_frame(a.act_role, a.tab, a.B, b, t);
      float v = a.act_store[f * a.A + c];
      if (a.act_role == TACORL_REPLAY_WINDOW && a.zero_pad && t >= w && c < a.A - 1) v = 0.f;
      a.act_out[((long long)b * nf + t) * a.A + c] = v;
    }
    return;
  }
  int k = 0;
  while (k + 1 < a.n_img && blk >= a.img[k + 1].plane0) ++k;
  const GatherImage& g = a.img[k];
  int p = blk - g.plane0;                      // plane = ((b * nf) + t) * 3 + c
  const int c = p % 3; p /= 3;
  const int t = p % g.nf;
  const int b = p / g.nf;
  const long long f = source_frame(g.role, a.tab, a.B, b, t);
  const int H = g.H, W = g.W;
  const long long plane = (long long)H * W;
  const unsigned char* __restrict__ src = g.store + (f * 3 + c) * plane;
  unsigned char* __restrict__ dst = g.out + (((long long)b * g.nf + t) * 3 + c) * plane;
  int sx = 0, sy = 0;
  if (g.shift) {
    const int* sh = g.shift + ((long long)b * g.n_slots + g.shift_slot + t) * 2;
    sx = sh[0] - a.pad; sy = sh[1] - a.pad;
  }
  const int W4 = W >> 2;
  const int units = H * W4;
  if (sx == 0 && sy == 0) {
    const uchar4* s4 = reinterpret_cast<const uchar4*>(src);
    uchar4* d4 = reinterpret_cast<uchar4*>(dst);
    for (int u = threadIdx.x; u < units; u += blockDim.x) d4[u] = s4[u];
    return;
  }
  for (int u = threadIdx.x; u < units; u += blockDim.x) {
    const int y = u / W4, x = (u - y * W4) * 4;
    const unsigned char* row = src + (long long)min(max(y + sy, 0), H - 1) * W;
    uchar4 v;
    v.x = row[min(max(x + sx, 0), W - 1)];
    v.y = row[min(max(x + 1 + sx, 0), W - 1)];
    v.z = row[min(max(x + 2 + sx, 0), W - 1)];
    v.w = row[min(max(x + 3 + sx, 0), W - 1)];
    reinterpret_cast<uchar4*>(dst)[u] = v;
  }
}

}  // namespace tacorl

using namespace tacorl;

extern "C" {

static int launch_sample(int kind, int B, int rows, int sweep, int min_window, int max_window, int n_mod, int n_slots,
                         int pad, unsigned long long neg_thr, unsigned long long seed, int rank, long long* step_dev,
                         const int* ep_end, long long frames, const int* valid, long long n_valid,
                         const unsigned* geom_thr, int n_geom, int* tab, int* shift, long long* out64,
                         const tacorl_replay_jitter* jitter, int* jit_order, float* jit_factors, void* stream) {
  TACORL_REQUIRE(kind >= KIND_PLAY_LMP && kind <= KIND_CQL, "replay_sample: unknown kind %d", kind);
  TACORL_REQUIRE(step_dev && ep_end && valid && tab && out64, "replay_sample: null pointer");
  TACORL_REQUIRE(B > 0 && frames > 0 && n_valid > 0, "replay_sample: empty batch, store or start table");
  TACORL_REQUIRE(rows > 0 && rows <= B, "replay_sample: %d rows for a batch of %d", rows, B);
  TACORL_REQUIRE(kind == KIND_CQL || (min_window >= 1 && max_window >= min_window),
                 "replay_sample: window bounds %d..%d", min_window, max_window);
  TACORL_REQUIRE(kind == KIND_PLAY_LMP || (geom_thr && n_geom > 0), "replay_sample: geometric table missing");
  TACORL_REQUIRE(!shift || (pad >= 0 && n_mod > 0 && n_slots > 0), "replay_sample: shift table shape");
  TACORL_REQUIRE(!jitter || (jit_order && jit_factors && n_mod > 0 && n_slots > 0), "replay_sample: jitter tables missing");
  JitterParams jit{};
  if (jitter) {
    TACORL_REQUIRE((jitter->ops & ~0xB) == 0, "replay_sample: jitter ops mask 0x%x (bits 0, 1, 3 only)", jitter->ops);
    jit.ops = jitter->ops;
    for (int i = 0; i < 3; ++i) { jit.lo[i] = jitter->lo[i]; jit.span[i] = jitter->span[i]; }
  }
  replay_sample_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(
      kind, B, rows, sweep, min_window, max_window, n_mod, n_slots, pad, neg_thr, (unsigned)seed,
      (unsigned)(seed >> 32) ^ ((unsigned)rank * 0x9E3779B9u), step_dev, ep_end, frames, valid, n_valid, geom_thr, n_geom,
      tab, shift, out64, jit, jitter ? jit_order : nullptr, jitter ? jit_factors : nullptr);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_replay_sample(int kind, int B, int min_window, int max_window, int n_mod, int n_slots, int pad,
                         unsigned long long neg_thr, unsigned long long seed, int rank, long long* step_dev,
                         const int* ep_end, long long frames, const int* valid, long long n_valid,
                         const unsigned* geom_thr, int n_geom, int* tab, int* shift, long long* out64,
                         const tacorl_replay_jitter* jitter, int* jit_order, float* jit_factors, void* stream) {
  return launch_sample(kind, B, B, 0, min_window, max_window, n_mod, n_slots, pad, neg_thr, seed, rank, step_dev, ep_end,
                       frames, valid, n_valid, geom_thr, n_geom, tab, shift, out64, jitter, jit_order, jit_factors,
                       stream);
}

int tacorl_replay_sweep(int kind, int B, int n, int min_window, int max_window, unsigned long long neg_thr,
                        unsigned long long seed, int rank, long long* cursor_dev, const int* ep_end, long long frames,
                        const int* valid, long long n_valid, const unsigned* geom_thr, int n_geom, int* tab,
                        long long* out64, void* stream) {
  return launch_sample(kind, B, n, 1, min_window, max_window, 0, 0, 0, neg_thr, seed, rank, cursor_dev, ep_end, frames,
                       valid, n_valid, geom_thr, n_geom, tab, nullptr, out64, nullptr, nullptr, nullptr, stream);
}

int tacorl_replay_gather_rows(int B, int n, int T, int pad, const int* tab, int n_images,
                              const tacorl_replay_image* images, const float* act_store, int A, int act_role,
                              int zero_pad, float* act_out, void* stream) {
  TACORL_REQUIRE(tab && B > 0 && T > 0, "replay_gather: null table / empty batch");
  TACORL_REQUIRE(n > 0 && n <= B, "replay_gather: %d rows for a batch of %d", n, B);
  TACORL_REQUIRE(n_images >= 0 && n_images <= kMaxImages, "replay_gather: %d images (at most %d)", n_images, kMaxImages);
  TACORL_REQUIRE(!act_out || (act_store && A > 0), "replay_gather: action store missing");
  GatherArgs a{};
  long long planes = 0;
  for (int i = 0; i < n_images; ++i) {
    const tacorl_replay_image& im = images[i];
    TACORL_REQUIRE(im.store && im.out, "replay_gather: image %d: null pointer", i);
    TACORL_REQUIRE(im.W % 4 == 0 && im.H > 0 && im.W > 0, "replay_gather: image %d: width %d is not a multiple of 4", i,
                   im.W);
    TACORL_REQUIRE(((uintptr_t)im.store & 3) == 0 && ((uintptr_t)im.out & 3) == 0, "replay_gather: image %d misaligned", i);
    TACORL_REQUIRE(im.role >= TACORL_REPLAY_WINDOW && im.role <= TACORL_REPLAY_GOAL, "replay_gather: image %d: role %d", i,
                   im.role);
    const int nf = im.role == TACORL_REPLAY_WINDOW ? T : 1;
    TACORL_REQUIRE(!im.shift || (im.shift_slot >= 0 && im.shift_slot + nf <= im.n_slots),
                   "replay_gather: image %d: shift slots %d + %d > %d", i, im.shift_slot, nf, im.n_slots);
    a.img[i] = GatherImage{im.store, im.out, im.shift, im.H, im.W, im.role, nf, im.shift_slot, im.n_slots, (int)planes};
    planes += (long long)n * nf * 3;
  }
  TACORL_REQUIRE(planes < (1LL << 30), "replay_gather: batch too large");
  a.n_img = n_images; a.n_planes = (int)planes;
  a.B = B; a.T = T; a.pad = pad; a.tab = tab;
  a.act_store = act_store; a.act_out = act_out; a.A = A; a.act_role = act_role; a.zero_pad = zero_pad;
  const long long blocks = planes + (act_out ? n : 0);
  if (blocks == 0) return 0;
  replay_gather_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(a);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_replay_gather(int B, int T, int pad, const int* tab, int n_images, const tacorl_replay_image* images,
                         const float* act_store, int A, int act_role, int zero_pad, float* act_out, void* stream) {
  return tacorl_replay_gather_rows(B, B, T, pad, tab, n_images, images, act_store, A, act_role, zero_pad, act_out,
                                   stream);
}

int tacorl_metrics_accumulate(const tacorl_metrics* m, double* acc, void* stream) {
  TACORL_REQUIRE(m && acc, "metrics_accumulate: null pointer");
  TACORL_REQUIRE(m->k >= 0 && m->k <= TACORL_METRICS_MAX, "metrics_accumulate: %d metrics (at most %d)", m->k,
                 TACORL_METRICS_MAX);
  TACORL_REQUIRE(m->n > 0, "metrics_accumulate: batch of %d items", m->n);
  for (int i = 0; i < m->k; ++i) TACORL_REQUIRE(m->value[i], "metrics_accumulate: metric %d: null pointer", i);
  metrics_accumulate_kernel<<<1, 32 * ((m->k + 32) / 32), 0, (cudaStream_t)stream>>>(*m, acc);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int tacorl_metrics_record(const tacorl_metrics* m, float* ring, int ring_rows, long long* step_dev, double* acc,
                          void* stream) {
  TACORL_REQUIRE(m && ring && step_dev && acc, "metrics_record: null pointer");
  TACORL_REQUIRE(m->k >= 0 && m->k <= TACORL_METRICS_MAX, "metrics_record: %d metrics (at most %d)", m->k,
                 TACORL_METRICS_MAX);
  TACORL_REQUIRE(ring_rows >= 1, "metrics_record: %d ring rows", ring_rows);
  metrics_record_kernel<<<1, TACORL_METRICS_MAX, 0, (cudaStream_t)stream>>>(*m, ring, ring_rows, step_dev, acc);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
