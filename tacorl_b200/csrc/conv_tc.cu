// Implicit-GEMM convolutions on the 5th-gen tensor cores (sm_100a): no im2col matrix is ever materialised.
//
//   rows (M)      = output pixels, 128 per tile, persistent CTAs loop over tiles
//   K blocks      = filter taps (or tap pairs): 64 bf16 = one 128-byte NHWC pixel run of the source activation
//   A operand     = gathered by 4 producer warps with 16-byte cp.async straight from the NHWC activation into
//                   128B-swizzled shared memory (thread r owns tile row r; out-of-image taps are zero-filled),
//                   fenced into the async proxy and handed to the MMA warp through an mbarrier ring
//   B operand     = the layer's packed bf16 weights, TMA-loaded ONCE per CTA and kept resident in shared memory
//   accumulator   = TMEM, double-buffered so the epilogue of tile i overlaps the MMAs of tile i+1
//   epilogue      = TMEM load -> bias + ReLU (forward) or ReLU gate of the saved activation (dgrad) -> NHWC bf16/fp32
//
// The same kernel runs conv1 (as a 2x2/stride-1 conv over a space-to-depth(4) copy of the image), conv2, conv3 forward,
// conv3 dgrad and the four stride-parity classes of conv2 dgrad.  conv_tc_wgrad_kernel computes the weight gradients
// with both operands MN-major (pixels are the UMMA K dimension).
// Reference semantics: nn.Conv2d x3 + ReLU of /root/reference/src/tacorl/networks/visual_encoders/encoder.py:369-390.
#include "common.cuh"
#include "internal.h"
#include "sm100.cuh"
#include <cuda_bf16.h>
#include <algorithm>

namespace tacorl {

constexpr int CV_MAXT = 16;
constexpr int CV_STAGES = 8;
constexpr int CV_THREADS = 192;     // TMA warp, MMA warp, 4 epilogue warps

struct ConvGeom {
  int BW, BH;                       // output patch per tile: BW x BH pixels, tile row r = a_l*BW + b_l, BW*BH <= 128
  int tiles_x, tiles_y, num_tiles;  // tiles per frame, total tiles (frames * tiles_x * tiles_y)
  int ntaps;
  int tap_x[CV_MAXT], tap_p[CV_MAXT], tap_y[CV_MAXT];   // source-view coordinates of tap t relative to the patch origin
  int RA, RB;                       // valid output-pixel grid of this launch per frame (a < RA, b < RB)
  // output pixel of row (a,b): (a*oys + oy0, b*oxs + ox0) in an (N, OH, OW, OC) tensor
  int OH, OW, oys, oy0, oxs, ox0;
};

struct ConvEpi {
  const float* bias;                // per output channel (forward) or null
  int relu;
  const __nv_bfloat16* gate;        // dgrad: saved activation at the output pixel; output zeroed where gate <= 0
  __nv_bfloat16* out_bf16;          // (N, OH, OW, BN) or null
  float* out_f32;                   // (N, OH, OW, BN) or null
};

// ---- cp.async gathers and wide stores (the TMA / tcgen05 primitives are in sm100.cuh)
__device__ __forceinline__ void cv_cp16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// arrive on `bar` once all cp.async issued so far by this thread have landed (no thread stall; the barrier's
// expected count already includes this arrival)
__device__ __forceinline__ void cv_cp_async_arrive(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void cv_st32(void* p, const uint32_t (&v)[8]) {     // one full 32-byte sector per lane
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void cv_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cv_wait_group() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cv_wait_group_dyn(int n) {   // n in [0, 4]
  switch (n) {
    case 0: cv_wait_group<0>(); break;
    case 1: cv_wait_group<1>(); break;
    case 2: cv_wait_group<2>(); break;
    case 3: cv_wait_group<3>(); break;
    default: cv_wait_group<4>(); break;
  }
}
__device__ __forceinline__ void cv_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------ forward / dgrad
// One tile = a BW x BH patch of output pixels of one frame (row r = a_l*BW + b_l, BW*BH <= 128).  For filter tap t
// the A operand of that tile is the same patch of the source activation shifted by the tap offset: ONE 5-D TMA box
// (64 channels x BW x 1 x BH x 1 frame) written straight into a 128B-swizzled stage.  Out-of-image taps (data
// gradients) and the ragged patch edges are zero-filled by TMA; stride-2 layers address the source through a
// (pixel pair, row parity) view so no element strides are needed.
template <int BN, int NTAPS>
__global__ void __launch_bounds__(CV_THREADS, 1)
conv_tc_kernel(const __grid_constant__ ConvGeom g, const __grid_constant__ CUtensorMap tmA,
               const __grid_constant__ CUtensorMap tmW, const ConvEpi ep) {
  constexpr uint32_t A_BYTES = 128 * 128;              // 128 rows x 64 bf16
  constexpr uint32_t W_TAP_BYTES = BN * 128;           // [BN][64] bf16, K-major SW128
  constexpr uint32_t ACC_COLS = BN < 32 ? 32 : BN;
  constexpr uint32_t TMEM_COLS = 2 * ACC_COLS;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t w_base = smem_u32(smem);
  const uint32_t a_base = w_base + g.ntaps * W_TAP_BYTES;            // multiple of 1024 (BN*128 with BN >= 32: 4096)
  uint64_t* bars = (uint64_t*)(smem + g.ntaps * W_TAP_BYTES + CV_STAGES * A_BYTES);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * CV_STAGES + 5);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + CV_STAGES + s); };
  auto tfull_bar = [&](int a) { return smem_u32(bars + 2 * CV_STAGES + a); };
  auto tempty_bar = [&](int a) { return smem_u32(bars + 2 * CV_STAGES + 2 + a); };
  const uint32_t w_bar = smem_u32(bars + 2 * CV_STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_frame = g.tiles_x * g.tiles_y;
  __shared__ float s_bias[BN];
  if (threadIdx.x < BN) s_bias[threadIdx.x] = ep.bias ? ep.bias[threadIdx.x] : 0.f;

  if (threadIdx.x == 0) {
    for (int s = 0; s < CV_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    mbar_init(w_bar, 1);
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer: resident weights (one box per tap), then one activation box per (tile, tap)
      mbar_expect_tx(w_bar, g.ntaps * W_TAP_BYTES);
      for (int t = 0; t < g.ntaps; ++t) tma_load_2d(w_base + t * W_TAP_BYTES, &tmW, 0, t * BN, w_bar);
      const uint32_t box_bytes = (uint32_t)(g.BW * g.BH) * 128;
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x) {
        const int n = tile / tiles_per_frame, rem = tile - n * tiles_per_frame;
        const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
        const int x0 = tx * g.BW, y0 = ty * g.BH;
        for (int t = 0; t < g.ntaps; ++t, ++it) {
          const int s = it % CV_STAGES;
          mbar_wait(empty_bar(s), ((it / CV_STAGES) & 1) ^ 1);
          mbar_expect_tx(full_bar(s), box_bytes);
          tma_load_5d(a_base + s * A_BYTES, &tmA, 0, x0 + g.tap_x[t], g.tap_p[t], y0 + g.tap_y[t], n, full_bar(s));
        }
      }
    }
  } else if (warp == 1) {
    {
      mbar_wait(w_bar, 0);
      constexpr uint32_t idesc = idesc_bf16(128, BN);
      // the whole warp runs the issue loop (warp-uniform descriptors in uniform registers), one elected lane issues; its
      // lanes wait through every ring phase in order and meet at each elect.sync, so each ring still has one in-order
      // waiter.  Descriptors are precomputed (weights: per tap and K step; stages: base + stage * size), leaving one 64-bit add
      // per operand per instruction
      uint64_t bdesc[NTAPS * 4];
#pragma unroll
      for (int i = 0; i < NTAPS * 4; ++i) bdesc[i] = smem_desc(w_base + (i >> 2) * W_TAP_BYTES + (i & 3) * 32, 16, 1024);
      const uint64_t adesc0 = smem_desc(a_base, 16, 1024);
      uint32_t it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++lt) {
        const uint32_t acc = lt & 1;
        mbar_wait(tempty_bar(acc), ((lt >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * ACC_COLS;
#pragma unroll
        for (int t = 0; t < NTAPS; ++t, ++it) {
          const int s = it % CV_STAGES;
          mbar_wait(full_bar(s), (it / CV_STAGES) & 1);
          tc_fence_after();
          const uint64_t adesc = adesc0 + (uint64_t)(s * (A_BYTES >> 4));
#pragma unroll
          for (int k = 0; k < 4; ++k) tc_mma_bf16_warp(tmem_d, adesc + 2 * k, bdesc[t * 4 + k], idesc, (t > 0 || k > 0) ? 1u : 0u);
          tc_commit_warp(empty_bar(s));
        }
        tc_commit_warp(tfull_bar(acc));
      }
    }
  } else {
    // ===== epilogue warps 2..5: TMEM lane quarter = warp % 4; lane r of the tile is patch pixel (r / BW, r % BW)
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int a_l = r / g.BW, b_l = r - a_l * g.BW;
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++lt) {
      const uint32_t acc = lt & 1;
      const int n = tile / tiles_per_frame, rem = tile - n * tiles_per_frame;
      const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
      const int a = ty * g.BH + a_l, b = tx * g.BW + b_l;
      const bool row_ok = a_l < g.BH && a < g.RA && b < g.RB;
      const long long opix = row_ok ? ((long long)n * g.OH + (a * g.oys + g.oy0)) * g.OW + (b * g.oxs + g.ox0) : 0;
      // prefetch the ReLU gate of this row (global latency) before blocking on the accumulator
      uint4 gate[BN / 8];
      if (ep.gate && row_ok) {
        const uint4* gp = reinterpret_cast<const uint4*>(ep.gate + opix * BN);
#pragma unroll
        for (int j = 0; j < BN / 8; ++j) gate[j] = __ldg(gp + j);
      }
      mbar_wait(tfull_bar(acc), (lt >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t rr[16];
        tc_ld16(tmem_base + acc * ACC_COLS + ((uint32_t)(q * 32) << 16) + c0, rr);
        if (!row_ok) continue;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]) + s_bias[c0 + j];
        if (ep.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (ep.gate) {
          const uint4 g0 = gate[c0 / 8], g1 = gate[c0 / 8 + 1];
          const __nv_bfloat162* h0 = reinterpret_cast<const __nv_bfloat162*>(&g0);
          const __nv_bfloat162* h1 = reinterpret_cast<const __nv_bfloat162*>(&g1);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f0 = __bfloat1622float2(h0[j]), f1 = __bfloat1622float2(h1[j]);
            if (f0.x <= 0.f) v[2 * j] = 0.f;
            if (f0.y <= 0.f) v[2 * j + 1] = 0.f;
            if (f1.x <= 0.f) v[8 + 2 * j] = 0.f;
            if (f1.y <= 0.f) v[8 + 2 * j + 1] = 0.f;
          }
        }
        if (ep.out_bf16) {
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            __nv_bfloat162 t2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
            pk[j] = *reinterpret_cast<uint32_t*>(&t2);
          }
          cv_st32(ep.out_bf16 + opix * BN + c0, pk);
        }
        if (ep.out_f32) {
          uint32_t lo[8], hi[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) { lo[j] = __float_as_uint(v[j]); hi[j] = __float_as_uint(v[8 + j]); }
          cv_st32(ep.out_f32 + opix * BN + c0, lo);
          cv_st32(ep.out_f32 + opix * BN + c0 + 8, hi);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------ linear-shift variant
// Stride-1 layers whose input and output share one row pitch W: output pixel with linear index p = a*W + b reads, for
// filter tap (ky, kx), input pixel p + ky*W + kx - the SAME linear pixel array shifted by a constant.  A tile is 128
// consecutive linear pixels of one frame; its whole input window (128 + max shift pixel rows of 128 bytes) is loaded
// ONCE by a single 2-D TMA box, and every tap's A operand is that stage addressed at a shifted start: the UMMA
// descriptor's start address simply advances by shift*128 bytes.  The tensor core applies the 128-byte swizzle to the
// absolute shared-memory address bits (the same bits TMA used when it wrote the stage), so a start address that is
// not aligned to the 1024-byte swizzle atom needs no further adjustment - measured: results are exact with the
// descriptor's base-offset field left 0 and wrong with it set to (shift & 7); tests/test_gpu_conv_tc.py.  L2->SM
// traffic per tile drops from ntaps x 16 KB to (128 + max shift) x 128 B; the columns b >= OW of each output row are
// computed and discarded (conv3: 21 of 23 kept).
struct ConvLinGeom {
  int W, OH, OW;                    // shared row pitch (input pixels per row), valid output grid
  int frame_rows;                   // input pixel rows per frame in the 2-D view (H*W)
  int tiles_per_frame, num_tiles;
  int ntaps, load_rows;             // load_rows = 128 + max shift, rounded up to 8
  int stages;
  int shift[CV_MAXT];
  // output pixel (a, b) -> (a*oys + oy0, b*oxs + ox0) of an (N, OHt, OWt, BN) tensor
  int OHt, OWt, oys, oy0, oxs, ox0;
};
constexpr int CL_MAX_STAGES = 8;    // ring depth g.stages <= 8: as many input windows in flight as shared memory holds

template <int BN, int NTAPS, int KSTEPS>
__global__ void __launch_bounds__(CV_THREADS, 1)
conv_lin_kernel(const __grid_constant__ ConvLinGeom g, const __grid_constant__ CUtensorMap tmA,
                const __grid_constant__ CUtensorMap tmW, const ConvEpi ep) {
  constexpr uint32_t W_TAP_BYTES = BN * 128;
  constexpr uint32_t ACC_COLS = BN < 32 ? 32 : BN;
  constexpr int NACC = 4;                       // accumulator ring: the epilogue may lag the MMAs by up to 3 tiles
  constexpr uint32_t TMEM_COLS = NACC * ACC_COLS;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t stage_bytes = ((uint32_t)g.load_rows * 128 + 1023) & ~1023u;
  const uint32_t w_base = smem_u32(smem);
  const uint32_t a_base = w_base + g.ntaps * W_TAP_BYTES;
  uint64_t* bars = (uint64_t*)(smem + g.ntaps * W_TAP_BYTES + g.stages * stage_bytes);
  const int CL_STAGES = g.stages;
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * CL_MAX_STAGES + 2 * NACC + 1);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + CL_MAX_STAGES + s); };
  auto tfull_bar = [&](int a) { return smem_u32(bars + 2 * CL_MAX_STAGES + a); };
  auto tempty_bar = [&](int a) { return smem_u32(bars + 2 * CL_MAX_STAGES + NACC + a); };
  const uint32_t w_bar = smem_u32(bars + 2 * CL_MAX_STAGES + 2 * NACC);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __shared__ float s_bias[BN];
  if (threadIdx.x < BN) s_bias[threadIdx.x] = ep.bias ? ep.bias[threadIdx.x] : 0.f;

  if (threadIdx.x == 0) {
    for (int s = 0; s < CL_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < NACC; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    mbar_init(w_bar, 1);
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(w_bar, g.ntaps * W_TAP_BYTES);
      for (int t = 0; t < g.ntaps; ++t) tma_load_2d(w_base + t * W_TAP_BYTES, &tmW, 0, t * BN, w_bar);
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++it) {
        const int n = tile / g.tiles_per_frame, k = tile - n * g.tiles_per_frame;
        const int s = it % CL_STAGES;
        mbar_wait(empty_bar(s), ((it / CL_STAGES) & 1) ^ 1);
        mbar_expect_tx(full_bar(s), (uint32_t)g.load_rows * 128);
        tma_load_2d(a_base + s * stage_bytes, &tmA, 0, n * g.frame_rows + k * 128, full_bar(s));
      }
    }
  } else if (warp == 1) {
    {
      mbar_wait(w_bar, 0);
      constexpr uint32_t idesc = idesc_bf16(128, BN);
      // The issue loop is warp-uniform scalar code (one elected lane issues): keep it to one 64-bit add per operand per
      // MMA.  Descriptor =
      // (constant high word, start address >> 4 in the low 14 bits); offsets below never carry out of that field
      // (shared memory is < 256 KB = 2^14 x 16 B).
      uint32_t aoff[NTAPS * KSTEPS];
      uint64_t bdesc[NTAPS * KSTEPS];
#pragma unroll
      for (int t = 0; t < NTAPS; ++t)
#pragma unroll
        for (int k = 0; k < KSTEPS; ++k) {
          aoff[t * KSTEPS + k] = ((uint32_t)g.shift[t] * 128 + k * 32) >> 4;
          bdesc[t * KSTEPS + k] = smem_desc(w_base + t * W_TAP_BYTES + k * 32, 16, 1024);
        }
      const uint64_t adesc0 = smem_desc(a_base, 16, 1024);
      const uint32_t stage16 = stage_bytes >> 4;
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it % NACC;
        const int s = it % CL_STAGES;
        mbar_wait(tempty_bar(acc), ((it / NACC) & 1) ^ 1);
        mbar_wait(full_bar(s), (it / CL_STAGES) & 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * ACC_COLS;
        const uint64_t adesc = adesc0 + (uint64_t)(s * stage16);
#pragma unroll
        for (int i = 0; i < NTAPS * KSTEPS; ++i) tc_mma_bf16_warp(tmem_d, adesc + aoff[i], bdesc[i], idesc, i > 0 ? 1u : 0u);
        tc_commit_warp(empty_bar(s));
        tc_commit_warp(tfull_bar(acc));
      }
    }
  } else {
    const int q = warp & 3;
    const int r = q * 32 + lane;
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++lt) {
      const uint32_t acc = lt % NACC;
      const int n = tile / g.tiles_per_frame, k = tile - n * g.tiles_per_frame;
      const int p = k * 128 + r, a = p / g.W, b = p - a * g.W;
      const bool row_ok = a < g.OH && b < g.OW;
      const long long opix = row_ok ? ((long long)n * g.OHt + (a * g.oys + g.oy0)) * g.OWt + (b * g.oxs + g.ox0) : 0;
      uint4 gate[BN / 8];
      if (ep.gate && row_ok) {
        const uint4* gp = reinterpret_cast<const uint4*>(ep.gate + opix * BN);
#pragma unroll
        for (int j = 0; j < BN / 8; ++j) gate[j] = __ldg(gp + j);
      }
      mbar_wait(tfull_bar(acc), (lt / NACC) & 1);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t rr[16];
        tc_ld16(tmem_base + acc * ACC_COLS + ((uint32_t)(q * 32) << 16) + c0, rr);
        if (!row_ok) continue;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]) + s_bias[c0 + j];
        if (ep.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (ep.gate) {
          const uint4 g0 = gate[c0 / 8], g1 = gate[c0 / 8 + 1];
          const __nv_bfloat162* h0 = reinterpret_cast<const __nv_bfloat162*>(&g0);
          const __nv_bfloat162* h1 = reinterpret_cast<const __nv_bfloat162*>(&g1);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f0 = __bfloat1622float2(h0[j]), f1 = __bfloat1622float2(h1[j]);
            if (f0.x <= 0.f) v[2 * j] = 0.f;
            if (f0.y <= 0.f) v[2 * j + 1] = 0.f;
            if (f1.x <= 0.f) v[8 + 2 * j] = 0.f;
            if (f1.y <= 0.f) v[8 + 2 * j + 1] = 0.f;
          }
        }
        if (ep.out_bf16) {
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            __nv_bfloat162 t2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
            pk[j] = *reinterpret_cast<uint32_t*>(&t2);
          }
          cv_st32(ep.out_bf16 + opix * BN + c0, pk);
        }
        if (ep.out_f32) {
          uint32_t lo[8], hi[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) { lo[j] = __float_as_uint(v[j]); hi[j] = __float_as_uint(v[8 + j]); }
          cv_st32(ep.out_f32 + opix * BN + c0, lo);
          cv_st32(ep.out_f32 + opix * BN + c0 + 8, hi);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------ fused conv2 data gradient
// dy1[2a+py][2b+px][c] = [y1 > 0] * sum_{j,i in {0,1}} sum_oc dy2[a-j][b-i][oc] * W2[oc][c][py+2j][px+2i].
// All four stride-parity classes (py, px) of output pixel pair-block (a, b) read the SAME four dy2 pixels, so one MMA
// per tap with N = 4 classes x 32 channels = 128 replaces four N = 32 launches that each re-read dy2.  A tile is a
// PW x PH = 16 x 8 patch of dy2 pixels loaded ONCE by a 4-D TMA box whose origin lies one pixel above / left of the
// tile's first output (out-of-image pixels are zero-filled: they are exactly the taps that fall off the gradient map);
// tap (j, i) is the stage read through a UMMA descriptor shifted by ((1-j)*PW + (1-i)) pixel rows, and the patch's
// last row and column only serve as halo (15 x 7 outputs (a, b) per tile, each producing a 2 x 2 block of dy1).
constexpr int DG_PW = 16, DG_PH = 8;
constexpr int DG_STAGES = 8;
struct Dgrad2Geom {
  int H1, W1, H2, W2;               // dy1 / y1 grid, dy2 grid
  int RA, RB;                       // pair-block grid: RA = ceil(H1 / 2), RB = ceil(W1 / 2)
  int tiles_x, tiles_y, num_tiles;
  int OHp, OWp;                     // frame height / row pitch (pixels) of dy1: H1 / W1, or larger (zero margin written elsewhere)
};

// 8 epilogue warps: the four parity classes of a tile are drained by two warps per TMEM lane quarter (classes 0-1 / 2-3);
// the kernel is epilogue-paced (gate loads + 4 x 64 B of packed bf16 per pixel block), not MMA- or DRAM-bound
constexpr int DG_THREADS = 64 + 8 * 32;
__global__ void __launch_bounds__(DG_THREADS, 1)
conv_dgrad2_kernel(const __grid_constant__ Dgrad2Geom g, const __grid_constant__ CUtensorMap tmA,
                   const __grid_constant__ CUtensorMap tmW, const __nv_bfloat16* __restrict__ y1,
                   __nv_bfloat16* __restrict__ dy1) {
  constexpr uint32_t A_BYTES = 128 * 128, W_TAP_BYTES = 128 * 128, ACC_COLS = 128, TMEM_COLS = 256;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t w_base = smem_u32(smem);
  const uint32_t a_base = w_base + 4 * W_TAP_BYTES;
  // (one spare tile after the ring: the shifted reads of the halo rows run up to 17 rows past the last stage)
  uint64_t* bars = (uint64_t*)(smem + 4 * W_TAP_BYTES + (DG_STAGES + 1) * A_BYTES);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * DG_STAGES + 5);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + DG_STAGES + s); };
  auto tfull_bar = [&](int a) { return smem_u32(bars + 2 * DG_STAGES + a); };
  auto tempty_bar = [&](int a) { return smem_u32(bars + 2 * DG_STAGES + 2 + a); };
  const uint32_t w_bar = smem_u32(bars + 2 * DG_STAGES + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_frame = g.tiles_x * g.tiles_y;

  if (threadIdx.x == 0) {
    for (int s = 0; s < DG_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }
    mbar_init(w_bar, 1);
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(w_bar, 4 * W_TAP_BYTES);
      for (int t = 0; t < 4; ++t) tma_load_2d(w_base + t * W_TAP_BYTES, &tmW, 0, t * 128, w_bar);
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++it) {
        const int n = tile / tiles_per_frame, rem = tile - n * tiles_per_frame;
        const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
        const int s = it % DG_STAGES;
        mbar_wait(empty_bar(s), ((it / DG_STAGES) & 1) ^ 1);
        mbar_expect_tx(full_bar(s), A_BYTES);
        tma_load_4d(a_base + s * A_BYTES, &tmA, 0, tx * (DG_PW - 1) - 1, ty * (DG_PH - 1) - 1, n, full_bar(s));
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      mbar_wait(w_bar, 0);
      constexpr uint32_t idesc = idesc_bf16(128, 128);
      uint32_t aoff[16];
      uint64_t bdesc[16];
#pragma unroll
      for (int t = 0; t < 4; ++t)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int j = t >> 1, i = t & 1;
          aoff[t * 4 + k] = (uint32_t)(((1 - j) * DG_PW + (1 - i)) * 128 + k * 32) >> 4;
          bdesc[t * 4 + k] = smem_desc(w_base + t * W_TAP_BYTES + k * 32, 16, 1024);
        }
      const uint64_t adesc0 = smem_desc(a_base, 16, 1024);
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it & 1;
        const int s = it % DG_STAGES;
        mbar_wait(tempty_bar(acc), ((it >> 1) & 1) ^ 1);
        mbar_wait(full_bar(s), (it / DG_STAGES) & 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * ACC_COLS;
        const uint64_t adesc = adesc0 + (uint64_t)(s * (A_BYTES >> 4));
#pragma unroll
        for (int i = 0; i < 16; ++i) tc_mma_bf16(tmem_d, adesc + aoff[i], bdesc[i], idesc, i > 0 ? 1u : 0u);
        tc_commit(empty_bar(s));
        tc_commit(tfull_bar(acc));
      }
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;                    // this warp's pair of parity classes
    const int r = q * 32 + lane;
    const int al = r / DG_PW, bl = r - al * DG_PW;
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++lt) {
      const uint32_t acc = lt & 1;
      const int n = tile / tiles_per_frame, rem = tile - n * tiles_per_frame;
      const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
      const int a = ty * (DG_PH - 1) + al, b = tx * (DG_PW - 1) + bl;
      const bool row_ok = al < DG_PH - 1 && bl < DG_PW - 1 && a < g.RA && b < g.RB;
      // ReLU gates of the 2 x 2 output block (global latency): all in flight before blocking on the accumulator
      bool okc[2];
      long long opixc[2], dpixc[2];
      uint4 gate[2][4];
#pragma unroll
      for (int c2 = 0; c2 < 2; ++c2) {
        const int oy = 2 * a + half, ox = 2 * b + c2;     // class = 2 * half + c2 = (py, px) = (half, c2)
        okc[c2] = row_ok && oy < g.H1 && ox < g.W1;
        opixc[c2] = okc[c2] ? ((long long)n * g.H1 + oy) * g.W1 + ox : 0;
        dpixc[c2] = okc[c2] ? ((long long)n * g.OHp + oy) * g.OWp + ox : 0;
        const uint4* gp = reinterpret_cast<const uint4*>(y1 + opixc[c2] * 32);   // (pixel 0 of the tensor when masked)
#pragma unroll
        for (int j = 0; j < 4; ++j) gate[c2][j] = __ldg(gp + j);
      }
      mbar_wait(tfull_bar(acc), (lt >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int c2 = 0; c2 < 2; ++c2) {
        const int cls = 2 * half + c2;
        const bool ok = okc[c2];
        const long long opix = dpixc[c2];
        uint32_t r2[2][16];                  // both 16-column halves of the class in flight before the one wait
        tc_ld16_nowait(tmem_base + acc * ACC_COLS + ((uint32_t)(q * 32) << 16) + cls * 32, r2[0]);
        tc_ld16_nowait(tmem_base + acc * ACC_COLS + ((uint32_t)(q * 32) << 16) + cls * 32 + 16, r2[1]);
        tc_ld_wait();
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          const uint32_t (&rr)[16] = r2[c0 / 16];
          if (!ok) continue;
          const uint4 g0 = gate[c2][c0 / 8], g1 = gate[c2][c0 / 8 + 1];
          const __nv_bfloat162* h0 = reinterpret_cast<const __nv_bfloat162*>(&g0);
          const __nv_bfloat162* h1 = reinterpret_cast<const __nv_bfloat162*>(&g1);
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(rr[j]);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f0 = __bfloat1622float2(h0[j]), f1 = __bfloat1622float2(h1[j]);
            if (f0.x <= 0.f) v[2 * j] = 0.f;
            if (f0.y <= 0.f) v[2 * j + 1] = 0.f;
            if (f1.x <= 0.f) v[8 + 2 * j] = 0.f;
            if (f1.y <= 0.f) v[8 + 2 * j + 1] = 0.f;
          }
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            __nv_bfloat162 t2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
            pk[j] = *reinterpret_cast<uint32_t*>(&t2);
          }
          cv_st32(dy1 + opix * 32 + c0, pk);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------ host side
// packed weights: [ntaps * BN rows][64] bf16, K-major; one [64][BN] box per tap
static int cv_weight_tmap(CUtensorMap* tm, const void* wp, int ntaps, int BN) {
  TACORL_REQUIRE(((uintptr_t)wp & 15) == 0, "conv_tc: packed weights must be 16-byte aligned");
  const cuuint64_t dims[2] = {64, (cuuint64_t)ntaps * BN}, strides[1] = {128};
  const cuuint32_t box[2] = {64, (cuuint32_t)BN};
  return encode_tmap_bf16(tm, "conv_tc(weights)", 2, wp, dims, strides, box);
}

// 5-D view of an NHWC bf16 activation for the patch boxes: (64 channels, x, p, y, n); strides in bytes.
struct ActView {
  const void* base;
  long long nx, np, ny, nn;
  long long sx, sp, sy, sn;
};
static int cv_act_tmap(CUtensorMap* tm, const ActView& v, int BW, int BH) {
  TACORL_REQUIRE(((uintptr_t)v.base & 15) == 0 && v.sx % 16 == 0 && v.sp % 16 == 0 && v.sy % 16 == 0 && v.sn % 16 == 0,
                 "conv_tc: activation view must be 16-byte aligned (strides %lld %lld %lld %lld)", v.sx, v.sp, v.sy, v.sn);
  const cuuint64_t dims[5] = {64, (cuuint64_t)v.nx, (cuuint64_t)v.np, (cuuint64_t)v.ny, (cuuint64_t)v.nn};
  const cuuint64_t strides[4] = {(cuuint64_t)v.sx, (cuuint64_t)v.sp, (cuuint64_t)v.sy, (cuuint64_t)v.sn};
  const cuuint32_t box[5] = {64, (cuuint32_t)BW, 1, (cuuint32_t)BH, 1};
  return encode_tmap_bf16(tm, "conv_tc(activation)", 5, v.base, dims, strides, box);
}

// patch shape with the fewest wasted accumulator rows: maximise RA*RB / (tiles * 128)
static void cv_choose_patch(int RA, int RB, int* BW, int* BH) {
  long long best = -1;
  *BW = 1; *BH = 1;
  for (int bw = 1; bw <= 128 && bw <= RB; ++bw)
    for (int bh = 1; bh * bw <= 128 && bh <= RA; ++bh) {
      const long long tiles = (long long)cdiv(RB, bw) * cdiv(RA, bh);
      // fewer tiles first; among equals prefer the wider patch (longer contiguous runs)
      const long long score = -tiles * 1024 + bw;
      if (best == -1 || score > best) { best = score; *BW = bw; *BH = bh; }
    }
}

template <int BN, int NTAPS>
static int cv_launch(const ConvGeom& g, const ActView& view, const void* wpacked, const ConvEpi& ep, cudaStream_t st) {
  CUtensorMap tw, ta;
  int rc = cv_weight_tmap(&tw, wpacked, g.ntaps, BN);
  if (rc) return rc;
  if ((rc = cv_act_tmap(&ta, view, g.BW, g.BH))) return rc;
  const size_t smem = (size_t)g.ntaps * BN * 128 + CV_STAGES * 128 * 128 + (2 * CV_STAGES + 5) * 8 + 16 + 1024;
  static size_t configured = 0;
  auto kern = conv_tc_kernel<BN, NTAPS>;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  const int ctas = g.num_tiles < persistent_ctas() ? g.num_tiles : persistent_ctas();
  kern<<<ctas, CV_THREADS, smem, st>>>(g, ta, tw, ep);
  TACORL_LAUNCH_CHECK();
  return 0;
}

// g: taps / output mapping / RA, RB filled in by the layer driver; the patch tiling is chosen here
static int conv_tc_run(ConvGeom g, int N, const ActView& view, int BN, const void* wpacked, const ConvEpi& ep,
                       cudaStream_t st) {
  if (N == 0 || g.RA <= 0 || g.RB <= 0) return 0;
  TACORL_REQUIRE(g.ntaps >= 1 && g.ntaps <= CV_MAXT, "conv_tc: bad tap count %d", g.ntaps);
  cv_choose_patch(g.RA, g.RB, &g.BW, &g.BH);
  g.tiles_x = cdiv(g.RB, g.BW); g.tiles_y = cdiv(g.RA, g.BH);
  g.num_tiles = N * g.tiles_x * g.tiles_y;
  if (BN == 32 && g.ntaps == 4) return cv_launch<32, 4>(g, view, wpacked, ep, st);
  if (BN == 64 && g.ntaps == 8) return cv_launch<64, 8>(g, view, wpacked, ep, st);
  if (BN == 64 && g.ntaps == 9) return cv_launch<64, 9>(g, view, wpacked, ep, st);
  set_last_error("conv_tc: unsupported output width %d / tap count %d", BN, g.ntaps);
  return -1;
}

// Linear-shift launch: src is an NHWC bf16 activation with 128-byte pixels, frame_rows pixel rows per frame.
template <int BN, int NTAPS, int KSTEPS>
static int cl_launch(ConvLinGeom g, int N, const void* src, const void* wpacked, const ConvEpi& ep, cudaStream_t st) {
  int max_shift = 0;
  for (int t = 0; t < g.ntaps; ++t) max_shift = g.shift[t] > max_shift ? g.shift[t] : max_shift;
  g.load_rows = (128 + max_shift + 7) & ~7;
  TACORL_REQUIRE(g.load_rows <= 256, "conv_lin: input window of %d pixel rows exceeds one TMA box", g.load_rows);
  const int lin = (g.OH - 1) * g.W + g.OW;            // linear extent of the valid outputs of one frame
  g.tiles_per_frame = cdiv(lin, 128);
  g.num_tiles = N * g.tiles_per_frame;
  CUtensorMap tw, ta;
  int rc = cv_weight_tmap(&tw, wpacked, g.ntaps, BN);
  if (rc) return rc;
  TACORL_REQUIRE(((uintptr_t)src & 15) == 0, "conv_lin: activation must be 16-byte aligned");
  const cuuint64_t dims[2] = {64, (cuuint64_t)N * g.frame_rows}, strides[1] = {128};
  const cuuint32_t box[2] = {64, (cuuint32_t)g.load_rows};
  if ((rc = encode_tmap_bf16(&ta, "conv_lin(activation)", 2, src, dims, strides, box))) return rc;
  const size_t stage = ((size_t)g.load_rows * 128 + 1023) & ~(size_t)1023;
  const size_t fixed = (size_t)g.ntaps * BN * 128 + (2 * CL_MAX_STAGES + 12) * 8 + 16 + 1024 + 256;
  g.stages = (int)std::min<size_t>(CL_MAX_STAGES, (227 * 1024 - fixed) / stage);
  TACORL_REQUIRE(g.stages >= 2, "conv_lin: input window of %zu bytes leaves no room for a stage ring", stage);
  const size_t smem = fixed - 256 + g.stages * stage;
  static size_t configured = 0;
  TACORL_REQUIRE(g.ntaps == NTAPS, "conv_lin: tap count mismatch");
  auto kern = conv_lin_kernel<BN, NTAPS, KSTEPS>;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  const int ctas = g.num_tiles < persistent_ctas() ? g.num_tiles : persistent_ctas();
  kern<<<ctas, CV_THREADS, smem, st>>>(g, ta, tw, ep);
  TACORL_LAUNCH_CHECK();
  return 0;
}

// conv3 forward, linear-shift form: y2 (N, H2, W2, 64) -> y3 fp32 (N, H3, W3, 64)
int conv_lin_conv3_fwd(const void* y2b, int N, int H2, int W2, int H3, int W3, const void* wp, const float* bias,
                       float* y3, cudaStream_t st) {
  if (128 + 2 * W2 + 2 > 256)      // input window larger than one TMA box (images wider than ~500 px): per-tap boxes
    return conv_tc_conv3_fwd(y2b, N, H2, W2, H3, W3, wp, bias, y3, st);
  ConvLinGeom g = {};
  g.W = W2; g.OH = H3; g.OW = W3; g.frame_rows = H2 * W2; g.ntaps = 9;
  for (int t = 0; t < 9; ++t) g.shift[t] = (t / 3) * W2 + (t % 3);
  g.OHt = H3; g.OWt = W3; g.oys = 1; g.oxs = 1;
  ConvEpi e = {bias, 1, nullptr, nullptr, y3};
  return cl_launch<64, 9, 4>(g, N, y2b, wp, e, st);
}
// conv1 forward on the s2d image (N, H1+1, W1+1, 64): 2x2 taps
int conv_lin_conv1_fwd(const void* xs, int N, int H1, int W1, const void* wp, const float* bias, void* y1b,
                       cudaStream_t st) {
  if (128 + (W1 + 1) + 1 > 256)    // images wider than ~510 px
    return conv_tc_conv1_fwd(xs, N, H1, W1, wp, bias, y1b, st);
  ConvLinGeom g = {};
  g.W = W1 + 1; g.OH = H1; g.OW = W1; g.frame_rows = (H1 + 1) * (W1 + 1); g.ntaps = 4;
  for (int t = 0; t < 4; ++t) g.shift[t] = (t >> 1) * (W1 + 1) + (t & 1);
  g.OHt = H1; g.OWt = W1; g.oys = 1; g.oxs = 1;
  ConvEpi e = {bias, 1, nullptr, (__nv_bfloat16*)y1b, nullptr};
  return cl_launch<32, 4, 3>(g, N, xs, wp, e, st);
}

// conv2 data gradient, all four stride-parity classes in one kernel (weights packed with mode 5)
// zero the right / bottom margin of an NHWC tensor stored in frames of Hp x Wp pixels whose valid part is H x W
__global__ void cv_zero_margin_kernel(uint4* __restrict__ t, int N, int H, int W, int Hp, int Wp, int chunks) {
  const int right = H * (Wp - W), all = right + (Hp - H) * Wp;
  const long long total = (long long)N * all * chunks;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % chunks);
    const long long r = i / chunks;
    const int m = (int)(r % all);
    const long long n = r / all;
    const int pp = m < right ? (m / (Wp - W)) * Wp + W + m % (Wp - W) : H * Wp + (m - right);
    t[(n * Hp * Wp + pp) * chunks + c] = make_uint4(0, 0, 0, 0);
  }
}

int conv_dgrad2_fused(const void* dy2b, int N, int H1, int W1, int H2, int W2, const void* wp5, const void* y1b, void* dy1b,
                      int out_pad, cudaStream_t st) {
  if (N == 0) return 0;
  CUtensorMap tw, ta;
  int rc = cv_weight_tmap(&tw, wp5, 4, 128);
  if (rc) return rc;
  TACORL_REQUIRE(((uintptr_t)dy2b & 15) == 0, "conv_dgrad2: dy2 must be 16-byte aligned");
  const cuuint64_t dims[4] = {64, (cuuint64_t)W2, (cuuint64_t)H2, (cuuint64_t)N};
  const cuuint64_t strides[3] = {128, (cuuint64_t)W2 * 128, (cuuint64_t)H2 * W2 * 128};
  const cuuint32_t box[4] = {64, DG_PW, DG_PH, 1};
  if ((rc = encode_tmap_bf16(&ta, "conv_dgrad2(dy2)", 4, dy2b, dims, strides, box))) return rc;
  Dgrad2Geom g = {};
  g.H1 = H1; g.W1 = W1; g.H2 = H2; g.W2 = W2; g.RA = (H1 + 1) / 2; g.RB = (W1 + 1) / 2;
  g.tiles_x = cdiv(g.RB, DG_PW - 1); g.tiles_y = cdiv(g.RA, DG_PH - 1);
  g.num_tiles = N * g.tiles_x * g.tiles_y;
  g.OHp = H1 + out_pad; g.OWp = W1 + out_pad;
  if (out_pad > 0) {
    const long long total = (long long)N * (H1 * out_pad + out_pad * g.OWp) * 4;
    cv_zero_margin_kernel<<<(int)min((long long)592, (total + 255) / 256), 256, 0, st>>>((uint4*)dy1b, N, H1, W1, g.OHp, g.OWp, 4);
    TACORL_LAUNCH_CHECK();
  }
  const size_t smem = 4 * 128 * 128 + (size_t)(DG_STAGES + 1) * 128 * 128 + (2 * DG_STAGES + 5) * 8 + 16 + 1024;
  static bool configured = false;
  if (!configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(conv_dgrad2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int ctas = g.num_tiles < persistent_ctas() ? g.num_tiles : persistent_ctas();
  conv_dgrad2_kernel<<<ctas, DG_THREADS, smem, st>>>(g, ta, tw, (const __nv_bfloat16*)y1b, (__nv_bfloat16*)dy1b);
  TACORL_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------ packing kernels
// mode 0: conv3 fwd   Wp[t=(ky,kx)][oc][c]            = W3[oc][c][ky][kx]            (9 taps, BN=64)
// mode 1: conv2 fwd   Wp[t=(ky,p)][oc][(kx-2p)*32+c]  = W2[oc][c][ky][kx]            (8 tap pairs, BN=64)
// mode 2: conv1 fwd   Wp[t=(dy,dx)][oc][q]            = W1[oc][c][4dy+py][4dx+px], q=(py*4+px)*3+c (<48, else 0)  (4 taps, BN=32)
// mode 3: conv3 dgrad Wp[t=(ky,kx)][c][oc]            = W3[oc][c][ky][kx]            (9 taps, BN=64)
// mode 4: conv2 dgrad Wp[cls=(py,px)][t=(j,i)][c][oc] = W2[oc][c][py+2j][px+2i]      (4 classes x 4 taps, BN=32)
// mode 5: conv2 dgrad Wp[t=(j,i)][cls*32 + c][oc]     = W2[oc][c][py+2j][px+2i]      (4 taps, BN=128: all classes fused)
struct PackJobs {
  int n;
  int mode[3];
  const float* W[3];
  __nv_bfloat16* Wp[3];
  int total[3];
};
// one launch packs up to three weight tensors (blockIdx.y = job): the 3 forward / 2 backward packs of an encoder pass
__global__ void cv_pack_kernel(const PackJobs jobs) {
  const int job = blockIdx.y;
  const int mode = jobs.mode[job], total = jobs.total[job];
  const float* __restrict__ W = jobs.W[job];
  __nv_bfloat16* __restrict__ Wp = jobs.Wp[job];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int k = i & 63;
  float v = 0.f;
  if (mode == 0) {
    const int oc = (i >> 6) & 63, t = i >> 12, ky = t / 3, kx = t % 3;
    v = W[((oc * 64 + k) * 3 + ky) * 3 + kx];
  } else if (mode == 1) {
    const int oc = (i >> 6) & 63, t = i >> 12, ky = t >> 1, p = t & 1, kx = 2 * p + (k >> 5), c = k & 31;
    v = W[((oc * 32 + c) * 4 + ky) * 4 + kx];
  } else if (mode == 2) {
    const int oc = (i >> 6) & 31, t = i >> 11, dy = t >> 1, dx = t & 1;
    if (k < 48) {
      const int c = k % 3, pp = k / 3, py = pp >> 2, px = pp & 3;
      v = W[((oc * 3 + c) * 8 + (4 * dy + py)) * 8 + (4 * dx + px)];
    }
  } else if (mode == 3) {
    const int c = (i >> 6) & 63, t = i >> 12, ky = t / 3, kx = t % 3;
    v = W[((k * 64 + c) * 3 + ky) * 3 + kx];
  } else if (mode == 4) {
    const int c = (i >> 6) & 31, t = (i >> 11) & 3, cls = i >> 13, py = cls >> 1, px = cls & 1, j = t >> 1, ii = t & 1;
    v = W[((k * 32 + c) * 4 + (py + 2 * j)) * 4 + (px + 2 * ii)];
  } else {
    const int nn = (i >> 6) & 127, t = i >> 13, cls = nn >> 5, c = nn & 31, py = cls >> 1, px = cls & 1, j = t >> 1, ii = t & 1;
    v = W[((k * 32 + c) * 4 + (py + 2 * j)) * 4 + (px + 2 * ii)];
  }
  Wp[i] = __float2bfloat16(v);
}

int conv_tc_pack_multi(int n, const int* modes, const float* const* Ws, void* const* Wps, cudaStream_t st) {
  static const int totals[6] = {9 * 64 * 64, 8 * 64 * 64, 4 * 32 * 64, 9 * 64 * 64, 16 * 32 * 64, 4 * 128 * 64};
  TACORL_REQUIRE(n >= 1 && n <= 3, "conv_tc_pack: 1..3 tensors per launch");
  PackJobs jobs;
  jobs.n = n;
  int most = 0;
  for (int j = 0; j < n; ++j) {
    TACORL_REQUIRE(modes[j] >= 0 && modes[j] < 6, "conv_tc_pack: bad mode");
    jobs.mode[j] = modes[j]; jobs.W[j] = Ws[j]; jobs.Wp[j] = (__nv_bfloat16*)Wps[j]; jobs.total[j] = totals[modes[j]];
    most = max(most, totals[modes[j]]);
  }
  cv_pack_kernel<<<dim3(cdiv(most, 256), n), 256, 0, st>>>(jobs);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int conv_tc_pack(int mode, const float* W, void* Wp, cudaStream_t st) {
  return conv_tc_pack_multi(1, &mode, &W, &Wp, st);
}

// fp32 NCHW image (N,3,H,W) -> bf16 space-to-depth(4) (N, SH, SW, 64), channel q = (py*4+px)*3 + c for q < 48, zero pad
// above (128-byte pixels = one TMA / UMMA swizzle row).  One thread per (n, Y, X, py): three float4 loads, 12 bf16 out.
__global__ void cv_s2d_kernel(const float* __restrict__ x, int H, int W, int SH, int SW, long long total,
                              __nv_bfloat16* __restrict__ xs) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int py = (int)(i & 3);
    long long t = i >> 2;
    const int X = (int)(t % SW); t /= SW;
    const int Y = (int)(t % SH);
    const long long n = t / SH;
    const int iy = 4 * Y + py;
    float4 c0 = make_float4(0, 0, 0, 0), c1 = c0, c2 = c0;
    if (iy < H && 4 * X + 3 < W) {
      const float* p = x + ((n * 3) * H + iy) * (long long)W + 4 * X;
      c0 = __ldg(reinterpret_cast<const float4*>(p));
      c1 = __ldg(reinterpret_cast<const float4*>(p + (long long)H * W));
      c2 = __ldg(reinterpret_cast<const float4*>(p + 2LL * H * W));
    }
    __nv_bfloat16* o = xs + ((n * SH + Y) * (long long)SW + X) * 64 + py * 12;
    if (py == 0) {                                      // channels 48..63 of the pixel
      reinterpret_cast<uint4*>(o + 48)[0] = make_uint4(0, 0, 0, 0);
      reinterpret_cast<uint4*>(o + 48)[1] = make_uint4(0, 0, 0, 0);
    }
    const float v[12] = {c0.x, c1.x, c2.x, c0.y, c1.y, c2.y, c0.z, c1.z, c2.z, c0.w, c1.w, c2.w};
    uint32_t pk[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      __nv_bfloat162 t2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      pk[j] = *reinterpret_cast<uint32_t*>(&t2);
    }
    uint2* op = reinterpret_cast<uint2*>(o);          // 24-byte run, 8-byte aligned
    op[0] = make_uint2(pk[0], pk[1]); op[1] = make_uint2(pk[2], pk[3]); op[2] = make_uint2(pk[4], pk[5]);
  }
}

// uint8 NCHW frames: scale/normalise (v = u8*scale + shift, i.e. ScaleImageTensor + Normalize of
// /root/reference/src/tacorl/utils/transforms.py:87-101 fused into the load) and space-to-depth in one pass.
// (Tried and measured slower, round 2: staging 40 input rows per CTA through shared memory for fully coalesced loads --
// the byte gathers out of shared memory cost more than the 32-byte global segments do: 233 us against 125 us.)
__global__ void cv_s2d_u8_kernel(const unsigned char* __restrict__ x, int H, int W, int SH, int SW, long long total,
                                 float scale, float shift, __nv_bfloat16* __restrict__ xs) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int py = (int)(i & 3);
    long long t = i >> 2;
    const int X = (int)(t % SW); t /= SW;
    const int Y = (int)(t % SH);
    const long long n = t / SH;
    const int iy = 4 * Y + py;
    float v[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) v[j] = 0.f;
    if (iy < H && 4 * X + 3 < W) {
      const unsigned char* p = x + ((n * 3) * H + iy) * (long long)W + 4 * X;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const uchar4 u = __ldg(reinterpret_cast<const uchar4*>(p + (long long)c * H * W));
        v[c] = fmaf((float)u.x, scale, shift); v[3 + c] = fmaf((float)u.y, scale, shift);
        v[6 + c] = fmaf((float)u.z, scale, shift); v[9 + c] = fmaf((float)u.w, scale, shift);
      }
    }
    __nv_bfloat16* o = xs + ((n * SH + Y) * (long long)SW + X) * 64 + py * 12;
    if (py == 0) {
      reinterpret_cast<uint4*>(o + 48)[0] = make_uint4(0, 0, 0, 0);
      reinterpret_cast<uint4*>(o + 48)[1] = make_uint4(0, 0, 0, 0);
    }
    uint32_t pk[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      __nv_bfloat162 t2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      pk[j] = *reinterpret_cast<uint32_t*>(&t2);
    }
    uint2* op = reinterpret_cast<uint2*>(o);
    op[0] = make_uint2(pk[0], pk[1]); op[1] = make_uint2(pk[2], pk[3]); op[2] = make_uint2(pk[4], pk[5]);
  }
}

int conv_tc_s2d_u8(const unsigned char* x, int N, int H, int W, int SH, int SW, float scale, float shift, void* xs,
                   cudaStream_t st) {
  TACORL_REQUIRE(W % 4 == 0 && ((uintptr_t)x & 3) == 0, "conv_tc_s2d_u8: image width must be a multiple of 4");
  const long long total = (long long)N * SH * SW * 4;
  if (total == 0) return 0;
  cv_s2d_u8_kernel<<<(int)min((long long)148 * 16, (total + 255) / 256), 256, 0, st>>>(x, H, W, SH, SW, total, scale,
                                                                                     shift, (__nv_bfloat16*)xs);
  TACORL_LAUNCH_CHECK();
  return 0;
}

__global__ void cv_u8_to_f32_kernel(long long n, const unsigned char* __restrict__ x, float scale, float shift,
                                    float* __restrict__ o) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    o[i] = fmaf((float)x[i], scale, shift);
}

int u8_to_f32_normalized(long long n, const unsigned char* x, float scale, float shift, float* out, cudaStream_t st) {
  if (n == 0) return 0;
  cv_u8_to_f32_kernel<<<(int)min((long long)148 * 16, (n + 255) / 256), 256, 0, st>>>(n, x, scale, shift, out);
  TACORL_LAUNCH_CHECK();
  return 0;
}

int conv_tc_s2d(const float* x, int N, int H, int W, int SH, int SW, void* xs, cudaStream_t st) {
  TACORL_REQUIRE(W % 4 == 0 && ((uintptr_t)x & 15) == 0, "conv_tc_s2d: image width must be a multiple of 4");
  const long long total = (long long)N * SH * SW * 4;
  if (total == 0) return 0;
  cv_s2d_kernel<<<(int)min((long long)148 * 16, (total + 255) / 256), 256, 0, st>>>(x, H, W, SH, SW, total,
                                                                                  (__nv_bfloat16*)xs);
  TACORL_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------ layer drivers
static ActView cv_plain_view(const void* base, int N, int H, int W) {      // NHWC, 64 channels (128-byte pixels)
  return ActView{base, W, 1, H, N, 128, 128, (long long)W * 128, (long long)H * W * 128};
}
// conv1 forward on the s2d image (N, H1+1, W1+1, 64: 48 real channels + zero pad): 2x2 taps, stride 1, BN = 32
int conv_tc_conv1_fwd(const void* xs, int N, int H1, int W1, const void* wp, const float* bias, void* y1b,
                      cudaStream_t st) {
  ConvGeom g = {};
  g.RA = H1; g.RB = W1; g.ntaps = 4;
  for (int t = 0; t < 4; ++t) { g.tap_y[t] = t >> 1; g.tap_x[t] = t & 1; }
  g.OH = H1; g.OW = W1; g.oys = 1; g.oxs = 1;
  ConvEpi e = {bias, 1, nullptr, (__nv_bfloat16*)y1b, nullptr};
  return conv_tc_run(g, N, cv_plain_view(xs, N, H1 + 1, W1 + 1), 32, wp, e, st);
}
// conv2 forward: 4x4 stride 2 over y1 (N, H1, W1, 32).  Source pixel (2a+ky, 2b+kx): y1 is viewed as
// (64 = pixel pair x 32 channels, pair index, row parity, row pair, frame), tap (ky, p) = box at pair b+p, row 2(a + ky/2) + ky%2.
int conv_tc_conv2_fwd(const void* y1b, int N, int H1, int W1, int H2, int W2, const void* wp, const float* bias,
                      void* y2b, cudaStream_t st) {
  ConvGeom g = {};
  g.RA = H2; g.RB = W2; g.ntaps = 8;
  for (int t = 0; t < 8; ++t) { const int ky = t >> 1; g.tap_x[t] = t & 1; g.tap_p[t] = ky & 1; g.tap_y[t] = ky >> 1; }
  g.OH = H2; g.OW = W2; g.oys = 1; g.oxs = 1;
  ConvEpi e = {bias, 1, nullptr, (__nv_bfloat16*)y2b, nullptr};
  const ActView v{y1b, W2 + 1, 2, H2 + 1, N, 128, (long long)W1 * 64, (long long)W1 * 128, (long long)H1 * W1 * 64};
  return conv_tc_run(g, N, v, 64, wp, e, st);
}
// conv3 forward: 3x3 stride 1 over y2 (C = 64): 9 taps; fp32 output for the soft-argmax
int conv_tc_conv3_fwd(const void* y2b, int N, int H2, int W2, int H3, int W3, const void* wp, const float* bias,
                      float* y3, cudaStream_t st) {
  ConvGeom g = {};
  g.RA = H3; g.RB = W3; g.ntaps = 9;
  for (int t = 0; t < 9; ++t) { g.tap_y[t] = t / 3; g.tap_x[t] = t % 3; }
  g.OH = H3; g.OW = W3; g.oys = 1; g.oxs = 1;
  ConvEpi e = {bias, 1, nullptr, nullptr, y3};
  return conv_tc_run(g, N, cv_plain_view(y2b, N, H2, W2), 64, wp, e, st);
}
// conv3 dgrad: dy2[iy][ix][c] = [y2>0] * sum_{ky,kx,oc} dy3[iy-ky][ix-kx][oc] W3[oc][c][ky][kx]   (TMA zero-fills iy-ky < 0 ...)
int conv_tc_conv3_dgrad(const void* dy3b, int N, int H2, int W2, int H3, int W3, const void* wp, const void* y2b,
                        void* dy2b, cudaStream_t st) {
  ConvGeom g = {};
  g.RA = H2; g.RB = W2; g.ntaps = 9;
  for (int t = 0; t < 9; ++t) { g.tap_y[t] = -(t / 3); g.tap_x[t] = -(t % 3); }
  g.OH = H2; g.OW = W2; g.oys = 1; g.oxs = 1;
  ConvEpi e = {nullptr, 0, (const __nv_bfloat16*)y2b, (__nv_bfloat16*)dy2b, nullptr};
  return conv_tc_run(g, N, cv_plain_view(dy3b, N, H3, W3), 64, wp, e, st);
}
// conv2 dgrad: four stride-parity classes (py,px); class rows (a,b) -> dy1 pixel (2a+py, 2b+px),
//   dy1 = [y1>0] * sum_{j,i in {0,1}, oc} dy2[a-j][b-i][oc] W2[oc][c][py+2j][px+2i]
int conv_tc_conv2_dgrad(const void* dy2b, int N, int H1, int W1, int H2, int W2, const void* wp_classes,
                        const void* y1b, void* dy1b, cudaStream_t st) {
  for (int cls = 0; cls < 4; ++cls) {
    const int py = cls >> 1, px = cls & 1;
    ConvGeom g = {};
    g.RA = (H1 - py + 1) / 2; g.RB = (W1 - px + 1) / 2; g.ntaps = 4;
    for (int t = 0; t < 4; ++t) { g.tap_y[t] = -(t >> 1); g.tap_x[t] = -(t & 1); }
    g.OH = H1; g.OW = W1; g.oys = 2; g.oy0 = py; g.oxs = 2; g.ox0 = px;
    ConvEpi e = {nullptr, 0, (const __nv_bfloat16*)y1b, (__nv_bfloat16*)dy1b, nullptr};
    int rc = conv_tc_run(g, N, cv_plain_view(dy2b, N, H2, W2), 32,
                         (const __nv_bfloat16*)wp_classes + (size_t)cls * 4 * 32 * 64, e, st);
    if (rc) return rc;
  }
  return 0;
}

}  // namespace tacorl

// ==========================================================================================
// Weight gradients: dW[oc][tap][c] = sum over output pixels m of dY[m][oc] * X[src_pixel(m, tap)][c].
// Pixels are the UMMA K dimension, so both operands are MN-major tiles of 64 pixel rows x 128 bytes:
//   A = dY rows (OC channels, zero-filled to 128 B), padded to M = 128 with a shared all-zero tile,
//   B = NT gathered activation tiles (one per tap / tap pair), N = NT*64 accumulator columns.
// Each CTA owns one tap group and one slice of the pixel range; partial sums go to a workspace and a small
// kernel reduces the slices and scatters into the torch weight-gradient layout.
namespace tacorl {

constexpr int WG_STAGES = 5;
constexpr int WG_PL = 4;              // producer lanes per pixel row (chunks j = c*WG_PL + h: whole 32-byte sectors per warp instruction)
constexpr int WG_PROD = 64 * WG_PL;   // producer threads; warps 0..3 also drain TMEM at the end
constexpr int WG_THREADS = WG_PROD + 32;   // + the MMA warp

struct WgradGeom {
  const __nv_bfloat16* dy;            // (M, OC) output gradient, NHWC rows
  int OC, dy_chunks;                  // OC*2/16 valid chunks per dY row
  const __nv_bfloat16* src;           // NHWC source activation (N, SH, SW, SC)
  int SH, SW, SC, kchunks;
  int RA, RB, M;                      // output pixel grid per frame, total rows
  int sy, sx;
  int NT;                             // taps per CTA (N = NT*64)
  int groups;                         // tap groups (gridDim.y)
  int dy_t[CV_MAXT], dx_t[CV_MAXT], coff[CV_MAXT];   // per (group*NT + j) source offsets
  int rows_per_split;                 // multiple of 64
  float* partial;                     // [splits][groups][OC][NT*64]
  float* bias_partial;                // [splits][OC] column sums of dY (bias gradient), written by group 0; may be null
};

__global__ void __launch_bounds__(WG_THREADS, 1) conv_tc_wgrad_kernel(const __grid_constant__ WgradGeom g) {
  constexpr uint32_t TILE = 64 * 128;                   // one 64-row x 128-byte MN-major tile
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t stage_bytes = (1 + g.NT) * TILE;
  const uint32_t base = smem_u32(smem);
  const uint32_t zero_tile = base + WG_STAGES * stage_bytes;
  const uint32_t ones_tile = zero_tile + TILE;          // all-ones B operand: dY^T x 1 = bias gradient
  uint64_t* bars = (uint64_t*)(smem + WG_STAGES * stage_bytes + 2 * TILE);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * WG_STAGES + 1);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + WG_STAGES + s); };
  const uint32_t done_bar = smem_u32(bars + 2 * WG_STAGES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int NCOLS = g.NT * 64;
  const bool with_bias = g.bias_partial != nullptr && blockIdx.y == 0;
  const int acc_cols = NCOLS + 16;                      // + one N = 16 accumulator block for the bias gradient
  const uint32_t tmem_cols = acc_cols <= 128 ? 128 : (acc_cols <= 256 ? 256 : 512);

  const int m_begin = blockIdx.x * g.rows_per_split;
  const int m_end = min(g.M, m_begin + g.rows_per_split);
  const int nkb = m_end > m_begin ? (m_end - m_begin + 63) / 64 : 0;
  const int grp = blockIdx.y;
  const int rows_per_frame = g.RA * g.RB;

  // zero tile (upper half of the M = 128 A operand)
  for (int i = threadIdx.x; i < (int)(TILE / 16); i += blockDim.x) {
    reinterpret_cast<uint4*>(smem + WG_STAGES * stage_bytes)[i] = make_uint4(0, 0, 0, 0);
    reinterpret_cast<uint4*>(smem + WG_STAGES * stage_bytes + TILE)[i] =
        make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);          // bf16 1.0 pairs
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < WG_STAGES; ++s) { mbar_init(full_bar(s), WG_PROD); mbar_init(empty_bar(s), 1); }
    mbar_init(done_bar, 1);
    mbar_init_fence();
  }
  if (warp == WG_PROD / 32) tmem_alloc(tmem_slot, tmem_cols);
  cv_fence_async();          // the generic-proxy zero fill must be visible to the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < WG_PROD / 32) {
    // WG_PL lanes gather pixel row p of the K block; lane h takes the 16-byte chunks c*WG_PL + h
    const int h = threadIdx.x % WG_PL, p = threadIdx.x / WG_PL;
    const uint32_t row_off = (uint32_t)p * 128, sw = (uint32_t)(p & 7);
    for (int i = 0; i < nkb; ++i) {
      const int s = i % WG_STAGES;
      const uint32_t ph = (i / WG_STAGES) & 1;
      mbar_wait(empty_bar(s), ph ^ 1);
      const uint32_t st = base + s * stage_bytes;
      const int m = m_begin + i * 64 + p;
      const bool ok = m < m_end;
      int n = 0, a = 0, b = 0;
      if (ok) { n = m / rows_per_frame; const int rem = m - n * rows_per_frame; a = rem / g.RB; b = rem - a * g.RB; }
      const __nv_bfloat16* dyp = g.dy + (long long)(ok ? m : 0) * g.OC;
#pragma unroll
      for (int c = 0; c < 8 / WG_PL; ++c) {
        const int j = WG_PL * c + h;
        cv_cp16(st + row_off + ((j ^ sw) << 4), dyp + j * 8, (ok && j < g.dy_chunks) ? 16u : 0u);
      }
      const __nv_bfloat16* frame = g.src + (long long)n * g.SH * g.SW * g.SC;
      for (int t = 0; t < g.NT; ++t) {
        const int tt = grp * g.NT + t;
        const __nv_bfloat16* sp = frame + ((long long)(a * g.sy + g.dy_t[tt]) * g.SW + (b * g.sx + g.dx_t[tt])) * g.SC + g.coff[tt];
        const uint32_t dst = st + (1 + t) * TILE + row_off;
#pragma unroll
        for (int c = 0; c < 8 / WG_PL; ++c) {
          const int j = WG_PL * c + h;
          cv_cp16(dst + ((j ^ sw) << 4), sp + j * 8, (ok && j < g.kchunks) ? 16u : 0u);
        }
      }
      cv_cp_async_arrive(full_bar(s));
    }
  } else if (warp == WG_PROD / 32) {
    if (lane == 0 && nkb > 0) {
      const uint32_t idesc = idesc_bf16(128, NCOLS, true, true);
      constexpr uint32_t idesc_b = idesc_bf16(128, 16, true, true);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % WG_STAGES;
        const uint32_t ph = (i / WG_STAGES) & 1;
        mbar_wait(full_bar(s), ph);
        cv_fence_async();
        tc_fence_after();
        const uint32_t a_src = base + s * stage_bytes, b_src = a_src + TILE;
#pragma unroll
        for (int k = 0; k < 4; ++k)     // 16 pixel rows (2048 B) per UMMA K step
          tc_mma_bf16(tmem_base, smem_desc(a_src + k * 2048, zero_tile - a_src, 1024), smem_desc(b_src + k * 2048, TILE, 1024),
                      idesc, (i > 0 || k > 0) ? 1u : 0u);
        if (with_bias) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            tc_mma_bf16(tmem_base + NCOLS, smem_desc(a_src + k * 2048, zero_tile - a_src, 1024),
                        smem_desc(ones_tile, TILE, 1024), idesc_b, (i > 0 || k > 0) ? 1u : 0u);
        }
        tc_commit(empty_bar(s));
      }
      tc_commit(done_bar);
    }
  }
  if (warp < 4) {   // the producer warps drain the accumulator: TMEM lane quarter = warp index
    const int q = warp;
    const int oc = q * 32 + lane;
    if (nkb > 0) { mbar_wait(done_bar, 0); tc_fence_after(); }
    float* P = g.partial + (((long long)blockIdx.x * g.groups + grp) * g.OC + oc) * NCOLS;
    if (q * 32 < g.OC) {
      for (int c0 = 0; c0 < NCOLS; c0 += 16) {
        uint32_t r[16];
        if (nkb > 0) tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r);
        else {
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = 0;
        }
        if (oc < g.OC) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            reinterpret_cast<float4*>(P + c0)[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                               __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
        }
      }
      if (with_bias) {
        uint32_t r[16];
        if (nkb > 0) tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + NCOLS, r);
        else r[0] = 0;
        if (oc < g.OC) g.bias_partial[(long long)blockIdx.x * g.OC + oc] = __uint_as_float(r[0]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == WG_PROD / 32) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// dW (torch layout) = beta*dW + sum over splits of partial, with the per-layer column -> (c, ky, kx) mapping
// layer 3: groups = 3 (ky), col = kx*64 + c;  layer 2: groups = 2, col = (kyl*2 + p)*64 + k, ky = 2g+kyl, kx = 2p+(k>>5), c = k&31;
// layer 1: groups = 1, col = t*64 + q (q < 48), t = (dy,dx), q = (py*4+px)*3 + c, ky = 4dy+py, kx = 4dx+px.
__global__ void conv_tc_wgrad_reduce_kernel(int layer, int splits, int groups, int OC, int NCOLS,
                                            const float* __restrict__ partial, float beta, float* __restrict__ dW,
                                            const float* __restrict__ bias_partial, float* __restrict__ db) {
  const int total = groups * OC * NCOLS;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) {
    const int oc = i - total;
    if (db && oc < OC) {
      float s = 0.f;
      for (int z = 0; z < splits; ++z) s += bias_partial[(long long)z * OC + oc];
      db[oc] = beta != 0.f ? fmaf(beta, db[oc], s) : s;
    }
    return;
  }
  const int col = i % NCOLS, oc = (i / NCOLS) % OC, grp = i / (NCOLS * OC);
  int idx = -1;
  if (layer == 3) {
    const int kx = col >> 6, c = col & 63;
    idx = ((oc * 64 + c) * 3 + grp) * 3 + kx;
  } else if (layer == 2) {
    const int k = col & 63, tp = col >> 6, kyl = tp >> 1, p = tp & 1;
    idx = ((oc * 32 + (k & 31)) * 4 + (2 * grp + kyl)) * 4 + (2 * p + (k >> 5));
  } else {
    const int q = col & 63, t = col >> 6;
    if (q < 48) {
      const int c = q % 3, pp = q / 3, py = pp >> 2, px = pp & 3;
      idx = ((oc * 3 + c) * 8 + (4 * (t >> 1) + py)) * 8 + (4 * (t & 1) + px);
    }
  }
  if (idx < 0) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += partial[(((long long)z * groups + grp) * OC + oc) * NCOLS + col];
  dW[idx] = beta != 0.f ? fmaf(beta, dW[idx], s) : s;
}

// layer: 1 (conv1 on the s2d image), 2, 3.  dyb: (N*RA*RB, OC) bf16; src: NHWC bf16 input activation of the layer.
// db (optional): bias gradient = column sums of dyb, from an extra N = 16 MMA against an all-ones operand.
int conv_tc_wgrad(int layer, const void* dyb, const void* src, int N, int SH, int SW, int RA, int RB, float beta,
                  float* dW, float* db, float* ws, size_t ws_bytes, cudaStream_t st) {
  WgradGeom g = {};
  g.dy = (const __nv_bfloat16*)dyb; g.src = (const __nv_bfloat16*)src;
  g.SH = SH; g.SW = SW; g.RA = RA; g.RB = RB; g.M = N * RA * RB;
  if (layer == 3) {
    g.OC = 64; g.SC = 64; g.kchunks = 8; g.sy = g.sx = 1; g.NT = 3; g.groups = 3;
    for (int t = 0; t < 9; ++t) { g.dy_t[t] = t / 3; g.dx_t[t] = t % 3; g.coff[t] = 0; }
  } else if (layer == 2) {
    g.OC = 64; g.SC = 32; g.kchunks = 8; g.sy = g.sx = 2; g.NT = 4; g.groups = 2;
    for (int t = 0; t < 8; ++t) { g.dy_t[t] = t >> 1; g.dx_t[t] = 2 * (t & 1); g.coff[t] = 0; }
  } else {
    g.OC = 32; g.SC = 64; g.kchunks = 6; g.sy = g.sx = 1; g.NT = 4; g.groups = 1;
    for (int t = 0; t < 4; ++t) { g.dy_t[t] = t >> 1; g.dx_t[t] = t & 1; g.coff[t] = 0; }
  }
  g.dy_chunks = g.OC / 8;
  if (g.M == 0) return 0;
  const int NCOLS = g.NT * 64;
  int splits = persistent_ctas() / g.groups;
  const int kblocks = (g.M + 63) / 64;
  if (splits > kblocks) splits = kblocks;
  const size_t per_split = ((size_t)g.groups * g.OC * NCOLS + g.OC) * sizeof(float);
  if ((size_t)splits * per_split > ws_bytes) splits = (int)(ws_bytes / per_split);
  TACORL_REQUIRE(ws && splits >= 1, "conv_tc_wgrad: workspace too small");
  g.rows_per_split = ((kblocks + splits - 1) / splits) * 64;
  splits = (g.M + g.rows_per_split - 1) / g.rows_per_split;
  g.partial = ws;
  g.bias_partial = db ? ws + (size_t)splits * g.groups * g.OC * NCOLS : nullptr;
  const size_t smem = (size_t)WG_STAGES * (1 + g.NT) * 8192 + 2 * 8192 + (2 * WG_STAGES + 1) * 8 + 16 + 1024;
  static size_t configured = 0;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  conv_tc_wgrad_kernel<<<dim3(splits, g.groups), WG_THREADS, smem, st>>>(g);
  TACORL_LAUNCH_CHECK();
  const int total = g.groups * g.OC * NCOLS;
  conv_tc_wgrad_reduce_kernel<<<cdiv(total + g.OC, 256), 256, 0, st>>>(layer, splits, g.groups, g.OC, NCOLS, ws, beta, dW,
                                                                       g.bias_partial, db);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // namespace tacorl

// ==========================================================================================
// Linear-shift weight gradient (stride-1 layers whose source and gradient tensors share one pixel-row pitch).
//   dW[oc][c][ky][kx] = sum_p dY[p][oc] * X[p + ky*W + kx][c],   p = linear pixel row over all frames
// holds when dY is stored at the SOURCE's row pitch W with zeros at the positions that are not outputs (the right /
// bottom margin of every frame): a zero gradient row contributes nothing, whatever source row it is paired with.  Then a
// K block of the implicit GEMM is simply 128 consecutive pixel rows: ONE TMA box of the source and one of dY per stage,
// and the taps are UMMA descriptors into those two windows -- no per-tap gathers (the cp.async kernel above moves each
// source row once per tap and each dY row once per tap group through the LSU).  Both operands are MN-major (pixels = K)
// and the M / N atoms of a descriptor OVERLAP in shared memory: their stride is a row shift, not a tile size.
//   B = source rows, N = 192 = the three taps kx = 0, 1, 2 of one kernel row: N-atom stride = 1 pixel row (128 bytes);
//   A = dY rows,     M = 128 = two kernel rows: M-atom 0 = dY[p], M-atom 1 = dY[p + W] (stride = W pixel rows), because
//       sum_p dY[p + W][oc] X[p + s][c] = sum_p' dY[p'][oc] X[p' + s - W][c] is the tap one kernel row above.
// Two MMAs per 16 pixel rows cover all nine taps: D0 (B shifted by W) = taps ky = 1 (lanes 0-63) and ky = 0 (lanes
// 64-127), D1 (B shifted by 2 W) = taps ky = 2 (lanes 0-63).  A third, N = 16 against an all-ones tile, is the bias
// gradient.  The pixel range starts at p = -W (TMA zero-fills negative rows) so that M-atom 1 sees every gradient row.
// fp32 accumulators stay in TMEM over the CTA's whole pixel range; partials -> fixed-order reduction kernel.
namespace tacorl {

constexpr int WL_KB = 128;          // pixel rows per K block
constexpr int WL_MAX_STAGES = 5;
constexpr int WL_THREADS = 192;     // warp 0: TMA, warp 1: MMA issue, warps 2-5: TMEM drain
constexpr int WL_COLS = 192 + 192 + 16;   // accumulator columns: D0 | D1 | bias

struct WgradLinGeom {
  int nkb;                          // K blocks in total (pixel rows -W .. rows-1)
  int kb_per_cta;
  int W;                            // row pitch of both tensors (pixels)
  int src_rows, dy_rows;            // rows per stage window (multiples of 8)
  int stages;                       // smem ring depth (2 .. WL_MAX_STAGES)
  float* partial;                   // [ctas][128 lanes][WL_COLS]
};

__global__ void __launch_bounds__(WL_THREADS, 1)
conv_wgrad_lin_kernel(const __grid_constant__ WgradLinGeom g, const __grid_constant__ CUtensorMap tmS,
                      const __grid_constant__ CUtensorMap tmD) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t src_bytes = (uint32_t)g.src_rows * 128, dy_bytes = (uint32_t)g.dy_rows * 128;   // multiples of 1024
  const uint32_t stage_bytes = src_bytes + dy_bytes;
  const uint32_t base = smem_u32(smem);
  const int WL_STAGES = g.stages;
  const uint32_t ones_tile = base + WL_STAGES * stage_bytes;       // 16 K rows x 128 B of bf16 1.0 (N = 16 uses 32 B of each)
  uint64_t* bars = (uint64_t*)(smem + WL_STAGES * stage_bytes + 2048);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * WL_MAX_STAGES + 1);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + WL_MAX_STAGES + s); };
  const uint32_t done_bar = smem_u32(bars + 2 * WL_MAX_STAGES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb_begin = blockIdx.x * g.kb_per_cta;
  const int kb_end = min(g.nkb, kb_begin + g.kb_per_cta);
  const int nkb = max(0, kb_end - kb_begin);

  for (int i = threadIdx.x; i < 2048 / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem + WL_STAGES * stage_bytes)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
  if (threadIdx.x == 0) {
    for (int s = 0; s < WL_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(done_bar, 1);
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  cv_fence_async();          // the generic-proxy fill of the ones tile must be visible to the tensor core
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % WL_STAGES;
        mbar_wait(empty_bar(s), ((i / WL_STAGES) & 1) ^ 1);
        const uint32_t st = base + s * stage_bytes;
        const int row0 = (kb_begin + i) * WL_KB;                   // source window starts at pixel row p0 + W = row0
        mbar_expect_tx(full_bar(s), src_bytes + dy_bytes);
        tma_load_2d(st, &tmS, 0, row0, full_bar(s));                 // rows outside the tensor arrive as zeros
        tma_load_2d(st + src_bytes, &tmD, 0, row0 - g.W, full_bar(s));
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && nkb > 0) {
      constexpr uint32_t idesc = idesc_bf16(128, 192, true, true), idesc_b = idesc_bf16(128, 16, true, true);
      const uint64_t ones_desc = smem_desc(ones_tile, 128, 1024);
      const uint32_t wrow = (uint32_t)g.W * 128;
      const uint64_t b0 = smem_desc(base, 128, 1024);                       // N-atom stride: one pixel row
      const uint64_t a0 = smem_desc(base + src_bytes, wrow, 1024);          // M-atom stride: one image row
      for (int i = 0; i < nkb; ++i) {
        const int s = i % WL_STAGES;
        mbar_wait(full_bar(s), (i / WL_STAGES) & 1);
        tc_fence_after();
        const uint64_t so = (uint64_t)((s * stage_bytes) >> 4);
#pragma unroll
        for (int k = 0; k < WL_KB / 16; ++k) {      // 16 pixel rows (2048 B) per UMMA K step
          const uint32_t acc = (i > 0 || k > 0) ? 1u : 0u;
          const uint64_t ad = a0 + so + (uint64_t)(k * 128), bd = b0 + so + (uint64_t)(k * 128);
          tc_mma_bf16(tmem_base, ad, bd, idesc, acc);
          tc_mma_bf16(tmem_base + 192, ad, bd + (uint64_t)(wrow >> 4), idesc, acc);
          tc_mma_bf16(tmem_base + 384, ad, ones_desc, idesc_b, acc);
        }
        tc_commit(empty_bar(s));
      }
      tc_commit(done_bar);
    }
  } else {
    const int q = warp & 3;                     // TMEM lane quarter this warp may read
    if (nkb > 0) { mbar_wait(done_bar, 0); tc_fence_after(); }
    float* P = g.partial + ((long long)blockIdx.x * 128 + (q * 32 + lane)) * WL_COLS;
#pragma unroll 1
    for (int c0 = 0; c0 < WL_COLS; c0 += 16) {
      uint32_t r[16];
      if (nkb > 0) tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r);
      else {
#pragma unroll
        for (int x = 0; x < 16; ++x) r[x] = 0;
      }
#pragma unroll
      for (int x = 0; x < 4; ++x)
        reinterpret_cast<float4*>(P + c0)[x] = make_float4(__uint_as_float(r[4 * x]), __uint_as_float(r[4 * x + 1]),
                                                           __uint_as_float(r[4 * x + 2]), __uint_as_float(r[4 * x + 3]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// partial [ctas][128 lanes][WL_COLS] -> dW3[oc][c][ky][kx] (torch layout) and db3[oc]; fixed summation order.
// columns 0..191: D0 (col = kx*64 + c): lanes 0-63 = tap ky 1, lanes 64-127 = tap ky 0; 192..383: D1: lanes 0-63 = ky 2;
// column 384: bias (lanes 0-63); lane % 64 = oc.
__global__ void conv_wgrad_lin_reduce3_kernel(int ctas, const float* __restrict__ partial, float beta,
                                              float* __restrict__ dW, float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;       // (lane, column), column fastest: coalesced partial reads
  const int total = 128 * WL_COLS;
  if (i >= total) return;
  const int col = i % WL_COLS, ln = i / WL_COLS, oc = ln & 63;
  int idx = -1;
  float* dst = dW;
  if (col < 384) {
    const int d = col >= 192, cc = col - 192 * d, kx = cc >> 6, c = cc & 63;
    const int ky = d ? (ln < 64 ? 2 : -1) : (ln < 64 ? 1 : 0);
    if (ky >= 0) idx = ((oc * 64 + c) * 3 + ky) * 3 + kx;
  } else if (col == 384 && ln < 64 && db) {
    idx = oc; dst = db;
  }
  if (idx < 0) return;
  float s = 0.f;
  for (int z = 0; z < ctas; ++z) s += partial[(long long)z * total + i];
  dst[idx] = beta != 0.f ? fmaf(beta, dst[idx], s) : s;
}

// conv3: y2b (N, H2, W2, 64) bf16, dy3p (N, H2, W2, 64) bf16 = the gradient w.r.t. conv3's pre-activation stored at y2's
// pitch, zero outside the (H2-2) x (W2-2) valid outputs.  Returns 1 when the shape is outside the kernel's range.
// ---- conv1 (on the space-to-depth image: 2 x 2 taps, 32 output channels).  The gradient rows are 64 bytes wide, so dY
// is the N operand in the 64-byte swizzle (N-atom = 32 channels) and the source the M operand:
//   A = source rows, M = 128 = the taps dx = 0, 1 (M-atom stride = 1 pixel row);
//   B = dY rows,     N = 64 = two kernel rows: N-atom 0 = dY[p], N-atom 1 = dY[p + W] (stride = W pixel rows of 64 B).
// With A shifted by W, ONE MMA per 16 pixel rows covers all four taps: columns 0-31 = taps dy = 1, columns 32-63 = dy = 0.
constexpr int WL1_COLS = 64 + 32;         // accumulator columns: D | bias

__global__ void __launch_bounds__(WL_THREADS, 1)
conv_wgrad_lin1_kernel(const __grid_constant__ WgradLinGeom g, const __grid_constant__ CUtensorMap tmS,
                       const __grid_constant__ CUtensorMap tmD) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t src_bytes = (uint32_t)g.src_rows * 128, dy_bytes = (uint32_t)g.dy_rows * 64;   // multiples of 1024
  const uint32_t stage_bytes = src_bytes + dy_bytes;
  const uint32_t base = smem_u32(smem);
  const int NST = g.stages;
  const uint32_t ones_tile = base + NST * stage_bytes;             // 2 M-atoms x 16 K rows x 128 B of bf16 1.0
  uint64_t* bars = (uint64_t*)(smem + NST * stage_bytes + 4096);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * WL_MAX_STAGES + 1);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + WL_MAX_STAGES + s); };
  const uint32_t done_bar = smem_u32(bars + 2 * WL_MAX_STAGES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb_begin = blockIdx.x * g.kb_per_cta;
  const int kb_end = min(g.nkb, kb_begin + g.kb_per_cta);
  const int nkb = max(0, kb_end - kb_begin);

  for (int i = threadIdx.x; i < 4096 / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem + NST * stage_bytes)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
  if (threadIdx.x == 0) {
    for (int s = 0; s < NST; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(done_bar, 1);
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  cv_fence_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % NST;
        mbar_wait(empty_bar(s), ((i / NST) & 1) ^ 1);
        const uint32_t st = base + s * stage_bytes;
        const int row0 = (kb_begin + i) * WL_KB;
        mbar_expect_tx(full_bar(s), src_bytes + dy_bytes);
        tma_load_2d(st, &tmS, 0, row0, full_bar(s));
        tma_load_2d(st + src_bytes, &tmD, 0, row0 - g.W, full_bar(s));
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && nkb > 0) {
      constexpr uint32_t idesc = idesc_bf16(128, 64, true, true), idesc_b = idesc_bf16(128, 32, true, true);
      const uint64_t ones_desc = smem_desc(ones_tile, 2048, 1024);
      const uint64_t a0 = smem_desc(base, 128, 1024);                                  // M-atom stride: one pixel row
      const uint64_t b0 = smem_desc(base + src_bytes, (uint32_t)g.W * 64, 512, UMMA_SW64);   // N-atom stride: one image row
      for (int i = 0; i < nkb; ++i) {
        const int s = i % NST;
        mbar_wait(full_bar(s), (i / NST) & 1);
        tc_fence_after();
        const uint64_t so = (uint64_t)((s * stage_bytes) >> 4);
#pragma unroll
        for (int k = 0; k < WL_KB / 16; ++k) {      // 16 pixel rows per UMMA K step: 2048 B of the source, 1024 B of dY
          const uint32_t acc = (i > 0 || k > 0) ? 1u : 0u;
          const uint64_t ad = a0 + so + (uint64_t)(k * 128), bd = b0 + so + (uint64_t)(k * 64);
          tc_mma_bf16(tmem_base, ad, bd, idesc, acc);
          tc_mma_bf16(tmem_base + 64, ones_desc, bd, idesc_b, acc);
        }
        tc_commit(empty_bar(s));
      }
      tc_commit(done_bar);
    }
  } else {
    const int q = warp & 3;
    if (nkb > 0) { mbar_wait(done_bar, 0); tc_fence_after(); }
    float* P = g.partial + ((long long)blockIdx.x * 128 + (q * 32 + lane)) * WL1_COLS;
#pragma unroll 1
    for (int c0 = 0; c0 < WL1_COLS; c0 += 16) {
      uint32_t r[16];
      if (nkb > 0) tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r);
      else {
#pragma unroll
        for (int x = 0; x < 16; ++x) r[x] = 0;
      }
#pragma unroll
      for (int x = 0; x < 4; ++x)
        reinterpret_cast<float4*>(P + c0)[x] = make_float4(__uint_as_float(r[4 * x]), __uint_as_float(r[4 * x + 1]),
                                                           __uint_as_float(r[4 * x + 2]), __uint_as_float(r[4 * x + 3]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

// partial [ctas][128 lanes = (dx, q)][WL1_COLS] -> dW1[oc][c][ky][kx] and db1[oc].  columns 0-31: tap dy = 1, 32-63: dy = 0
// (oc = col % 32); columns 64-95: bias (any lane; lane 0 is used).  q = (py*4 + px)*3 + c < 48, ky = 4 dy + py, kx = 4 dx + px.
__global__ void conv_wgrad_lin_reduce1_kernel(int ctas, const float* __restrict__ partial, float beta,
                                              float* __restrict__ dW, float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int total = 128 * WL1_COLS;
  if (i >= total) return;
  const int col = i % WL1_COLS, ln = i / WL1_COLS;
  int idx = -1;
  float* dst = dW;
  if (col < 64) {
    const int oc = col & 31, dy = col < 32 ? 1 : 0, dx = ln >> 6, q = ln & 63;
    if (q < 48) {
      const int c = q % 3, pp = q / 3, py = pp >> 2, px = pp & 3;
      idx = ((oc * 3 + c) * 8 + (4 * dy + py)) * 8 + (4 * dx + px);
    }
  } else if (ln == 0 && db) {
    idx = col - 64; dst = db;
  }
  if (idx < 0) return;
  float s = 0.f;
  for (int z = 0; z < ctas; ++z) s += partial[(long long)z * total + i];
  dst[idx] = beta != 0.f ? fmaf(beta, dst[idx], s) : s;
}

bool conv_lin_conv1_wgrad_ok(int Wp) {
  return tmap_encoder_available() && ((WL_KB + Wp + 15) & ~15) <= 256;
}

// conv1: xs (N, Hp, Wp, 64) bf16 space-to-depth image, dy1p (N, Hp, Wp, 32) bf16 = the gradient w.r.t. conv1's
// pre-activation at the image's pitch, zero in the last row / column of every frame.  1: shape outside the kernel's range.
int conv_lin_conv1_wgrad(const void* dy1p, const void* xs, int N, int Hp, int Wp, float beta, float* dW, float* db,
                         float* ws, size_t ws_bytes, cudaStream_t st) {
  if (N == 0) return 0;
  if (!tmap_encoder_available()) return 1;
  WgradLinGeom g = {};
  g.W = Wp;
  g.src_rows = (WL_KB + 1 + 7) & ~7;               // window rows 0 .. 127 + 1 (tap dx = 1)
  g.dy_rows = (WL_KB + Wp + 15) & ~15;             // rows 0 .. 127 + Wp (N-atom 1); x 64 B must be a multiple of 1024
  if (g.dy_rows > 256) return 1;
  const long long rows = (long long)N * Hp * Wp;
  g.nkb = (int)((rows + Wp + WL_KB - 1) / WL_KB);
  int ctas = persistent_ctas();
  if (ctas > g.nkb) ctas = g.nkb;
  const size_t per_cta = (size_t)128 * WL1_COLS * sizeof(float);
  if ((size_t)ctas * per_cta > ws_bytes) ctas = (int)(ws_bytes / per_cta);
  TACORL_REQUIRE(ws && ctas >= 1, "conv_lin_wgrad: workspace too small");
  g.kb_per_cta = (g.nkb + ctas - 1) / ctas;
  ctas = (g.nkb + g.kb_per_cta - 1) / g.kb_per_cta;
  g.partial = ws;
  CUtensorMap ts, td;
  int rc;
  TACORL_REQUIRE((((uintptr_t)xs | (uintptr_t)dy1p) & 15) == 0, "conv_lin_wgrad: tensors must be 16-byte aligned");
  const cuuint64_t s_dims[2] = {64, (cuuint64_t)rows}, s_strides[1] = {128};
  const cuuint64_t d_dims[2] = {32, (cuuint64_t)rows}, d_strides[1] = {64};
  const cuuint32_t s_box[2] = {64, (cuuint32_t)g.src_rows}, d_box[2] = {32, (cuuint32_t)g.dy_rows};
  if ((rc = encode_tmap_bf16(&ts, "conv_lin_wgrad(source)", 2, xs, s_dims, s_strides, s_box))) return rc;
  if ((rc = encode_tmap_bf16(&td, "conv_lin_wgrad(gradient)", 2, dy1p, d_dims, d_strides, d_box, CU_TENSOR_MAP_SWIZZLE_64B)))
    return rc;
  const size_t stage = (size_t)g.src_rows * 128 + (size_t)g.dy_rows * 64;
  const size_t fixed = 4096 + (2 * WL_MAX_STAGES + 1) * 8 + 16 + 1024;
  g.stages = (int)std::min<size_t>(WL_MAX_STAGES, (227 * 1024 - fixed) / stage);
  if (g.stages < 2) return 1;
  const size_t smem = fixed + g.stages * stage;
  static size_t configured = 0;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(conv_wgrad_lin1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  conv_wgrad_lin1_kernel<<<ctas, WL_THREADS, smem, st>>>(g, ts, td);
  TACORL_LAUNCH_CHECK();
  conv_wgrad_lin_reduce1_kernel<<<cdiv(128 * WL1_COLS, 256), 256, 0, st>>>(ctas, ws, beta, dW, db);
  TACORL_LAUNCH_CHECK();
  return 0;
}

bool conv_lin_conv3_wgrad_ok(int W2) {
  return tmap_encoder_available() && ((WL_KB + W2 + 2 + 7) & ~7) <= 256;
}

int conv_lin_conv3_wgrad(const void* dy3p, const void* y2b, int N, int H2, int W2, float beta, float* dW, float* db,
                         float* ws, size_t ws_bytes, cudaStream_t st) {
  if (N == 0) return 0;
  if (!tmap_encoder_available()) return 1;
  WgradLinGeom g = {};
  g.W = W2;
  g.src_rows = (WL_KB + W2 + 2 + 7) & ~7;          // window rows 0 .. 127 + W2 + 2 (D1, kx = 2)
  g.dy_rows = (WL_KB + W2 + 7) & ~7;               // rows 0 .. 127 + W2 (M-atom 1)
  if (g.src_rows > 256 || g.dy_rows > 256) return 1;
  const long long rows = (long long)N * H2 * W2;
  g.nkb = (int)((rows + W2 + WL_KB - 1) / WL_KB);
  int ctas = persistent_ctas();
  if (ctas > g.nkb) ctas = g.nkb;
  const size_t per_cta = (size_t)128 * WL_COLS * sizeof(float);
  if ((size_t)ctas * per_cta > ws_bytes) ctas = (int)(ws_bytes / per_cta);
  TACORL_REQUIRE(ws && ctas >= 1, "conv_lin_wgrad: workspace too small");
  g.kb_per_cta = (g.nkb + ctas - 1) / ctas;
  ctas = (g.nkb + g.kb_per_cta - 1) / g.kb_per_cta;
  g.partial = ws;
  CUtensorMap ts, td;
  int rc;
  TACORL_REQUIRE((((uintptr_t)y2b | (uintptr_t)dy3p) & 15) == 0, "conv_lin_wgrad: tensors must be 16-byte aligned");
  const cuuint64_t dims[2] = {64, (cuuint64_t)rows}, strides[1] = {128};
  const cuuint32_t s_box[2] = {64, (cuuint32_t)g.src_rows}, d_box[2] = {64, (cuuint32_t)g.dy_rows};
  if ((rc = encode_tmap_bf16(&ts, "conv_lin_wgrad(source)", 2, y2b, dims, strides, s_box))) return rc;
  if ((rc = encode_tmap_bf16(&td, "conv_lin_wgrad(gradient)", 2, dy3p, dims, strides, d_box))) return rc;
  const size_t stage = (size_t)(g.src_rows + g.dy_rows) * 128;
  const size_t fixed = 2048 + (2 * WL_MAX_STAGES + 1) * 8 + 16 + 1024;
  g.stages = (int)std::min<size_t>(WL_MAX_STAGES, (227 * 1024 - fixed) / stage);
  if (g.stages < 2) return 1;
  const size_t smem = fixed + g.stages * stage;
  static size_t configured = 0;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(conv_wgrad_lin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  conv_wgrad_lin_kernel<<<ctas, WL_THREADS, smem, st>>>(g, ts, td);
  TACORL_LAUNCH_CHECK();
  conv_wgrad_lin_reduce3_kernel<<<cdiv(128 * WL_COLS, 256), 256, 0, st>>>(ctas, ws, beta, dW, db);
  TACORL_LAUNCH_CHECK();
  return 0;
}

}  // namespace tacorl

// ==========================================================================================
// Diagnostic entry point (tests/test_gpu_conv_tc.py): runs ONE implicit-GEMM convolution op on fp32 inputs
// (staged to bf16 exactly as the encoder does) so each kernel can be checked tightly against torch's conv in fp64.
namespace tacorl {
__global__ void cv_bf16_to_f32_kernel(long long n, const __nv_bfloat16* __restrict__ a, float* __restrict__ o) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    o[i] = __bfloat162float(a[i]);
}
static int cv_to_f32(long long n, const void* a, float* o, cudaStream_t st) {
  cv_bf16_to_f32_kernel<<<(int)min((long long)1184, (n + 255) / 256), 256, 0, st>>>(n, (const __nv_bfloat16*)a, o);
  TACORL_LAUNCH_CHECK();
  return 0;
}
}  // namespace tacorl

extern "C" int tacorl_conv_tc_debug(int op, const float* in0, const float* in1, const float* Wt, const float* bias, int N,
                                    int H, int W, float* out, void* ws, size_t ws_bytes, void* stream) {
  using namespace tacorl;
  cudaStream_t st = (cudaStream_t)stream;
  const int H1 = (H - 8) / 4 + 1, W1 = (W - 8) / 4 + 1, H2 = (H1 - 4) / 2 + 1, W2 = (W1 - 4) / 2 + 1, H3 = H2 - 2, W3 = W2 - 2;
  const long long P1 = (long long)H1 * W1, P2 = (long long)H2 * W2, P3 = (long long)H3 * W3;
  Arena ar(ws, ws_bytes);
  __nv_bfloat16* wp = ar.take<__nv_bfloat16>(16 * 64 * 64);
  __nv_bfloat16* a0 = ar.take<__nv_bfloat16>((size_t)N * (H1 + 1) * (W1 + 1) * 64 + (size_t)N * P1 * 64);
  __nv_bfloat16* a1 = ar.take<__nv_bfloat16>((size_t)N * (H1 + 1) * (W1 + 1) * 64 + (size_t)N * P1 * 64);
  __nv_bfloat16* ob = ar.take<__nv_bfloat16>((size_t)N * P1 * 64);
  float* wsf = ar.take<float>((32 << 20) / 4);
  TACORL_REQUIRE(wp && a0 && a1 && ob && wsf, "conv_tc_debug: workspace too small");
  int rc;
  switch (op) {
    case 1:
      if ((rc = conv_tc_pack(2, Wt, wp, st))) return rc;
      if ((rc = conv_tc_s2d(in0, N, H, W, H1 + 1, W1 + 1, a0, st))) return rc;
      if ((rc = conv_tc_conv1_fwd(a0, N, H1, W1, wp, bias, ob, st))) return rc;
      return cv_to_f32(N * P1 * 32, ob, out, st);
    case 2:
      if ((rc = conv_tc_pack(1, Wt, wp, st))) return rc;
      if ((rc = cast_bf16_2d(in0, 32, N * P1, 32, a0, 32, st))) return rc;
      if ((rc = conv_tc_conv2_fwd(a0, N, H1, W1, H2, W2, wp, bias, ob, st))) return rc;
      return cv_to_f32(N * P2 * 64, ob, out, st);
    case 3:
      if ((rc = conv_tc_pack(0, Wt, wp, st))) return rc;
      if ((rc = cast_bf16_2d(in0, 64, N * P2, 64, a0, 64, st))) return rc;
      return conv_tc_conv3_fwd(a0, N, H2, W2, H3, W3, wp, bias, out, st);
    case 4:
      if ((rc = conv_tc_pack(3, Wt, wp, st))) return rc;
      if ((rc = cast_bf16_2d(in0, 64, N * P3, 64, a0, 64, st))) return rc;
      if ((rc = cast_bf16_2d(in1, 64, N * P2, 64, a1, 64, st))) return rc;
      if ((rc = conv_tc_conv3_dgrad(a0, N, H2, W2, H3, W3, wp, a1, ob, st))) return rc;
      return cv_to_f32(N * P2 * 64, ob, out, st);
    case 5:
      if ((rc = conv_tc_pack(4, Wt, wp, st))) return rc;
      if ((rc = cast_bf16_2d(in0, 64, N * P2, 64, a0, 64, st))) return rc;
      if ((rc = cast_bf16_2d(in1, 32, N * P1, 32, a1, 32, st))) return rc;
      if ((rc = conv_tc_conv2_dgrad(a0, N, H1, W1, H2, W2, wp, a1, ob, st))) return rc;
      return cv_to_f32(N * P1 * 32, ob, out, st);
    case 6:
      if ((rc = cast_bf16_2d(in0, 64, N * P3, 64, a0, 64, st))) return rc;
      if ((rc = cast_bf16_2d(in1, 64, N * P2, 64, a1, 64, st))) return rc;
      return conv_tc_wgrad(3, a0, a1, N, H2, W2, H3, W3, 0.f, out, out + 64 * 64 * 9, wsf, 32 << 20, st);
    case 7:
      if ((rc = cast_bf16_2d(in0, 64, N * P2, 64, a0, 64, st))) return rc;
      if ((rc = cast_bf16_2d(in1, 32, N * P1, 32, a1, 32, st))) return rc;
      return conv_tc_wgrad(2, a0, a1, N, H1, W1, H2, W2, 0.f, out, out + 64 * 32 * 16, wsf, 32 << 20, st);
    case 8:
      if ((rc = cast_bf16_2d(in0, 32, N * P1, 32, a0, 32, st))) return rc;
      if ((rc = conv_tc_s2d(in1, N, H, W, H1 + 1, W1 + 1, a1, st))) return rc;
      return conv_tc_wgrad(1, a0, a1, N, H1 + 1, W1 + 1, H1, W1, 0.f, out, out + 32 * 3 * 64, wsf, 32 << 20, st);
    case 11:     // conv1 forward, linear-shift kernel
      if ((rc = conv_tc_pack(2, Wt, wp, st))) return rc;
      if ((rc = conv_tc_s2d(in0, N, H, W, H1 + 1, W1 + 1, a0, st))) return rc;
      if ((rc = conv_lin_conv1_fwd(a0, N, H1, W1, wp, bias, ob, st))) return rc;
      return cv_to_f32(N * P1 * 32, ob, out, st);
    case 15:     // conv2 data gradient, four parity classes fused into one kernel
      if ((rc = conv_tc_pack(5, Wt, wp, st))) return rc;
      if ((rc = cast_bf16_2d(in0, 64, N * P2, 64, a0, 64, st))) return rc;
      if ((rc = cast_bf16_2d(in1, 32, N * P1, 32, a1, 32, st))) return rc;
      if ((rc = conv_dgrad2_fused(a0, N, H1, W1, H2, W2, wp, a1, ob, 0, st))) return rc;
      return cv_to_f32(N * P1 * 32, ob, out, st);
    case 16: {   // conv3 weight gradient, linear-shift kernel: in0 = dy3 at y2's pitch (N, H2, W2, 64), zero margins
      if ((rc = cast_bf16_2d(in0, 64, N * P2, 64, a0, 64, st))) return rc;
      if ((rc = cast_bf16_2d(in1, 64, N * P2, 64, a1, 64, st))) return rc;
      rc = conv_lin_conv3_wgrad(a0, a1, N, H2, W2, 0.f, out, out + 64 * 64 * 9, wsf, 32 << 20, st);
      if (rc == 1) set_last_error("conv_tc_debug: linear-shift weight gradient does not cover this shape");
      return rc;
    }
    case 18: {   // conv1 weight gradient, linear-shift kernel: in0 = dy1 at the s2d image's pitch (N, H1+1, W1+1, 32)
      if ((rc = cast_bf16_2d(in0, 32, (long long)N * (H1 + 1) * (W1 + 1), 32, a0, 32, st))) return rc;
      if ((rc = conv_tc_s2d(in1, N, H, W, H1 + 1, W1 + 1, a1, st))) return rc;
      rc = conv_lin_conv1_wgrad(a0, a1, N, H1 + 1, W1 + 1, 0.f, out, out + 32 * 3 * 64, wsf, 32 << 20, st);
      if (rc == 1) set_last_error("conv_tc_debug: linear-shift weight gradient does not cover this shape");
      return rc;
    }
    case 13:     // conv3 forward, linear-shift kernel
      if ((rc = conv_tc_pack(0, Wt, wp, st))) return rc;
      if ((rc = cast_bf16_2d(in0, 64, N * P2, 64, a0, 64, st))) return rc;
      return conv_lin_conv3_fwd(a0, N, H2, W2, H3, W3, wp, bias, out, st);
    default:
      set_last_error("conv_tc_debug: unknown op %d", op);
      return -1;
  }
}
