// bf16 tensor-core GEMM for sm_100a: TMA (cp.async.bulk.tensor) -> 128B-swizzled shared memory ->
// tcgen05.mma (single-thread issue, cta_group::1, UMMA 128 x BN x 16) with the fp32 accumulator in TMEM ->
// tcgen05.ld epilogue (alpha/beta/bias/activation, fp32 and/or bf16 stores, or split-K partials).
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM lane quarter = warp_idx % 4).  A kStages-deep mbarrier ring connects
// producer and issuer; tcgen05.commit releases ring slots and finally signals the epilogue.
//
// Operand layouts: each operand is either K-major ([rows][K], K contiguous; one 64-wide K slab per
// stage, canonical SW128 K-major atoms, SBO = 1024 B) or MN-major ([K][rows], rows contiguous; 64x64
// boxes, canonical SW128 MN-major atoms, SBO = 1024 B between 8-row K groups, LBO = 8192 B between
// 64-wide MN groups).  MN-major lets dX = dZ.W and dW = dZ^T.X run on the tensors as stored.
#include "common.cuh"
#include "internal.h"
#include <cuda.h>
#include <cuda_bf16.h>
#include <algorithm>

namespace tacorl {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;          // bf16 elements = 128 bytes = one swizzle row
constexpr int TC_UMMA_K = 16;
constexpr int TC_THREADS = 192;

// ------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tc_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// SM100 shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout SWIZZLE_128B=2 [61,64).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

struct TcEpilogue {
  float alpha, beta;
  float* C; long long ldc;              // fp32 output (may be null if only bf16 output is wanted)
  __nv_bfloat16* Cb; long long ldcb;    // optional bf16 copy of the (post-activation) output
  const float* bias;                    // per column
  int act;
  float* Cpre; long long ldpre;
  float* partial;                       // split-K: raw accumulators [z][M][N]
  const float* gate; long long ldgate;  // optional ReLU gate: output forced to 0 where gate[row][col] <= 0
};

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// Epilogue math for one 16-column chunk of one output row, with 16-byte vector accesses when the row is
// aligned and the chunk is fully inside the matrix (scalar guarded accesses otherwise).
__device__ __forceinline__ void tc_epilogue_chunk(const TcEpilogue& ep, const uint32_t (&r)[16], int row, int col0,
                                                  int N, int zslice, int M) {
  const bool full = col0 + 16 <= N;
  if (ep.partial) {
    float* P = ep.partial + ((long long)zslice * M + row) * N + col0;
    if (full && (N & 3) == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        reinterpret_cast<float4*>(P)[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                      __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (col0 + j < N) P[j] = __uint_as_float(r[j]);
    }
    return;
  }
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = ep.alpha * __uint_as_float(r[j]);
  float* Crow = ep.C ? ep.C + (long long)row * ep.ldc + col0 : nullptr;
  const bool vecC = full && Crow && ((ep.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(ep.C) & 15) == 0);
  if (ep.beta != 0.f && Crow) {
    if (vecC) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 c = reinterpret_cast<const float4*>(Crow)[j];
        v[4 * j] = fmaf(ep.beta, c.x, v[4 * j]); v[4 * j + 1] = fmaf(ep.beta, c.y, v[4 * j + 1]);
        v[4 * j + 2] = fmaf(ep.beta, c.z, v[4 * j + 2]); v[4 * j + 3] = fmaf(ep.beta, c.w, v[4 * j + 3]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (col0 + j < N) v[j] = fmaf(ep.beta, Crow[j], v[j]);
    }
  }
  if (ep.bias) {
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N) v[j] += __ldg(ep.bias + col0 + j);
  }
  if (ep.Cpre) {
    float* Prow = ep.Cpre + (long long)row * ep.ldpre + col0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N) Prow[j] = v[j];
  }
  if (ep.act == ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
  } else if (ep.act == ACT_SILU) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = v[j] / (1.f + __expf(-v[j]));
  }
  if (ep.gate) {
    const float* Grow = ep.gate + (long long)row * ep.ldgate + col0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (col0 + j < N && Grow[j] <= 0.f) v[j] = 0.f;
  }
  if (Crow) {
    if (vecC) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        reinterpret_cast<float4*>(Crow)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (col0 + j < N) Crow[j] = v[j];
    }
  }
  if (ep.Cb) {
    __nv_bfloat16* Brow = ep.Cb + (long long)row * ep.ldcb + col0;
    if (full && ((ep.ldcb & 7) == 0) && ((reinterpret_cast<uintptr_t>(ep.Cb) & 15) == 0)) {
      uint32_t pk[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        pk[j] = *reinterpret_cast<uint32_t*>(&t);
      }
      reinterpret_cast<uint4*>(Brow)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      reinterpret_cast<uint4*>(Brow)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (col0 + j < N) Brow[j] = __float2bfloat16(v[j]);
    }
  }
}

// Persistent over output tiles: CTA b processes tiles b, b + gridDim.x, ...; two TMEM accumulator stages let the
// epilogue of tile i overlap the MMAs of tile i+1; the smem ring runs continuously across tiles.
template <int BN, bool A_MN, bool B_MN, int kStages>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, TcEpilogue ep,
               int M, int N, int K, int kblocks_per_split) {
  constexpr uint32_t A_BYTES = TC_BM * TC_BK * 2;     // 16 KB
  constexpr uint32_t B_BYTES = BN * TC_BK * 2;
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t ACC_COLS = BN < 32 ? 32 : BN;
  constexpr uint32_t TMEM_COLS = 2 * ACC_COLS;        // power of two >= 64
  static_assert(!B_MN || BN % 64 == 0, "MN-major B needs 64-wide boxes");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment is required by the 128B swizzle atoms
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + kStages * STAGE_BYTES);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_kb = (K + TC_BK - 1) / TC_BK;
  const int kb_begin = blockIdx.z * kblocks_per_split;
  const int kb_end = min(total_kb, kb_begin + kblocks_per_split);
  const int nkb = kb_end - kb_begin;
  const int tiles_n = (N + BN - 1) / BN;
  const int num_tiles = ((M + TC_BM - 1) / TC_BM) * tiles_n;

  const uint32_t smem_base = smem_u32(smem);
  auto full_bar = [&](int s) { return smem_u32(bars + s); };
  auto empty_bar = [&](int s) { return smem_u32(bars + kStages + s); };
  auto tfull_bar = [&](int a) { return smem_u32(bars + 2 * kStages + a); };
  auto tempty_bar = [&](int a) { return smem_u32(bars + 2 * kStages + 2 + a); };

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0 && nkb > 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * TC_BM, n0 = (tile % tiles_n) * BN;
        for (int i = 0; i < nkb; ++i, ++it) {
          const int s = it % kStages;
          const uint32_t ph = (it / kStages) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_expect_tx(full_bar(s), STAGE_BYTES);
          const int k0 = (kb_begin + i) * TC_BK;
          const uint32_t a_dst = smem_base + s * STAGE_BYTES, b_dst = a_dst + A_BYTES;
          if (!A_MN) {
            tma_load_2d(a_dst, &tmA, k0, m0, full_bar(s));
          } else {
            tma_load_2d(a_dst, &tmA, m0, k0, full_bar(s));
            tma_load_2d(a_dst + 8192, &tmA, m0 + 64, k0, full_bar(s));
          }
          if (!B_MN) {
            tma_load_2d(b_dst, &tmB, k0, n0, full_bar(s));
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j) tma_load_2d(b_dst + j * 8192, &tmB, n0 + j * 64, k0, full_bar(s));
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && nkb > 0) {
      // instruction descriptor: D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1, a_major bit15, b_major bit16,
      // N>>3 at [17,23), M>>4 at [24,29)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      uint32_t it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++lt) {
        const uint32_t acc = lt & 1;
        mbar_wait(tempty_bar(acc), ((lt >> 1) & 1) ^ 1);     // epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * ACC_COLS;
        for (int i = 0; i < nkb; ++i, ++it) {
          const int s = it % kStages;
          const uint32_t ph = (it / kStages) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t a_src = smem_base + s * STAGE_BYTES, b_src = a_src + A_BYTES;
#pragma unroll
          for (int k = 0; k < TC_BK / TC_UMMA_K; ++k) {
            // K-major: advance 16 elements (32 B) inside the 128 B swizzle row; MN-major: 16 K-rows of 128 B
            const uint64_t ad = A_MN ? make_smem_desc(a_src + k * 2048, 8192, 1024) : make_smem_desc(a_src + k * 32, 16, 1024);
            const uint64_t bd = B_MN ? make_smem_desc(b_src + k * 2048, 8192, 1024) : make_smem_desc(b_src + k * 32, 16, 1024);
            tc_mma_bf16(tmem_d, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
          }
          tc_commit(empty_bar(s));          // slot reusable once these MMAs have read it
        }
        tc_commit(tfull_bar(acc));          // accumulator complete
      }
    }
  } else {
    // ---- epilogue: TMEM lane quarter q holds rows m0 + 32q .. +31
    const int q = warp & 3;
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++lt) {
      const int m0 = (tile / tiles_n) * TC_BM, n0 = (tile % tiles_n) * BN;
      const int row = m0 + q * 32 + lane;
      const uint32_t acc = lt & 1;
      if (nkb > 0) {
        mbar_wait(tfull_bar(acc), (lt >> 1) & 1);
        tc_fence_after();
      }
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t r[16];
        if (nkb > 0) {
          tc_ld16(tmem_base + acc * ACC_COLS + ((uint32_t)(q * 32) << 16) + c0, r);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = 0;
        }
        if (row < M && n0 + c0 < N) tc_epilogue_chunk(ep, r, row, n0 + c0, N, blockIdx.z, M);
      }
      if (nkb > 0) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));     // this warp's TMEM reads of the stage are complete
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}


// ------------------------------------------------------------------------------------------ skinny cluster split-K
// Recurrent steps (h_t = act(C + h_{t-1} W^T), batch <= 128 rows, 2048 x 2048 weights) are latency bound: every
// CTA of an ordinary N-tiled GEMM streams the whole K extent of both operands through one SM.  Here a cluster of
// RS_KS CTAs splits K instead: CTA r loads K slab r of the activations (UMMA M = 128 rows, only the batch rows are
// fetched) and of one NT-column weight tile (UMMA N), keeps its partial accumulator in TMEM, spills it to its own
// shared memory, and after one cluster barrier pulls a 1/RS_KS slice of the batch rows from all peers through
// distributed shared memory (16-byte ld.shared::cluster; measured faster than pushing with st.shared::cluster),
// sums them in a fixed order and applies the fused epilogue.  No partial sums travel through L2 and there is no
// second kernel.  At most 15 clusters of 8 CTAs are co-resident on a B200 (148 SMs in GPCs of 16-20), so N is cut
// into <= 15 tiles of NT = 16*ceil(N/240) columns: one wave, 120 SMs busy.
constexpr int RS_KS = 8;
constexpr int RS_MAX_TILES = 15;
constexpr int RS_EPI = 512;          // 16 epilogue warps: enough loads in flight to hide the DSMEM / global latency
constexpr int RS_THREADS = RS_EPI + 32;   // + warp 16: barrier setup, TMEM allocation, TMA and MMA issue
constexpr int RS_MAXE = 2;           // float4 elements per thread in the reduction: 16 rows x 256 columns / 4 / 512 threads
#ifdef TACORL_STEP_PROFILE
__device__ unsigned long long g_step_prof[16];
__device__ unsigned long long g_cta_prof[2][256][2];     // [previous / last launch][cta][start, end]
#define RS_CTA_STAMP(which)                                                              \
  if (tid == 0) {                                                                        \
    const int c_ = blockIdx.y * gridDim.x + blockIdx.x;                                  \
    unsigned long long t_;                                                               \
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                             \
    if (which == 0) { g_cta_prof[0][c_][0] = g_cta_prof[1][c_][0]; g_cta_prof[0][c_][1] = g_cta_prof[1][c_][1]; } \
    g_cta_prof[1][c_][which] = t_;                                                       \
  }
#define RS_STAMP(i)                                                                      \
  if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0) {                                  \
    unsigned long long t_;                                                               \
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                             \
    g_step_prof[i] = t_;                                                                 \
  }                                                                                      \
  __syncwarp();
#define RS_STAMP_T(i)                                                                    \
  if (blockIdx.x == 0 && blockIdx.y == 0) {                                              \
    unsigned long long t_;                                                               \
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                             \
    g_step_prof[i] = t_;                                                                 \
  }
#else
#define RS_STAMP(i)
#define RS_STAMP_T(i)
#define RS_CTA_STAMP(which)
#endif

__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float4 ld_dsmem_v4(uint32_t local_addr, uint32_t cta) {
  uint32_t remote;
  float4 v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(cta));
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(remote)
               : "memory");
  return v;
}

// grid (RS_KS, tiles): blockIdx.x = K slab = cluster rank, blockIdx.y = N tile.  A: [M][K] bf16, W: [N][K] bf16.
__global__ void __cluster_dims__(RS_KS, 1, 1) __launch_bounds__(RS_THREADS, 1)
skinny_cluster_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                      const TcEpilogue ep, int M, int Mpad, int N, int NT, int kb_per_cta) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t A_TILE = 128 * 128, W_BYTES = (uint32_t)NT * 128, STAGE = A_TILE + ((W_BYTES + 1023) & ~1023u);
  const int SP = NT + 4;                                                       // padded row pitch of S (floats)
  const int per = Mpad / RS_KS;                                                // batch rows finished by each CTA
  const size_t stage_total = (size_t)kb_per_cta * STAGE, s_bytes = (size_t)Mpad * SP * 4;
  float* S = (float*)smem;                                                     // partial D, aliases the drained stages
  uint64_t* bars = (uint64_t*)(smem + (stage_total > s_bytes ? stage_total : ((s_bytes + 1023) & ~(size_t)1023)));
  uint32_t* tmem_slot = (uint32_t*)(bars + 9);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = blockIdx.x;                                            // == %cluster_ctarank (grid.x == RS_KS)
  const int n0 = blockIdx.y * NT;
  const uint32_t tmem_cols = NT <= 32 ? 32 : (NT <= 64 ? 64 : (NT <= 128 ? 128 : 256));
  const uint32_t done_bar = smem_u32(bars + 8);
  RS_CTA_STAMP(0)
  RS_STAMP(0)

  if (tid == RS_EPI) {
    for (int s = 0; s < kb_per_cta; ++s) mbar_init(smem_u32(bars + s), 1);
    mbar_init(done_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == RS_EPI / 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  RS_STAMP(1)

  if (tid == RS_EPI) {
    const int k_begin = (int)rank * kb_per_cta * TC_BK;
    for (int s = 0; s < kb_per_cta; ++s) {                                     // the whole slab is in flight at once
      const uint32_t bar = smem_u32(bars + s), dst = smem_u32(smem + (size_t)s * STAGE);
      mbar_expect_tx(bar, (uint32_t)Mpad * 128 + W_BYTES);
      tma_load_2d(dst, &tmA, k_begin + s * TC_BK, 0, bar);                     // Mpad batch rows (rows >= M zero-filled)
      tma_load_2d(dst + A_TILE, &tmW, k_begin + s * TC_BK, n0, bar);           // NT weight rows (rows >= N zero-filled)
    }
    // UMMA rows Mpad..127 read stale shared memory: those accumulator lanes are never drained
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    RS_STAMP_T(2)
    for (int s = 0; s < kb_per_cta; ++s) {
      mbar_wait(smem_u32(bars + s), 0);
      tc_fence_after();
      if (s == 0) { RS_STAMP_T(3) }
      const uint32_t a_src = smem_u32(smem + (size_t)s * STAGE), w_src = a_src + A_TILE;
#pragma unroll
      for (int k = 0; k < TC_BK / TC_UMMA_K; ++k)
        tc_mma_bf16(tmem_base, make_smem_desc(a_src + k * 32, 16, 1024), make_smem_desc(w_src + k * 32, 16, 1024), idesc,
                    (s > 0 || k > 0) ? 1u : 0u);
    }
    tc_commit(done_bar);
    RS_STAMP_T(4)
  }
  // This CTA finishes batch rows [rank*per, (rank+1)*per) of the tile in groups of 4 columns: element e = (row, group)
  // = (e / NT4, e % NT4); epilogue thread t takes e = t, t + 512.  Fetch the epilogue operands (old C, gate, bias)
  // now: they do not depend on the accumulators.
  const int NT4 = NT >> 2, elems = per * NT4;
  float4 cold[RS_MAXE], gt[RS_MAXE], bs[RS_MAXE];
  if (tid < RS_EPI) {
    // branch-free addressing (masked elements read element 0) so the loads of one operand issue back to back
    long long offc[RS_MAXE], offg[RS_MAXE];
    int colc[RS_MAXE];
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) {
      const int e = tid + i * RS_EPI;
      const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
#ifdef RS_EXP_NOPREFETCH
      const bool ok = false;
#else
      const bool ok = e < elems && b < M && col < N;
#endif
      offc[i] = ok ? (long long)b * ep.ldc + col : 0;
      offg[i] = ok ? (long long)b * ep.ldgate + col : 0;
      colc[i] = ok ? col : 0;
    }
    const bool has_c = ep.beta != 0.f && ep.C != nullptr;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f), one = make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) cold[i] = has_c ? *reinterpret_cast<const float4*>(ep.C + offc[i]) : zero;
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) gt[i] = ep.gate ? *reinterpret_cast<const float4*>(ep.gate + offg[i]) : one;
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) bs[i] = ep.bias ? __ldg(reinterpret_cast<const float4*>(ep.bias + colc[i])) : zero;
  }
#ifdef TACORL_STEP_PROFILE
  RS_STAMP(12)
#endif
  if (tid < RS_EPI) {
    mbar_wait(done_bar, 0);
    tc_fence_after();
  }
  RS_STAMP(5)
  // partial accumulator -> shared memory S[b][n] (row pitch NT + 4 floats: conflict-free float4 stores); warp w drains
  // TMEM lane quarter w % 4 (batch rows), column chunks w / 4, w / 4 + 4, ...
  if (tid < RS_EPI) {
    const int q = warp & 3;
    if (q * 32 < Mpad) {
      float* Srow = S + (q * 32 + lane) * SP;
      for (int c0 = (warp >> 2) * 16; c0 < NT; c0 += 64) {
        uint32_t r[16];
        tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          reinterpret_cast<float4*>(Srow + c0)[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                                __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
      }
    }
  }
  tc_fence_before();
  RS_STAMP(6)
  cluster_sync_all();
  RS_STAMP(7)
  if (tid >= RS_EPI) {                      // issuer warp: TMEM is drained; stay for the closing cluster barrier
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
    return;
  }
  // pull the RS_KS peers' partials of my rows (16-byte DSMEM loads, all in flight before the first use) and sum
  // them in a fixed order
  float4 acc[RS_MAXE];
  {
    float4 part[RS_MAXE][RS_KS];
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) {
      const int e = tid + i * RS_EPI;
      const int bi = e / NT4, n = (e - bi * NT4) * 4;
      const uint32_t addr = smem_u32(S + ((int)rank * per + (e < elems ? bi : 0)) * SP + (e < elems ? n : 0));
#pragma unroll
      for (int q = 0; q < RS_KS; ++q) part[i][q] = ld_dsmem_v4(addr, (q + rank) & (RS_KS - 1));   // staggered: 8 CTAs read 8 different peers
    }
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int q = 0; q < RS_KS; ++q) { v.x += part[i][q].x; v.y += part[i][q].y; v.z += part[i][q].z; v.w += part[i][q].w; }
      acc[i] = v;
    }
  }
  RS_STAMP(8)
  // My reads of the peers' shared memory are done (the register operand makes the arrive wait for the loaded
  // values): arrive now, wait only before exiting.  (A relaxed arrive here faults intermittently for >= 96 rows.)
  {
    float dep = 0.f;
#pragma unroll
    for (int i = 0; i < RS_MAXE; ++i) dep += acc[i].x + acc[i].y + acc[i].z + acc[i].w;
#ifndef RS_EXP_LATEARRIVE
    asm volatile("barrier.cluster.arrive.release.aligned;" ::"f"(dep) : "memory");
#endif
  }
#pragma unroll
  for (int i = 0; i < RS_MAXE; ++i) {
    const int e = tid + i * RS_EPI;
    const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
    if (e >= elems || b >= M || col >= N) continue;
    float v[4] = {acc[i].x, acc[i].y, acc[i].z, acc[i].w};
    const float c4[4] = {cold[i].x, cold[i].y, cold[i].z, cold[i].w};
    const float g4[4] = {gt[i].x, gt[i].y, gt[i].z, gt[i].w};
    const float b4[4] = {bs[i].x, bs[i].y, bs[i].z, bs[i].w};
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = fmaf(ep.beta, c4[j], ep.alpha * v[j]) + b4[j];
    if (ep.Cpre) *reinterpret_cast<float4*>(ep.Cpre + (long long)b * ep.ldpre + col) = make_float4(v[0], v[1], v[2], v[3]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (ep.act == ACT_RELU) v[j] = fmaxf(v[j], 0.f);
      else if (ep.act == ACT_SILU) v[j] = v[j] / (1.f + __expf(-v[j]));
      if (g4[j] <= 0.f) v[j] = 0.f;
    }
    if (ep.C) *reinterpret_cast<float4*>(ep.C + (long long)b * ep.ldc + col) = make_float4(v[0], v[1], v[2], v[3]);
    if (ep.Cb) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
      uint2 pk = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
      *reinterpret_cast<uint2*>(ep.Cb + (long long)b * ep.ldcb + col) = pk;
    }
  }
  RS_STAMP(9)
#ifdef RS_EXP_LATEARRIVE
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
#endif
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");             // peers may still be reading my partials
  RS_STAMP(10)
  RS_STAMP(11)
  RS_CTA_STAMP(1)
}

// ------------------------------------------------------------------------------------------ persistent recurrence
// A whole sequence of dependent recurrent steps  C[tau] = epilogue(C[tau] + A[tau - dtau] . W^T)  in ONE launch of the
// cluster split-K layout above: the CTA's weight slab (NT columns x K/RS_KS, <= 72 KB) is loaded once and stays in
// shared memory, TMEM and the barriers are set up once, and a step only moves the (batch x K/RS_KS) slab of the
// previous hidden state.  Steps are chained by per-tile arrival counters in global memory: the CTAs of N tile j bump
// flags[j] (release, gpu scope) after their rows of step s are stored; a CTA starts step s + 1 once the tiles covering
// ITS K slab have all RS_KS arrivals for step s (acquire) - no grid-wide barrier, no host involvement.
// All clusters must be co-resident (checked on the host with cudaOccupancyMaxActiveClusters); a bounded spin marks
// g_rnn_seq_timeouts instead of hanging if that assumption is ever violated.  Per-step arithmetic (operand tiles, summation
// order, epilogue) is exactly skinny_cluster_kernel's, so both paths produce bit-identical results.
struct SeqArgs {
  int n_steps;                            // steps of this launch: s = 0 .. n_steps-1, output time tau = tau0 + s*dtau
  int tau0, dtau;                         // A operand of step s = bf16 rows of time tau - dtau (3-D tensor map, z = time)
  float beta;
  float* C; long long ldc, c_ts;          // fp32 in (pre-activation / upstream gradient) and out; row pitch, time stride
  const float* gate; long long ldgate, gate_ts;
  __nv_bfloat16* Cb; long long cb_ts;     // dense bf16 copy of the output (row pitch N): the next step's A operand
  int act;
  unsigned* flags;                        // [tiles] arrival counters, zero before the launch
};
__device__ unsigned g_rnn_seq_timeouts = 0;   // flag waits that gave up (never expected; read by tacorl_rnn_seq_timeouts)
// Arrival counters of the persistent recurrence kernels: [lane][tile].  Zero at module load and SELF-CLEANING: the last
// CTA of a launch to finish (nobody polls any more by then) resets them, so no launch needs a memset in front of it
// (8 memset nodes + their launch gaps per training step otherwise).  Persistent launches never overlap (chained).
__device__ unsigned g_rnn_flags[2][32];
__device__ unsigned g_rnn_done = 0;
__device__ __forceinline__ void rnn_launch_epilogue(int tid) {
  if (tid == 0) {
    __threadfence();
    const unsigned total = gridDim.x * gridDim.y * gridDim.z;
    if (atomicAdd(&g_rnn_done, 1u) == total - 1) {
#pragma unroll
      for (int i = 0; i < 64; ++i) (&g_rnn_flags[0][0])[i] = 0;
      __threadfence();
      g_rnn_done = 0;
    }
  }
}
#ifdef TACORL_STEP_PROFILE                    // stage stamps of one CTA at step 8 (scripts/prof/step_prof.cu)
__device__ long long g_seq_prof[16];
#define SQ_STAMP(i) if (step == 8 && blockIdx.x == 1 && blockIdx.y == 3) g_seq_prof[i] = clock64();
#else
#define SQ_STAMP(i)
#endif

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Spins until the arrival counters flags[j_lo..j_hi] have all reached `want` (acquire, gpu scope).  Returns false after a
// bounded wait (counted in g_rnn_seq_timeouts) so that a violated co-residency assumption cannot hang the launch.
__device__ __forceinline__ bool rnn_wait_tiles(const unsigned* flags, int j_lo, int j_hi, unsigned want) {
  for (int j = j_lo; j <= j_hi; ++j) {
    unsigned spins = 0;
    while (ld_acquire_gpu(flags + j) < want)
      if (++spins > (1u << 21)) { atomicAdd(&g_rnn_seq_timeouts, 1u); return false; }
  }
  return true;
}

__global__ void __cluster_dims__(RS_KS, 1, 1) __launch_bounds__(RS_THREADS, 1)
rnn_seq_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const SeqArgs sa,
               int M, int Mpad, int N, int NT, int kb_per_cta) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t A_TILE = 128 * 128, W_BYTES = (uint32_t)NT * 128, W_STAGE = (W_BYTES + 1023) & ~1023u;
  const int SP = NT + 4;
  const int per = Mpad / RS_KS;
  uint8_t* w_smem = smem;                                              // resident weight slab: kb x [NT][64] bf16
  uint8_t* a_smem = smem + (size_t)kb_per_cta * W_STAGE;               // hidden-state slab of the current step
  float* S = (float*)(a_smem + (size_t)kb_per_cta * A_TILE);           // partial accumulators, read by the peers
  uint64_t* bars = (uint64_t*)((uint8_t*)S + (((size_t)((Mpad + 31) & ~31) * SP * 4 + 1023) & ~(size_t)1023));
  uint32_t* tmem_slot = (uint32_t*)(bars + 10);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = blockIdx.x;
  const int tile = blockIdx.y, n0 = tile * NT, tiles = gridDim.y;
  const uint32_t tmem_cols = NT <= 32 ? 32 : (NT <= 64 ? 64 : (NT <= 128 ? 128 : 256));
  const uint32_t done_bar = smem_u32(bars + 8), w_bar = smem_u32(bars + 9);

  if (tid == RS_EPI) {
    for (int s = 0; s < kb_per_cta; ++s) mbar_init(smem_u32(bars + s), 1);
    mbar_init(done_bar, 1);
    mbar_init(w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == RS_EPI / 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int k_begin = (int)rank * kb_per_cta * TC_BK;

  if (tid == RS_EPI) {                                                  // the weight slab, once
    mbar_expect_tx(w_bar, (uint32_t)kb_per_cta * W_BYTES);
    for (int s = 0; s < kb_per_cta; ++s)
      tma_load_2d(smem_u32(w_smem + (size_t)s * W_STAGE), &tmW, k_begin + s * TC_BK, n0, w_bar);
  }
  const int NT4 = NT >> 2, elems = per * NT4;
  bool dead = false;                                                    // a flag wait timed out: stop waiting

  for (int step = 0; step < sa.n_steps; ++step) {
    const int tau = sa.tau0 + step * sa.dtau;
    const uint32_t ph = (uint32_t)step & 1u;
    float4 cold[RS_MAXE], gt[RS_MAXE];
    if (warp == RS_EPI / 32) {
      // lane s waits for the (one or two) tiles producing K block s and loads that block (as in rnn_wave_kernel)
      if (lane == 0) { SQ_STAMP(0) }
      bool bad = false;
      if (lane < kb_per_cta) {
        const int k0 = k_begin + lane * TC_BK;
        if (step > 0 && !dead)
          bad = !rnn_wait_tiles(g_rnn_flags[0], k0 / NT, min(tiles - 1, (k0 + TC_BK - 1) / NT), (unsigned)(RS_KS * step));
        asm volatile("fence.proxy.async.global;" ::: "memory");
        const uint32_t bar = smem_u32(bars + lane);
        mbar_expect_tx(bar, (uint32_t)Mpad * 128);
        tma_load_3d(smem_u32(a_smem + (size_t)lane * A_TILE), &tmA, k0, 0, tau - sa.dtau, bar);
      }
      if (__any_sync(0xffffffffu, bad)) dead = true;
      if (lane == 0) {
        SQ_STAMP(1)
        if (step == 0) mbar_wait(w_bar, 0);
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        SQ_STAMP(2)
        for (int s = 0; s < kb_per_cta; ++s) {
          mbar_wait(smem_u32(bars + s), ph);
          tc_fence_after();
          if (s == 0) { SQ_STAMP(3) }
          const uint32_t a_src = smem_u32(a_smem + (size_t)s * A_TILE), w_src = smem_u32(w_smem + (size_t)s * W_STAGE);
#pragma unroll
          for (int k = 0; k < TC_BK / TC_UMMA_K; ++k)
            tc_mma_bf16(tmem_base, make_smem_desc(a_src + k * 32, 16, 1024), make_smem_desc(w_src + k * 32, 16, 1024), idesc,
                        (s > 0 || k > 0) ? 1u : 0u);
        }
        tc_commit(done_bar);
        SQ_STAMP(4)
      }
      __syncwarp();
    } else {
      // epilogue operands of this step do not depend on the recurrence: fetch them while the MMAs run
      const float* Ct = sa.C + (long long)tau * sa.c_ts;
      const float* Gt = sa.gate ? sa.gate + (long long)tau * sa.gate_ts : nullptr;
      long long offc[RS_MAXE], offg[RS_MAXE];
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
        const bool ok = e < elems && b < M && col < N;
        offc[i] = ok ? (long long)b * sa.ldc + col : 0;
        offg[i] = ok ? (long long)b * sa.ldgate + col : 0;
      }
      const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f), one = make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) cold[i] = sa.beta != 0.f ? *reinterpret_cast<const float4*>(Ct + offc[i]) : zero;
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) gt[i] = Gt ? *reinterpret_cast<const float4*>(Gt + offg[i]) : one;
      mbar_wait(done_bar, ph);
      tc_fence_after();
      if (tid == 0) { SQ_STAMP(5) }
    }
    if (step > 0) asm volatile("barrier.cluster.wait.aligned;" ::: "memory");   // peers finished reading my previous S
    if (warp < RS_EPI / 32) {
      const int q = warp & 3;
      if (q * 32 < Mpad) {
        float* Srow = S + (q * 32 + lane) * SP;
#pragma unroll
        for (int h = 0; h < 2; ++h) {         // two TMEM loads in flight per wait
          uint32_t r[2][16];
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int c0 = (warp >> 2) * 16 + 64 * (2 * h + i);
            if (c0 < NT) tc_ld16_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r[i]);
          }
          tc_ld_wait();
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int c0 = (warp >> 2) * 16 + 64 * (2 * h + i);
            if (c0 < NT) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                reinterpret_cast<float4*>(Srow + c0)[j] = make_float4(__uint_as_float(r[i][4 * j]), __uint_as_float(r[i][4 * j + 1]),
                                                                      __uint_as_float(r[i][4 * j + 2]), __uint_as_float(r[i][4 * j + 3]));
            }
          }
        }
      }
    }
    tc_fence_before();
    if (tid == 0) { SQ_STAMP(6) }
    cluster_sync_all();
    tc_fence_after();
    if (tid == 0) { SQ_STAMP(7) }
    float4 acc[RS_MAXE];
    if (warp < RS_EPI / 32) {
      float4 part[RS_MAXE][RS_KS];
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4;
        const uint32_t addr = smem_u32(S + ((int)rank * per + (e < elems ? bi : 0)) * SP + (e < elems ? n : 0));
#pragma unroll
        for (int q = 0; q < RS_KS; ++q) part[i][q] = ld_dsmem_v4(addr, (q + rank) & (RS_KS - 1));   // staggered: 8 CTAs read 8 different peers
      }
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < RS_KS; ++q) { v.x += part[i][q].x; v.y += part[i][q].y; v.z += part[i][q].z; v.w += part[i][q].w; }
        acc[i] = v;
      }
      float dep = 0.f;
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) dep += acc[i].x + acc[i].y + acc[i].z + acc[i].w;
      asm volatile("barrier.cluster.arrive.release.aligned;" ::"f"(dep) : "memory");
      if (tid == 0) { SQ_STAMP(8) }
      // epilogue: the bf16 copy (the next step's operand) first, then the arrival, then the fp32 store
      float* Ct = sa.C + (long long)tau * sa.c_ts;
      __nv_bfloat16* Bt = sa.Cb + (long long)tau * sa.cb_ts;
      float4 outv[RS_MAXE];
      bool okv[RS_MAXE];
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
        okv[i] = e < elems && b < M && col < N;
        float v[4] = {acc[i].x, acc[i].y, acc[i].z, acc[i].w};
        const float c4[4] = {cold[i].x, cold[i].y, cold[i].z, cold[i].w};
        const float g4[4] = {gt[i].x, gt[i].y, gt[i].z, gt[i].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          v[j] = fmaf(sa.beta, c4[j], v[j]);
          if (sa.act == ACT_RELU) v[j] = fmaxf(v[j], 0.f);
          if (g4[j] <= 0.f) v[j] = 0.f;
        }
        outv[i] = make_float4(v[0], v[1], v[2], v[3]);
        if (okv[i]) {
          __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
          *reinterpret_cast<uint2*>(Bt + (long long)b * N + col) =
              make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        }
      }
      asm volatile("fence.proxy.async.global;" ::: "memory");
      if (tid == 0) { SQ_STAMP(9) }
      asm volatile("bar.sync 1, %0;" ::"n"(RS_EPI) : "memory");
      // (the release is cumulative over the stores bar.sync ordered before it: no separate fence)
      if (tid == 0) { red_release_gpu_add(&g_rnn_flags[0][tile], 1u); SQ_STAMP(10) }
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
        if (okv[i]) *reinterpret_cast<float4*>(Ct + (long long)b * sa.ldc + col) = outv[i];
      }
    } else {
      asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    }
  }
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
  if (warp == RS_EPI / 32) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
  rnn_launch_epilogue(tid);
}

// ------------------------------------------------------------------------------------------ two-lane persistent recurrence
// rnn_seq_kernel with the K split over 4-CTA clusters and up to TWO independent recurrences ("lanes": the forward and
// the reverse direction of a bidirectional layer, each with its own weights, buffers and arrival counters) running
// side by side in one launch: grid (4, tiles, lanes), 16 tiles of NT = 128 columns per lane for a 2048-wide layer
// = 64 CTAs per lane, 128 of the 148 SMs for both.  Per CTA: W slab NT x K/4 (128 KB bf16 at K = 2048) resident,
// the (batch x K/4) slab of h_{t-1} at a Mpad x 128 B pitch per 64-wide K block (64 KB at batch 64), partials S.
// Against the 8-way split: the DSMEM reduce-scatter moves half the bytes (4 partials of 16 rows x 128 columns per
// CTA instead of 8 x 8 rows x 144), the MMA count per CTA doubles (32 x 128x128x16, still ~1 us), and two lanes no
// longer time-share the SMs launch by launch (the BiRNN issued 2 x 16 per-step launches per layer, each holding 120
// SMs).  A single lane leaves 84 SMs to whatever else is in flight (weight-gradient GEMMs on a side stream).
// Batch rows <= 64 (above that the h slab does not fit next to the weights: rnn_seq_kernel).  Per-step arithmetic is
// deterministic and independent of the number of lanes (bit-identical results 1-lane vs 2-lane).
constexpr int RW_KS = 4;
constexpr int RW_MAX_TILES = 16;
struct WaveLane {
  int n_steps, tau0, dtau, act;           // steps s = 0 .. n_steps-1 write time tau0 + s*dtau from A[time tau - dtau]
  float beta;
  float* C; long long ldc, c_ts;          // fp32 pre-activation / upstream gradient in, result out
  const float* gate; long long ldgate, gate_ts;
  __nv_bfloat16* Cb; long long ldcb, cb_ts;   // bf16 copy of the result = the next step's A operand (row pitch, time stride)
  unsigned* flags;                        // [tiles] arrival counters, zero before the launch
};
struct WaveArgs { WaveLane lane[2]; };
#ifdef TACORL_STEP_PROFILE                    // stage stamps of one CTA at step 32 (scripts/prof/step_prof.cu)
__device__ long long g_wave_prof[48];
#define WV_STAMP(i) if (step == 32 && blockIdx.x == 1 && blockIdx.y == 3 && blockIdx.z == 0) g_wave_prof[i] = clock64();
#else
#define WV_STAMP(i)
#endif

__global__ void __launch_bounds__(RS_THREADS, 1)
rnn_wave_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmW0,
                const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmW1,
                const __grid_constant__ WaveArgs wa, int M, int Mpad, int N, int NT, int kb_per_cta) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t W_BYTES = (uint32_t)NT * 128, W_STAGE = (W_BYTES + 1023) & ~1023u, A_PITCH = (uint32_t)Mpad * 128;
  const int SP = NT + 4;
  const int per = Mpad / RW_KS;
  uint8_t* w_smem = smem;                                              // resident weight slab: kb x [NT][64] bf16
  uint8_t* a_smem = smem + (size_t)kb_per_cta * W_STAGE;               // h slab of the current step: kb x [Mpad][64] bf16
  // (UMMA M = 128 reads 128 rows from each stage base: rows >= Mpad are the next stage / the head of S -- never drained)
  float* S = (float*)(a_smem + (size_t)kb_per_cta * A_PITCH);          // partial accumulators, read by the peers
  uint64_t* bars = (uint64_t*)((uint8_t*)S + (((size_t)((Mpad + 31) & ~31) * SP * 4 + 1023) & ~(size_t)1023));
  uint32_t* tmem_slot = (uint32_t*)(bars + 10);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = blockIdx.x;                                    // == %cluster_ctarank (cluster dims (4,1,1))
  const int tile = blockIdx.y, n0 = tile * NT, tiles = gridDim.y;
  const WaveLane& sa = wa.lane[blockIdx.z];
  const CUtensorMap* tmA = blockIdx.z ? &tmA1 : &tmA0;
  const CUtensorMap* tmW = blockIdx.z ? &tmW1 : &tmW0;
  const uint32_t tmem_cols = NT <= 32 ? 32 : (NT <= 64 ? 64 : 128);
  const uint32_t done_bar = smem_u32(bars + 8), w_bar = smem_u32(bars + 9);

  if (tid == RS_EPI) {
    for (int s = 0; s < kb_per_cta; ++s) mbar_init(smem_u32(bars + s), 1);
    mbar_init(done_bar, 1);
    mbar_init(w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == RS_EPI / 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int k_begin = (int)rank * kb_per_cta * TC_BK;

  if (tid == RS_EPI) {                                                  // the weight slab, once
    mbar_expect_tx(w_bar, (uint32_t)kb_per_cta * W_BYTES);
    for (int s = 0; s < kb_per_cta; ++s)
      tma_load_2d(smem_u32(w_smem + (size_t)s * W_STAGE), tmW, k_begin + s * TC_BK, n0, w_bar);
  }
  const int NT4 = NT >> 2, elems = per * NT4;
  bool dead = false;                                                    // a flag wait timed out: stop waiting

  for (int step = 0; step < sa.n_steps; ++step) {
    const int tau = sa.tau0 + step * sa.dtau;
    const uint32_t ph = (uint32_t)step & 1u;
    float4 cold[RS_MAXE], gt[RS_MAXE];
    if (warp == RS_EPI / 32) {
      // K block s of the h slab is loaded by lane s as soon as the tiles that produce it have all arrived: when the
      // slowest producer arrives, only its own blocks are still to be fetched.  Each lane's TMA read is ordered after
      // its own acquire by the proxy fence.
      if (lane == 0) { WV_STAMP(0) }
      bool bad = false;
      if (lane < kb_per_cta) {
        const int k0 = k_begin + lane * TC_BK;
        if (step > 0 && !dead)
          bad = !rnn_wait_tiles(g_rnn_flags[blockIdx.z], k0 / NT, min(tiles - 1, (k0 + TC_BK - 1) / NT), (unsigned)(RW_KS * step));
        WV_STAMP(24 + lane)
        asm volatile("fence.proxy.async.global;" ::: "memory");
        const uint32_t bar = smem_u32(bars + lane);
        mbar_expect_tx(bar, A_PITCH);
        tma_load_3d(smem_u32(a_smem + (size_t)lane * A_PITCH), tmA, k0, 0, tau - sa.dtau, bar);
        WV_STAMP(32 + lane)
      }
      if (__any_sync(0xffffffffu, bad)) dead = true;
      if (lane == 0) {
        WV_STAMP(2)
        if (step == 0) mbar_wait(w_bar, 0);
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        for (int s = 0; s < kb_per_cta; ++s) {
          mbar_wait(smem_u32(bars + s), ph);
          tc_fence_after();
          WV_STAMP(16 + s)
          const uint32_t a_src = smem_u32(a_smem + (size_t)s * A_PITCH), w_src = smem_u32(w_smem + (size_t)s * W_STAGE);
#pragma unroll
          for (int k = 0; k < TC_BK / TC_UMMA_K; ++k)
            tc_mma_bf16(tmem_base, make_smem_desc(a_src + k * 32, 16, 1024), make_smem_desc(w_src + k * 32, 16, 1024), idesc,
                        (s > 0 || k > 0) ? 1u : 0u);
        }
        tc_commit(done_bar);
        WV_STAMP(4)
      }
      __syncwarp();
    } else {
      // epilogue operands of this step do not depend on the recurrence: fetch them while the MMAs run
      const float* Ct = sa.C + (long long)tau * sa.c_ts;
      const float* Gt = sa.gate ? sa.gate + (long long)tau * sa.gate_ts : nullptr;
      long long offc[RS_MAXE], offg[RS_MAXE];
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
        const bool ok = e < elems && b < M && col < N;
        offc[i] = ok ? (long long)b * sa.ldc + col : 0;
        offg[i] = ok ? (long long)b * sa.ldgate + col : 0;
      }
      const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f), one = make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) cold[i] = sa.beta != 0.f ? *reinterpret_cast<const float4*>(Ct + offc[i]) : zero;
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) gt[i] = Gt ? *reinterpret_cast<const float4*>(Gt + offg[i]) : one;
      mbar_wait(done_bar, ph);
      tc_fence_after();
      if (tid == 0) { WV_STAMP(5) }
    }
    if (step > 0) asm volatile("barrier.cluster.wait.aligned;" ::: "memory");   // peers finished reading my previous S
    if (tid == 0) { WV_STAMP(3) }
    if (warp < RS_EPI / 32) {
      const int q = warp & 3;
      if (q * 32 < Mpad) {
        float* Srow = S + (q * 32 + lane) * SP;
        uint32_t r[2][16];
#pragma unroll
        for (int i = 0; i < 2; ++i) {           // two TMEM loads in flight per wait: column chunks w/4*16 + {0, 64}
          const int c0 = (warp >> 2) * 16 + 64 * i;
          if (c0 < NT) tc_ld16_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r[i]);
        }
        tc_ld_wait();
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = (warp >> 2) * 16 + 64 * i;
          if (c0 < NT) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              reinterpret_cast<float4*>(Srow + c0)[j] = make_float4(__uint_as_float(r[i][4 * j]), __uint_as_float(r[i][4 * j + 1]),
                                                                    __uint_as_float(r[i][4 * j + 2]), __uint_as_float(r[i][4 * j + 3]));
          }
        }
      }
    }
    tc_fence_before();
    if (tid == 0) { WV_STAMP(6) }
    cluster_sync_all();
    tc_fence_after();
    if (tid == 0) { WV_STAMP(7) }
    float4 acc[RS_MAXE];
    if (warp < RS_EPI / 32) {
      float4 part[RS_MAXE][RW_KS];
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4;
        const uint32_t addr = smem_u32(S + ((int)rank * per + (e < elems ? bi : 0)) * SP + (e < elems ? n : 0));
#pragma unroll
        for (int q = 0; q < RW_KS; ++q) part[i][q] = ld_dsmem_v4(addr, (q + rank) & (RW_KS - 1));   // staggered peers
      }
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {        // fixed order (K slab rank, rank+1, ...): deterministic
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < RW_KS; ++q) { v.x += part[i][q].x; v.y += part[i][q].y; v.z += part[i][q].z; v.w += part[i][q].w; }
        acc[i] = v;
      }
      float dep = 0.f;
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) dep += acc[i].x + acc[i].y + acc[i].z + acc[i].w;
      asm volatile("barrier.cluster.arrive.release.aligned;" ::"f"(dep) : "memory");
      if (tid == 0) { WV_STAMP(8) }
      // epilogue: the bf16 copy (the next step's operand) first, then the arrival, then the fp32 store
      float* Ct = sa.C + (long long)tau * sa.c_ts;
      __nv_bfloat16* Bt = sa.Cb + (long long)tau * sa.cb_ts;
      float4 outv[RS_MAXE];
      bool okv[RS_MAXE];
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
        okv[i] = e < elems && b < M && col < N;
        float v[4] = {acc[i].x, acc[i].y, acc[i].z, acc[i].w};
        const float c4[4] = {cold[i].x, cold[i].y, cold[i].z, cold[i].w};
        const float g4[4] = {gt[i].x, gt[i].y, gt[i].z, gt[i].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          v[j] = fmaf(sa.beta, c4[j], v[j]);
          if (sa.act == ACT_RELU) v[j] = fmaxf(v[j], 0.f);
          if (g4[j] <= 0.f) v[j] = 0.f;
        }
        outv[i] = make_float4(v[0], v[1], v[2], v[3]);
        if (okv[i]) {
          __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
          *reinterpret_cast<uint2*>(Bt + (long long)b * sa.ldcb + col) =
              make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        }
      }
      asm volatile("fence.proxy.async.global;" ::: "memory");
      if (tid == 0) { WV_STAMP(9) }
      asm volatile("bar.sync 1, %0;" ::"n"(RS_EPI) : "memory");
      // (the release is cumulative over the stores bar.sync ordered before it: no separate fence)
      if (tid == 0) { red_release_gpu_add(&g_rnn_flags[blockIdx.z][tile], 1u); WV_STAMP(10) }
#pragma unroll
      for (int i = 0; i < RS_MAXE; ++i) {
        const int e = tid + i * RS_EPI;
        const int bi = e / NT4, n = (e - bi * NT4) * 4, b = (int)rank * per + bi, col = n0 + n;
        if (okv[i]) *reinterpret_cast<float4*>(Ct + (long long)b * sa.ldc + col) = outv[i];
      }
      if (tid == 0) { WV_STAMP(11) }
    } else {
      asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    }
  }
  if (sa.n_steps > 0) asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
  if (warp == RS_EPI / 32) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
  rnn_launch_epilogue(tid);
}

// ------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D bf16 tensor map: inner dimension `inner` (contiguous), `outer` rows of pitch `ld` elements.
static int make_tmap(CUtensorMap* tm, const void* base, long long inner, long long outer, long long ld,
                     int box_inner, int box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  TACORL_REQUIRE(fn, "gemm_tc: cuTensorMapEncodeTiled is not available from the driver");
  TACORL_REQUIRE(((uintptr_t)base & 15) == 0 && (ld * 2) % 16 == 0,
                 "gemm_tc: TMA operand must be 16-byte aligned with a 16-byte multiple pitch (ld=%lld)", ld);
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  TACORL_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled failed (%d) inner=%lld outer=%lld ld=%lld", (int)r,
                 inner, outer, ld);
  return 0;
}

template <int BN, bool A_MN, bool B_MN>
static int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const TcEpilogue& ep, int M, int N, int K,
                     int splits, cudaStream_t st) {
  constexpr int kStages = BN >= 128 ? 5 : 6;
  constexpr size_t smem = (size_t)kStages * (TC_BM * TC_BK * 2 + BN * TC_BK * 2) + (2 * kStages + 4) * 8 + 16 + 1024;
  static bool configured = false;
  auto kern = gemm_tc_kernel<BN, A_MN, B_MN, kStages>;
  if (!configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int total_kb = cdiv(K, TC_BK);
  const int per = cdiv(total_kb, splits);
  const int zs = cdiv(total_kb, per);
  const long long tiles = (long long)cdiv(N, BN) * cdiv(M, TC_BM);
  const int ctas = (int)min(tiles, (long long)max(1, 148 / zs));   // persistent: ~one CTA per SM in total
  dim3 grid(ctas, 1, zs);
  kern<<<grid, TC_THREADS, smem, st>>>(ta, tb, ep, M, N, K, per);
  TACORL_LAUNCH_CHECK();
  return 0;
}

__global__ void tc_splitk_reduce_kernel(int M, int N, int splits, const float* __restrict__ partial, TcEpilogue ep) {
  const long long total = (long long)M * N;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(idx / N), col = (int)(idx % N);
    float s = 0.f;
    for (int z = 0; z < splits; ++z) s += partial[(long long)z * total + idx];
    float v = ep.alpha * s;
    if (ep.beta != 0.f && ep.C) v = fmaf(ep.beta, ep.C[(long long)row * ep.ldc + col], v);
    if (ep.bias) v += __ldg(ep.bias + col);
    if (ep.Cpre) ep.Cpre[(long long)row * ep.ldpre + col] = v;
    if (ep.act == ACT_RELU) v = fmaxf(v, 0.f);
    else if (ep.act == ACT_SILU) v = v / (1.f + __expf(-v));
    if (ep.gate && ep.gate[(long long)row * ep.ldgate + col] <= 0.f) v = 0.f;
    if (ep.C) ep.C[(long long)row * ep.ldc + col] = v;
    if (ep.Cb) ep.Cb[(long long)row * ep.ldcb + col] = __float2bfloat16(v);
  }
}

// C[M][N] = epilogue(A[M][K] . W[N][K]^T) for M <= 128 through skinny_cluster_kernel; returns 1 when the shape is
// outside what the kernel covers (the caller then uses the tiled kernel).
static int launch_skinny_cluster(const void* A, long long lda, const void* W, long long ldw, int M, int N, int K,
                                 const TcEpilogue& ep, cudaStream_t st) {
  if (M < 1 || M > 128 || K % (TC_BK * RS_KS) != 0 || N % 4 != 0) return 1;
  auto al16 = [](const void* p, long long ld, int elt) { return p == nullptr || (((uintptr_t)p & 15) == 0 && (ld * elt) % 16 == 0); };
  if (!al16(ep.C, ep.ldc, 4) || !al16(ep.gate, ep.ldgate, 4) || !al16(ep.Cpre, ep.ldpre, 4) || !al16(ep.bias, 4, 4) ||
      !(ep.Cb == nullptr || (((uintptr_t)ep.Cb & 7) == 0 && ep.ldcb % 4 == 0)))
    return 1;
  const int Mpad = (M + 15) & ~15, kb = K / (TC_BK * RS_KS);
  const int NT = 16 * cdiv(N, 16 * RS_MAX_TILES), tiles = cdiv(N, NT);
  if (NT > 256 || kb > 8 || (Mpad / RS_KS) * (NT / 4) > RS_MAXE * RS_EPI) return 1;
  const size_t stage = 128 * 128 + (((size_t)NT * 128 + 1023) & ~(size_t)1023);
  const size_t s_bytes = ((size_t)Mpad * (NT + 4) * 4 + 1023) & ~(size_t)1023;
  const size_t smem = std::max((size_t)kb * stage, s_bytes) + 9 * 8 + 16 + 1024;
  if (smem > 227 * 1024) return 1;
  CUtensorMap ta, tw;
  int rc;
  if ((rc = make_tmap(&ta, A, K, M, lda, 64, Mpad))) return rc;
  if ((rc = make_tmap(&tw, W, K, N, ldw, 64, NT))) return rc;
  static size_t configured = 0;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(skinny_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  skinny_cluster_kernel<<<dim3(RS_KS, tiles), RS_THREADS, smem, st>>>(ta, tw, ep, M, Mpad, N, NT, kb);
  TACORL_LAUNCH_CHECK();
  return 0;
}

static int g_rnn_seq_enabled = -1;
bool rnn_seq_enabled() {
  if (g_rnn_seq_enabled < 0) { const char* e = getenv("TACORL_RNN_SEQ"); g_rnn_seq_enabled = !(e && e[0] == '0'); }
  return g_rnn_seq_enabled != 0;
}
void rnn_seq_set_enabled(int on) { g_rnn_seq_enabled = on < 0 ? 0 : (on > 2 ? 2 : on); }   // 2: lanes launched one by one
int rnn_seq_mode() { rnn_seq_enabled(); return g_rnn_seq_enabled; }

// Two persistent launches must never be co-scheduled (each spin-waits on its own clusters being resident): chain
// them through an event, whatever streams they are issued on.  Inside a stream capture the chain only links
// launches of the same capture (an event recorded elsewhere cannot be waited on there; the graph launch itself is
// stream-ordered after earlier work).
static cudaEvent_t g_chain_ev[64] = {};
static cudaStream_t g_chain_stream[64] = {};
static unsigned long long g_chain_capture[64] = {};
static bool g_chain_recorded[64] = {};
static int chain_slot(cudaStream_t st, int* dev, unsigned long long* cid) {
  TACORL_CHECK_CUDA(cudaGetDevice(dev));
  TACORL_REQUIRE(*dev >= 0 && *dev < 64, "persistent launch: device index %d out of range", *dev);
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  *cid = 0;
  TACORL_CHECK_CUDA(cudaStreamGetCaptureInfo(st, &cs, cid));
  if (cs != cudaStreamCaptureStatusActive) *cid = 0;
  if (!g_chain_ev[*dev]) TACORL_CHECK_CUDA(cudaEventCreateWithFlags(&g_chain_ev[*dev], cudaEventDisableTiming));
  return 0;
}
static int persistent_chain_enter(cudaStream_t st) {
  int dev; unsigned long long cid; int rc;
  if ((rc = chain_slot(st, &dev, &cid))) return rc;
  // (a launch on the stream of the previous persistent launch is ordered behind it already)
  if (g_chain_recorded[dev] && g_chain_capture[dev] == cid && g_chain_stream[dev] != st)
    TACORL_CHECK_CUDA(cudaStreamWaitEvent(st, g_chain_ev[dev], 0));
  return 0;
}
static int persistent_chain_leave(cudaStream_t st) {
  int dev; unsigned long long cid; int rc;
  if ((rc = chain_slot(st, &dev, &cid))) return rc;
  TACORL_CHECK_CUDA(cudaEventRecord(g_chain_ev[dev], st));
  g_chain_recorded[dev] = true; g_chain_capture[dev] = cid; g_chain_stream[dev] = st;
  return 0;
}

// Runs n_steps dependent steps C[tau] = epi(beta*C[tau] + A[tau - dtau] . W^T), tau = tau0 + s*dtau, in one launch of
// rnn_seq_kernel.  Ab: dense bf16 [T][M][K] (K == N: the recurrence feeds its own output back), W: bf16 [N][K].
// Returns 1 when the shape / device cannot run the persistent kernel (the caller then launches step by step).
int rnn_seq_tc(const void* Ab, int T, const void* W, long long ldw, int M, int N, int K, int tau0, int dtau, int n_steps,
               float beta, float* C, long long ldc, long long c_ts, const float* gate, long long ldgate, long long gate_ts,
               void* Cb, int act, unsigned* flags, cudaStream_t st) {
  if (!rnn_seq_enabled() || n_steps < 2) return 1;
  if (M < 1 || M > 128 || K != N || K % (TC_BK * RS_KS) != 0 || N % 4 != 0 || !Cb || !C || !flags) return 1;
  auto al16 = [](const void* p, long long ld) { return p == nullptr || (((uintptr_t)p & 15) == 0 && (ld * 4) % 16 == 0); };
  if (!al16(C, ldc) || !al16(C, c_ts) || !al16(gate, ldgate) || !al16(gate, gate_ts) || ((uintptr_t)Cb & 15) != 0) return 1;
  const int Mpad = (M + 15) & ~15, kb = K / (TC_BK * RS_KS);
  const int NT = 16 * cdiv(N, 16 * RS_MAX_TILES), tiles = cdiv(N, NT);
  if (NT > 256 || kb > 8 || (Mpad / RS_KS) * (NT / 4) > RS_MAXE * RS_EPI) return 1;
  const size_t w_stage = ((size_t)NT * 128 + 1023) & ~(size_t)1023;
  const size_t s_bytes = ((size_t)((Mpad + 31) & ~31) * (NT + 4) * 4 + 1023) & ~(size_t)1023;
  const size_t smem = (size_t)kb * (w_stage + 128 * 128) + s_bytes + 10 * 8 + 16 + 1024;
  if (smem > 227 * 1024) return 1;
  static size_t configured = 0;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(rnn_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  {   // every cluster of the grid must be resident at once: the steps are chained by spin-waits on peers
    static size_t checked_smem = 0;
    static int max_clusters = 0;
    if (checked_smem != smem) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(RS_KS, tiles); cfg.blockDim = dim3(RS_THREADS); cfg.dynamicSmemBytes = smem;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = RS_KS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, rnn_seq_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
      max_clusters = n; checked_smem = smem;
    }
    if (max_clusters < tiles) return 1;
  }
  CUtensorMap ta, tw;
  int rc;
  {
    EncodeTiledFn fn = get_encode_fn();
    TACORL_REQUIRE(fn, "rnn_seq: cuTensorMapEncodeTiled is not available from the driver");
    TACORL_REQUIRE(((uintptr_t)Ab & 15) == 0, "rnn_seq: hidden-state buffer must be 16-byte aligned");
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)M, (cuuint64_t)T};
    cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)M * K * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)Mpad, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(&ta, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(Ab), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    TACORL_REQUIRE(r == CUDA_SUCCESS, "rnn_seq: cuTensorMapEncodeTiled failed (%d) K=%d M=%d T=%d", (int)r, K, M, T);
  }
  if ((rc = make_tmap(&tw, W, K, N, ldw, 64, NT))) return rc;
  SeqArgs sa;
  sa.n_steps = n_steps; sa.tau0 = tau0; sa.dtau = dtau; sa.beta = beta; sa.C = C; sa.ldc = ldc; sa.c_ts = c_ts;
  sa.gate = gate; sa.ldgate = ldgate; sa.gate_ts = gate_ts; sa.Cb = (__nv_bfloat16*)Cb; sa.cb_ts = (long long)M * N;
  sa.act = act; sa.flags = flags;
  int rc2;
  if ((rc2 = persistent_chain_enter(st))) return rc2;
  rnn_seq_kernel<<<dim3(RS_KS, tiles), RS_THREADS, smem, st>>>(ta, tw, sa, M, Mpad, N, NT, kb);
  TACORL_LAUNCH_CHECK();
  if ((rc2 = persistent_chain_leave(st))) return rc2;
  return 0;
}

// Runs n_lanes (1 or 2) independent recurrences of n_steps dependent steps each in ONE launch of rnn_wave_kernel.
// Returns 1 when the shape / device cannot run it (the caller falls back to rnn_seq_tc / step-by-step launches).
int rnn_wave_tc(const WaveLaneHost* lanes, int n_lanes, int T, int M, int N, int K, cudaStream_t st) {
  if (!rnn_seq_enabled() || n_lanes < 1 || n_lanes > 2) return 1;
  if (n_lanes == 2 && rnn_seq_mode() == 2) {      // diagnostic mode: the same arithmetic, one lane per launch
    int rc = rnn_wave_tc(lanes, 1, T, M, N, K, st);
    return rc ? rc : rnn_wave_tc(lanes + 1, 1, T, M, N, K, st);
  }
  if (M < 1 || M > 64 || K != N || K % (TC_BK * RW_KS) != 0 || N % 4 != 0) return 1;
  const int Mpad = (M + 15) & ~15, kb = K / (TC_BK * RW_KS);
  const int NT = 16 * cdiv(N, 16 * RW_MAX_TILES), tiles = cdiv(N, NT);
  if (NT > 128 || kb > 8 || (Mpad / RW_KS) * (NT / 4) > RS_MAXE * RS_EPI) return 1;
  auto al16 = [](const void* p, long long ld) { return p == nullptr || (((uintptr_t)p & 15) == 0 && (ld * 4) % 16 == 0); };
  int max_steps = 0;
  for (int l = 0; l < n_lanes; ++l) {
    const WaveLaneHost& h = lanes[l];
    if (!h.Ab || !h.W || !h.C || !h.Cb || !h.flags || h.n_steps < 0) return 1;
    if (!al16(h.C, h.ldc) || !al16(h.C, h.c_ts) || !al16(h.gate, h.ldgate) || !al16(h.gate, h.gate_ts)) return 1;
    if (((uintptr_t)h.Cb & 7) != 0 || h.ldcb % 4 != 0 || h.cb_ts % 4 != 0) return 1;
    if (((uintptr_t)h.Ab & 15) != 0 || (h.lda * 2) % 16 != 0 || (h.a_ts * 2) % 16 != 0) return 1;
    max_steps = std::max(max_steps, h.n_steps);
  }
  if (max_steps < 2) return 1;
  const size_t w_stage = ((size_t)NT * 128 + 1023) & ~(size_t)1023, a_pitch = (size_t)Mpad * 128;
  const size_t s_bytes = ((size_t)((Mpad + 31) & ~31) * (NT + 4) * 4 + 1023) & ~(size_t)1023;
  // the last h stage is read as a 128-row UMMA operand: keep 16 KB behind its base inside the allocation
  const size_t tail = std::max(a_pitch + s_bytes + 256, (size_t)16384 + 256);
  const size_t smem = (size_t)kb * w_stage + (size_t)(kb - 1) * a_pitch + tail + 1024;
  if (smem > 227 * 1024) return 1;
  static size_t configured = 0;
  if (smem > configured) {
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(rnn_wave_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TACORL_CHECK_CUDA(cudaFuncSetAttribute(rnn_wave_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 0));
    configured = smem;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(RW_KS, tiles, n_lanes); cfg.blockDim = dim3(RS_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = RW_KS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  {   // every cluster of the grid must be resident at once: the steps are chained by spin-waits on peers
    static size_t checked_smem = 0;
    static int max_clusters = 0;
    if (checked_smem != smem) {
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, rnn_wave_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
      max_clusters = n; checked_smem = smem;
    }
    if (max_clusters < tiles * n_lanes) return 1;
  }
  EncodeTiledFn fn = get_encode_fn();
  TACORL_REQUIRE(fn, "rnn_wave: cuTensorMapEncodeTiled is not available from the driver");
  CUtensorMap ta[2], tw[2];
  WaveArgs wa;
  int rc;
  for (int l = 0; l < 2; ++l) {
    const WaveLaneHost& h = lanes[l < n_lanes ? l : 0];
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)M, (cuuint64_t)T};
    cuuint64_t strides[2] = {(cuuint64_t)h.lda * 2, (cuuint64_t)h.a_ts * 2};
    cuuint32_t box[3] = {64, (cuuint32_t)Mpad, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(&ta[l], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(h.Ab), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    TACORL_REQUIRE(r == CUDA_SUCCESS, "rnn_wave: cuTensorMapEncodeTiled failed (%d) K=%d M=%d T=%d", (int)r, K, M, T);
    if ((rc = make_tmap(&tw[l], h.W, K, N, h.ldw, 64, NT))) return rc;
    WaveLane& d = wa.lane[l];
    d.n_steps = l < n_lanes ? h.n_steps : 0; d.tau0 = h.tau0; d.dtau = h.dtau; d.act = h.act; d.beta = h.beta;
    d.C = h.C; d.ldc = h.ldc; d.c_ts = h.c_ts; d.gate = h.gate; d.ldgate = h.ldgate; d.gate_ts = h.gate_ts;
    d.Cb = (__nv_bfloat16*)h.Cb; d.ldcb = h.ldcb; d.cb_ts = h.cb_ts; d.flags = h.flags;
  }
  if ((rc = persistent_chain_enter(st))) return rc;
  void* args[] = {&ta[0], &tw[0], &ta[1], &tw[1], &wa, (void*)&M, (void*)&Mpad, (void*)&N, (void*)&NT, (void*)&kb};
  TACORL_CHECK_CUDA(cudaLaunchKernelExC(&cfg, (const void*)rnn_wave_kernel, args));
  note_launch();
  if ((rc = persistent_chain_leave(st))) return rc;
  return 0;
}

unsigned rnn_seq_timeouts() {
  unsigned v = 0;
  cudaMemcpyFromSymbol(&v, g_rnn_seq_timeouts, sizeof(v));
  return v;
}

// Core entry: bf16 operands already in global memory.
//   A: a_mn ? stored [K][M] (pitch lda) : stored [M][K];   B: b_mn ? stored [K][N] : stored [N][K].
int gemm_tc_bf16(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, int M, int N,
                 int K, const TcArgs& e, float* ws, size_t ws_bytes, cudaStream_t st) {
  if (M == 0 || N == 0) return 0;
  TACORL_REQUIRE(K > 0, "gemm_tc: K must be positive");
  int BN = N <= 32 ? 32 : (N <= 64 ? 64 : 128);
  // skinny-M recurrent steps: many narrow N tiles (one fused kernel, no split-K round trip) beat 16 wide ones
  const bool skinny = M <= TC_BM && N >= 512 && K <= 8192 && e.split_k == 0;
  if (skinny) BN = b_mn ? 64 : 32;
  if (b_mn && BN < 64) BN = 64;
  int rc;
  if (skinny && !a_mn && !b_mn) {   // recurrent steps: cluster split-K with an in-cluster reduction
    TcEpilogue ep;
    ep.alpha = e.alpha; ep.beta = e.beta; ep.C = e.C; ep.ldc = e.ldc; ep.Cb = (__nv_bfloat16*)e.Cb; ep.ldcb = e.ldcb;
    ep.bias = e.bias; ep.act = e.act; ep.Cpre = e.Cpre; ep.ldpre = e.ldpre; ep.partial = nullptr;
    ep.gate = e.gate; ep.ldgate = e.ldgate;
    rc = launch_skinny_cluster(A, lda, B, ldb, M, N, K, ep, st);
    if (rc <= 0) return rc;
  }
  CUtensorMap ta, tb;
  if ((rc = a_mn ? make_tmap(&ta, A, M, K, lda, 64, 64) : make_tmap(&ta, A, K, M, lda, 64, TC_BM))) return rc;
  if ((rc = b_mn ? make_tmap(&tb, B, N, K, ldb, 64, 64) : make_tmap(&tb, B, K, N, ldb, 64, BN))) return rc;
  const long long ctas = (long long)cdiv(M, TC_BM) * cdiv(N, BN);
  const int total_kb = cdiv(K, TC_BK);
  int splits = e.split_k;
  if (splits <= 0) {
    splits = 1;
    if (ws && !skinny && ctas < 74 && total_kb >= 8) splits = (int)min((long long)cdiv(148, ctas), (long long)(total_kb / 4));
  }
  if (splits > total_kb) splits = total_kb;
  if (splits > 1 && (!ws || (size_t)splits * M * N * 4 > ws_bytes)) {
    splits = ws ? (int)(ws_bytes / ((size_t)M * N * 4)) : 1;
    if (splits < 1) splits = 1;
  }
  TcEpilogue ep;
  ep.alpha = e.alpha; ep.beta = e.beta; ep.C = e.C; ep.ldc = e.ldc; ep.Cb = (__nv_bfloat16*)e.Cb; ep.ldcb = e.ldcb;
  ep.bias = e.bias; ep.act = e.act; ep.Cpre = e.Cpre; ep.ldpre = e.ldpre; ep.partial = splits > 1 ? ws : nullptr;
  ep.gate = e.gate; ep.ldgate = e.ldgate;
#define TC_DISPATCH(BNV)                                                                                   \
  if (BN == BNV) {                                                                                         \
    if (!a_mn && !b_mn) rc = launch_tc<BNV, false, false>(ta, tb, ep, M, N, K, splits, st);                \
    else if (a_mn && !b_mn) rc = launch_tc<BNV, true, false>(ta, tb, ep, M, N, K, splits, st);             \
    else if (!a_mn && b_mn) rc = launch_tc<(BNV < 64 ? 64 : BNV), false, true>(ta, tb, ep, M, N, K, splits, st); \
    else rc = launch_tc<(BNV < 64 ? 64 : BNV), true, true>(ta, tb, ep, M, N, K, splits, st);               \
  }
  rc = -1;
  TC_DISPATCH(32) TC_DISPATCH(64) TC_DISPATCH(128)
#undef TC_DISPATCH
  if (rc) return rc;
  if (splits > 1) {
    // the kernel may have used fewer z-slices than `splits` when the K blocks do not divide evenly
    const int per = cdiv(total_kb, splits);
    const int used = cdiv(total_kb, per);
    ep.partial = nullptr;
    long long total = (long long)M * N;
    tc_splitk_reduce_kernel<<<(int)min((long long)1184, (total + 255) / 256), 256, 0, st>>>(M, N, used, ws, ep);
    TACORL_LAUNCH_CHECK();
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ fp32 -> bf16 staging
__global__ void cast_bf16_2d_kernel(const float* __restrict__ src, long long lds, long long rows, int cols,
                                    __nv_bfloat16* __restrict__ dst, long long ldd) {
  const long long total = rows * ldd;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / ldd; const int c = (int)(i % ldd);
    dst[i] = __float2bfloat16(c < cols ? src[r * lds + c] : 0.f);
  }
}

int cast_bf16_2d(const float* src, long long lds, long long rows, int cols, void* dst, long long ldd, cudaStream_t st) {
  if (rows == 0) return 0;
  long long total = rows * ldd;
  cast_bf16_2d_kernel<<<(int)min((long long)148 * 8, (total + 255) / 256), 256, 0, st>>>(src, lds, rows, cols,
                                                                                        (__nv_bfloat16*)dst, ldd);
  TACORL_LAUNCH_CHECK();
  return 0;
}

// dst[c][r] = bf16(src[r][c]) : 32x32 tiles through shared memory
__global__ void cast_transpose_bf16_kernel(const float* __restrict__ src, long long lds, int rows, int cols,
                                           __nv_bfloat16* __restrict__ dst, long long ldd) {
  __shared__ float tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? src[(long long)r * lds + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) dst[(long long)c * ldd + r] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}

int cast_transpose_bf16(const float* src, long long lds, int rows, int cols, void* dst, long long ldd, cudaStream_t st) {
  if (rows == 0 || cols == 0) return 0;
  cast_transpose_bf16_kernel<<<dim3(cdiv(cols, 32), cdiv(rows, 32)), dim3(32, 8), 0, st>>>(src, lds, rows, cols,
                                                                                          (__nv_bfloat16*)dst, ldd);
  TACORL_LAUNCH_CHECK();
  return 0;
}

// GemmArgs (fp32 operands, any transposition) on the tensor cores: operands are staged to bf16 in `ws`
// in their stored orientation (no transposes: stored-[K][rows] operands use the MN-major descriptors).
int gemm_tc_from_f32(const GemmArgs& g, float* ws, size_t ws_bytes, cudaStream_t st) {
  if (g.M == 0 || g.N == 0) return 0;
  // tiny contractions (goal-encoder / policy / Q MLPs at batch 64, distribution heads): two staging casts plus a
  // 148-SM tensor-core launch cost more than the whole fp32 FFMA GEMM, and fp32 is strictly more accurate
  if ((long long)g.M * g.N * g.K < (1LL << 24)) return gemm_f32(g, ws, ws_bytes, st);
  TACORL_REQUIRE(ws, "gemm_tc: workspace required");
  const long long a_rows = g.transA ? g.K : g.M, a_cols = g.transA ? g.M : g.K;
  const long long b_rows = g.transB ? g.N : g.K, b_cols = g.transB ? g.K : g.N;
  const long long lda = (a_cols + 7) & ~7LL, ldb = (b_cols + 7) & ~7LL;
  // caller-maintained bf16 copies (dense, pitch = column count) replace the staging cast when TMA can read them
  const bool a_ready = g.A_bf16 && lda == a_cols && ((uintptr_t)g.A_bf16 & 15) == 0;
  const bool b_ready = g.B_bf16 && ldb == b_cols && ((uintptr_t)g.B_bf16 & 15) == 0;
  Arena ar(ws, ws_bytes);
  const __nv_bfloat16* Ab = a_ready ? (const __nv_bfloat16*)g.A_bf16 : ar.take<__nv_bfloat16>((size_t)a_rows * lda);
  const __nv_bfloat16* Bb = b_ready ? (const __nv_bfloat16*)g.B_bf16 : ar.take<__nv_bfloat16>((size_t)b_rows * ldb);
  TACORL_REQUIRE(Ab && Bb, "gemm_tc: workspace too small for bf16 staging (%lld + %lld elements)", a_rows * lda,
                 b_rows * ldb);
  int rc;
  if (!a_ready && (rc = cast_bf16_2d(g.A, g.lda, a_rows, (int)a_cols, (void*)Ab, lda, st))) return rc;
  if (!b_ready && (rc = cast_bf16_2d(g.B, g.ldb, b_rows, (int)b_cols, (void*)Bb, ldb, st))) return rc;
  TcArgs e;
  e.alpha = g.alpha; e.beta = g.beta; e.C = g.C; e.ldc = g.ldc; e.bias = g.bias; e.act = g.act; e.Cpre = g.Cpre;
  e.ldpre = g.ldpre; e.split_k = g.split_k;
  return gemm_tc_bf16(Ab, lda, g.transA ? 1 : 0, Bb, ldb, g.transB ? 0 : 1, g.M, g.N, g.K, e,
                      (float*)(ar.base + ar.off), ar.left(), st);
}

}  // namespace tacorl
