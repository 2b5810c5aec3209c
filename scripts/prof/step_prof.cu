// Stage-level timing of the recurrent-step kernels (development tool, not part of the library).
// Build + run:  bash scripts/prof/build_step_prof.sh && build/step_prof
// Includes gemm_tc.cu directly with -DTACORL_STEP_PROFILE so the kernel records %globaltimer stamps.
#include "../../tacorl_b200/csrc/gemm_tc.cu"
#include <cstdio>
#include <vector>
#include <algorithm>

using namespace tacorl;
extern "C" const char* tacorl_last_error();

int main(int argc, char** argv) {
  const int M = argc > 1 ? atoi(argv[1]) : 128, N = 2048, K = 2048, STEPS = 64;
  __nv_bfloat16 *A, *W, *Cb;
  float *C, *ws;
  cudaMalloc(&A, (size_t)2 * 128 * K * 2); cudaMalloc(&W, (size_t)N * K * 2); cudaMalloc(&Cb, (size_t)2 * 128 * N * 2);
  cudaMalloc(&C, (size_t)128 * N * 4); cudaMalloc(&ws, 64 << 20);
  cudaMemset(A, 0, (size_t)2 * 128 * K * 2); cudaMemset(W, 0, (size_t)N * K * 2); cudaMemset(C, 0, (size_t)128 * N * 4);
  cudaStream_t st; cudaStreamCreate(&st);
  {  // how many clusters of each size can be co-resident (1 CTA / SM at ~200 KB of shared memory)?
    cudaFuncSetAttribute(skinny_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(skinny_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    for (int smem : {200 * 1024, 100 * 1024}) for (int cs : {1, 2, 4, 8, 16}) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(cs, 64); cfg.blockDim = dim3(RS_THREADS); cfg.dynamicSmemBytes = smem;
      cudaLaunchAttribute at; at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = cs; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
      cfg.attrs = &at; cfg.numAttrs = 1;
      int n = -1;
      cudaError_t e = cudaOccupancyMaxActiveClusters(&n, skinny_cluster_kernel, &cfg);
      printf("smem %3d KB cluster size %2d: max active clusters %d (%d CTAs) %s\n", smem >> 10, cs, n, n * cs, e == cudaSuccess ? "" : cudaGetErrorString(e));
    }
    cudaGetLastError();
  }
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int mode = 0; mode < 2; ++mode) {
    // mode 0: cluster split-K kernel (split_k = 0 -> skinny), mode 1: tiled kernel (split_k = 1 disables skinny)
    auto run = [&]() {
      for (int s = 0; s < STEPS; ++s) {
        TcArgs e; e.C = C; e.ldc = N; e.beta = 1.f; e.act = ACT_RELU; e.split_k = mode == 0 ? 0 : 1;
        e.Cb = Cb + (size_t)((s + 1) & 1) * 128 * N; e.ldcb = N;
        int rc = gemm_tc_bf16(Cb + (size_t)(s & 1) * 128 * N, N, 0, W, K, 0, M, N, K, e, ws, 64 << 20, st);
        if (rc) { printf("gemm failed at step %d: %s\n", s, tacorl_last_error()); exit(1); }
        if (getenv("STEP_SYNC")) {
          cudaError_t er = cudaStreamSynchronize(st);
          if (er != cudaSuccess) { printf("kernel of step %d failed: %s\n", s, cudaGetErrorString(er)); exit(1); }
        }
      }
    };
    run(); cudaStreamSynchronize(st);
    cudaGraph_t g; cudaGraphExec_t ge;
    cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
    run();
    cudaStreamEndCapture(st, &g);
    cudaGraphInstantiate(&ge, g, 0);
    for (int i = 0; i < 3; ++i) cudaGraphLaunch(ge, st);
    cudaEventRecord(e0, st);
    for (int i = 0; i < 10; ++i) cudaGraphLaunch(ge, st);
    cudaEventRecord(e1, st);
    cudaStreamSynchronize(st);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("mode %d (M=%d): %.2f us per dependent step (graph of %d steps)\n", mode, M, ms * 1000 / (10 * STEPS), STEPS);
    if (cudaGetLastError() != cudaSuccess) printf("CUDA error\n");
#ifdef TACORL_STEP_PROFILE
    if (mode == 0) {
      unsigned long long h[16];
      cudaMemcpyFromSymbol(h, g_step_prof, sizeof(h));
      const char* names[] = {"start", "setup done", "tma issued", "first stage landed", "all mma issued", "mma done",
                             "S stored", "cluster sync 1", "dsmem loaded", "stores issued", "cluster sync 2", "end"};
      for (int i = 1; i < 12; ++i) printf("  %-20s +%6llu ns (t=%llu)\n", names[i], h[i] - h[i - 1], h[i] - h[0]);
      printf("  (prefetch issued at t=%llu)\n", h[12] - h[0]);
      static unsigned long long c[2][256][2];
      cudaMemcpyFromSymbol(c, g_cta_prof, sizeof(c));
      unsigned long long s0 = ~0ull, s1 = 0, e0 = 0, e1 = ~0ull, ps0 = ~0ull, pe0 = 0;
      for (int i = 0; i < 120; ++i) {
        s0 = std::min(s0, c[1][i][0]); s1 = std::max(s1, c[1][i][0]);
        e0 = std::max(e0, c[1][i][1]); e1 = std::min(e1, c[1][i][1]);
        ps0 = std::min(ps0, c[0][i][0]); pe0 = std::max(pe0, c[0][i][1]);
      }
      printf("  last launch: first CTA start -> last CTA start %llu ns, first CTA end at %llu, last CTA end at %llu ns\n",
             s1 - s0, e1 - s0, e0 - s0);
      for (int cl = 0; cl < 15; ++cl) {
        unsigned long long a = ~0ull, b = 0;
        for (int r = 0; r < 8; ++r) { a = std::min(a, c[1][cl * 8 + r][0]); b = std::max(b, c[1][cl * 8 + r][1]); }
        printf("    cluster %2d: start +%llu end +%llu\n", cl, a - s0, b - s0);
      }
      printf("  previous launch: span %llu ns; gap previous last-end -> this first-start %lld ns; period %llu ns\n",
             pe0 - ps0, (long long)(s0 - pe0), s0 - ps0);
    }
#endif
  }
  {  // persistent recurrence: STEPS dependent steps in one launch
    const int T = STEPS + 1;
    __nv_bfloat16* hb; float* Cs; unsigned* flags;
    cudaMalloc(&hb, (size_t)T * M * N * 2); cudaMalloc(&Cs, (size_t)T * M * N * 4); cudaMalloc(&flags, 256);
    cudaMemset(hb, 0, (size_t)T * M * N * 2); cudaMemset(Cs, 0, (size_t)T * M * N * 4);
    auto run = [&]() {
      int rc = rnn_seq_tc(hb, T, W, K, M, N, K, 1, 1, STEPS, 1.f, Cs, N, (long long)M * N, nullptr, 0, 0, hb, ACT_RELU, flags, st);
      if (rc) { printf("rnn_seq_tc rc=%d %s\n", rc, tacorl_last_error()); exit(1); }
    };
    run(); cudaStreamSynchronize(st);
    for (int i = 0; i < 3; ++i) run();
    cudaEventRecord(e0, st);
    for (int i = 0; i < 10; ++i) run();
    cudaEventRecord(e1, st);
    cudaStreamSynchronize(st);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("persistent (M=%d): %.2f us per dependent step (%d steps per launch), timeouts %u\n", M, ms * 1000 / (10 * STEPS), STEPS,
           rnn_seq_timeouts());
#ifdef TACORL_STEP_PROFILE
    long long h[16];
    cudaMemcpyFromSymbol(h, g_seq_prof, sizeof(h));
    const char* nm[] = {"issuer: step start", "flags ok", "tma issued", "first A stage landed", "mma issued+commit",
                        "epi: mma done", "S stored", "cluster sync A", "dsmem summed + arrive B", "bf16 stored + fence",
                        "bar + flag released"};
    for (int i = 0; i < 11; ++i) printf("  %-26s t=%6lld cyc (+%lld)\n", nm[i], h[i] - h[0], i ? h[i] - h[i - 1] : 0);
#endif
  }
  for (int n_lanes = 1; n_lanes <= 2; ++n_lanes) {  // two-lane persistent recurrence at batch 64: STEPS steps per lane
    const int MW = 64, T = STEPS + 1;
    __nv_bfloat16* hb[2]; float* Cs[2]; unsigned* flags[2];
    WaveLaneHost lanes[2];
    for (int l = 0; l < n_lanes; ++l) {
      cudaMalloc(&hb[l], (size_t)T * MW * N * 2); cudaMalloc(&Cs[l], (size_t)T * MW * N * 4); cudaMalloc(&flags[l], 256);
      cudaMemset(hb[l], 0, (size_t)T * MW * N * 2); cudaMemset(Cs[l], 0, (size_t)T * MW * N * 4);
      WaveLaneHost& h = lanes[l];
      h.Ab = hb[l]; h.lda = K; h.a_ts = (long long)MW * K; h.W = W; h.ldw = K;
      h.tau0 = l ? T - 2 : 1; h.dtau = l ? -1 : 1; h.n_steps = STEPS; h.beta = 1.f;
      h.C = Cs[l]; h.ldc = N; h.c_ts = (long long)MW * N; h.Cb = hb[l]; h.ldcb = N; h.cb_ts = (long long)MW * N;
      h.act = ACT_RELU; h.flags = flags[l];
    }
    auto run = [&]() {
      int rc = rnn_wave_tc(lanes, n_lanes, T, MW, N, K, st);
      if (rc) { printf("rnn_wave_tc rc=%d %s\n", rc, tacorl_last_error()); exit(1); }
    };
    run(); cudaStreamSynchronize(st);
    for (int i = 0; i < 3; ++i) run();
    cudaEventRecord(e0, st);
    for (int i = 0; i < 10; ++i) run();
    cudaEventRecord(e1, st);
    cudaStreamSynchronize(st);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("wave %d-lane (M=%d): %.2f us per dependent step (%d steps per launch), timeouts %u, %s\n", n_lanes, MW,
           ms * 1000 / (10 * STEPS), STEPS, rnn_seq_timeouts(), cudaGetErrorString(cudaGetLastError()));
#ifdef TACORL_STEP_PROFILE
    long long h[48];
    cudaMemcpyFromSymbol(h, g_wave_prof, sizeof(h));
    const char* nm[12] = {"issuer: step start", "flags ok", "all TMA issued", "epi: previous S free",
                          "mma issued+commit", "epi: mma done", "S stored", "cluster sync", "dsmem summed + arrive",
                          "bf16 stored + fence", "flag released", "fp32 stored"};
    printf("  stage stamps of CTA (1, 3) at step 32, cycles after the issuer's step start:\n");
    for (int i = 0; i < 48; ++i) {
      if (i > 0 && h[i] == 0) continue;
      char buf[64];
      if (i < 12) snprintf(buf, sizeof(buf), "%s", nm[i]);
      else if (i >= 16 && i < 24) snprintf(buf, sizeof(buf), "K block %d landed", i - 16);
      else if (i >= 24 && i < 32) snprintf(buf, sizeof(buf), "K block %d counters seen", i - 24);
      else if (i >= 32 && i < 40) snprintf(buf, sizeof(buf), "K block %d TMA issued", i - 32);
      else snprintf(buf, sizeof(buf), "stamp %d", i);
      printf("  %-26s t=%6lld cyc\n", buf, h[i] - h[0]);
    }
    const long long zero[48] = {};
    cudaMemcpyToSymbol(g_wave_prof, zero, sizeof(zero));
#endif
    for (int l = 0; l < n_lanes; ++l) { cudaFree(hb[l]); cudaFree(Cs[l]); cudaFree(flags[l]); }
  }
  return 0;
}
