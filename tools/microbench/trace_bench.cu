// Section timeline of the headline kernel: builds stft_w32x2p_kernel with SG_XP_TRACE and prints, for the 12 warps of
// CTA 0 and each of their first pairs, how long each section of the rotation ran (busy: from leaving one group barrier to
// arriving at the next) and how long the warp then waited at the barrier for the rest of its group (clock64 of lane 0).
// The summary gives the mean per section and rank, and the share of a step lost to waits: what moving a cut can win.
// Table values do not influence timing (no data-dependent branch), so the plan is filled with finite placeholders.
// Build: nvcc -O3 -std=c++17 --expt-relaxed-constexpr -DSG_XP_TRACE -gencode arch=compute_100a,code=sm_100a \
//        -I../../spectrogram_b200/csrc -o trace_bench trace_bench.cu
//        (-DTRACE_CUT=<100 ab + 10 bc + ca, the value of xp_cut(ab, bc, ca)> traces another cut placement than the product's)
// usage: trace_bench [n_clips]
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "kernel_w32x2p.cuh"

using namespace sg;

#ifndef TRACE_CUT
#define TRACE_CUT (xp_cuts<kOutU8, 12, 8>())
#endif

int main(int argc, char** argv) {
  const int n_clips = argc > 1 ? atoi(argv[1]) : 256;
  constexpr int NW = 12, OUT = kOutU8, HOPJ = 8;
  const long long clip_len = 441000, fpc = 1 + (clip_len - 2048) / 512;
  float* pcm; cudaMalloc(&pcm, (size_t)n_clips * clip_len * 4);
  std::vector<float> h(clip_len);
  for (long long i = 0; i < clip_len; ++i) h[i] = 0.5f * sinf(0.001f * i * (1.f + 1e-5f * i));
  for (int c = 0; c < n_clips; ++c) cudaMemcpy(pcm + (size_t)c * clip_len, h.data(), clip_len * 4, cudaMemcpyHostToDevice);
  uint8_t* out; cudaMalloc(&out, (size_t)n_clips * fpc * 1024);
  std::vector<float> win(4096, 0.5f);
  std::vector<float2> tw2(31 * 32, make_float2(0.8f, -0.6f)), ut(16 * 32, make_float2(0.6f, -0.8f));
  float* d_win; float2 *d_tw2, *d_ut;
  cudaMalloc(&d_win, win.size() * 4); cudaMalloc(&d_tw2, tw2.size() * 8); cudaMalloc(&d_ut, ut.size() * 8);
  cudaMemcpy(d_win, win.data(), win.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(d_tw2, tw2.data(), tw2.size() * 8, cudaMemcpyHostToDevice);
  cudaMemcpy(d_ut, ut.data(), ut.size() * 8, cudaMemcpyHostToDevice);
  long long* trace; const size_t tn = (size_t)NW * kXpTraceIters * kXpTracePoints;
  cudaMalloc(&trace, tn * 8); cudaMemset(trace, 0, tn * 8);
  cudaMemcpyToSymbol(g_xp_trace, &trace, sizeof(trace));
  FrameGeom g{pcm, clip_len, clip_len, fpc, (long long)n_clips * fpc, 0, 2048, 512};
  W32Plan pl{d_win, d_tw2, d_ut};
  Epilogue ep{3.0103f, -72.f, 10.97f, 100.f, 364.f, 1.f / 4096, nullptr};
  constexpr int smem = XpShape<NW>::kSmemBytes;
  constexpr int CUT = TRACE_CUT;
  auto kernel = stft_w32x2p_kernel<OUT, NW, HOPJ, 0, CUT>;
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 3; ++rep) {
    cudaEventRecord(e0);
    kernel<<<148, NW * 32, smem>>>(g, pl, ep, out);
    cudaEventRecord(e1);
    if (cudaDeviceSynchronize() != cudaSuccess) { printf("kernel failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 1; }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("# %.4f ms, %.1f M frames/s (traced build)\n", ms, n_clips * fpc / ms * 1e-3);
  }
  std::vector<long long> t(tn);
  cudaMemcpy(t.data(), trace, tn * 8, cudaMemcpyDeviceToHost);
  long long t0 = -1;
  for (auto v : t) if (v && (t0 < 0 || v < t0)) t0 = v;
  // points (kernel_w32x2p.cuh): 0 top of the pair, 1 / 2 arrive at / leave A | B, 3 / 4 B | C, 5 / 6 C | A.  Section A
  // starts when the warp leaves the previous pair's C | A barrier (the first pair: at point 0, after the lead-in steps).
  printf("# cut ab %d bc %d ca %d\n", CUT / 100, CUT / 10 % 10, CUT % 10);
  printf("# warp rank iter    start  A_busy AB_wait  B_busy BC_wait  C_busy CA_wait   total\n");
  double busy[3][3] = {}, wait[3][3] = {};   // [rank][section]
  long long n[3] = {};
  for (int w = 0; w < NW; ++w) {
    long long prev = 0;
    for (int it = 0; it < kXpTraceIters; ++it) {
      const long long* r = &t[((size_t)w * kXpTraceIters + it) * kXpTracePoints];
      if (!r[0] || !r[6]) break;
      const long long a0 = it == 0 ? r[0] : prev;
      const long long b[3] = {r[1] - a0, r[3] - r[2], r[5] - r[4]}, q[3] = {r[2] - r[1], r[4] - r[3], r[6] - r[5]};
      printf("%4d %4d %4d %8lld  %6lld  %6lld  %6lld  %6lld  %6lld  %6lld  %6lld\n", w, w / 4, it, a0 - t0, b[0], q[0], b[1],
             q[1], b[2], q[2], r[6] - a0);
      if (it >= 2)   // the first pairs run while the other CTAs ramp up
        for (int k = 0; k < 3; ++k) { busy[w / 4][k] += b[k]; wait[w / 4][k] += q[k]; }
      n[w / 4] += it >= 2;
      prev = r[6];
    }
  }
  printf("# mean cycles per pair from pair 2 on: section busy / wait at the barrier that ends it\n");
  printf("# rank      A busy/wait      B busy/wait      C busy/wait   step  wait share\n");
  double all_b = 0, all_w = 0;
  for (int k = 0; k < 3; ++k) {
    if (!n[k]) continue;
    double sb = 0, sw = 0;
    printf("# %4d", k);
    for (int s = 0; s < 3; ++s) {
      printf("   %6.0f / %5.0f", busy[k][s] / n[k], wait[k][s] / n[k]);
      sb += busy[k][s]; sw += wait[k][s];
    }
    printf("  %5.0f  %9.1f %%\n", (sb + sw) / n[k] / 3, 100. * sw / (sb + sw));
    all_b += sb; all_w += sw;
  }
  printf("# all ranks: waits are %.1f %% of a step\n", 100. * all_w / (all_b + all_w));
  return 0;
}
