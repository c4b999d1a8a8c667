// Phase timeline of the headline kernel: builds stft_w32x2p_kernel with SG_XP_TRACE and prints, for the 12 warps of
// CTA 0, when each phase of each pair starts (clock64, relative to the CTA's first record).  Answers: do the warps of a
// scheduler sit in the same phase at the same time (convoy), and how long does each phase take under contention?
// Table values do not influence timing (no data-dependent branch), so the plan is filled with finite placeholders.
// Build: nvcc -O3 -std=c++17 --expt-relaxed-constexpr -DSG_XP_TRACE -gencode arch=compute_100a,code=sm_100a \
//        -I../../spectrogram_b200/csrc -o trace_bench trace_bench.cu
// usage: trace_bench [n_clips]
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "kernel_w32x2p.cuh"

using namespace sg;

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
  cudaFuncSetAttribute(stft_w32x2p_kernel<OUT, NW, HOPJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 3; ++rep) {
    cudaEventRecord(e0);
    stft_w32x2p_kernel<OUT, NW, HOPJ><<<148, NW * 32, smem>>>(g, pl, ep, out);
    cudaEventRecord(e1);
    if (cudaDeviceSynchronize() != cudaSuccess) { printf("kernel failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 1; }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("# %.4f ms, %.1f M frames/s (traced build)\n", ms, n_clips * fpc / ms * 1e-3);
  }
  std::vector<long long> t(tn);
  cudaMemcpy(t.data(), trace, tn * 8, cudaMemcpyDeviceToHost);
  long long t0 = -1;
  for (auto v : t) if (v && (t0 < 0 || v < t0)) t0 = v;
  // phase p = [point p, point p+1): 0 window+pass1, 1 exchange stores + the A|B step barrier, 2 exchange loads, 3 pass 2,
  // 4 mirror shuffles + the B|C step barrier + untangle (+ next pair's loads), 5 epilogue; the C|A barrier falls between
  // a pair's point 6 and the next pair's point 0 (kernel_w32x2p.cuh, rotation)
  printf("# warp iter start  window+p1 xstore xload pass2 untangle epilogue  total\n");
  for (int w = 0; w < NW; ++w)
    for (int it = 0; it < kXpTraceIters; ++it) {
      const long long* r = &t[((size_t)w * kXpTraceIters + it) * kXpTracePoints];
      if (!r[0] || !r[6]) continue;
      printf("%2d %2d %8lld  %6lld %6lld %6lld %6lld %6lld %6lld  %6lld\n", w, it, r[0] - t0, r[1] - r[0], r[2] - r[1],
             r[3] - r[2], r[4] - r[3], r[5] - r[4], r[6] - r[5], r[6] - r[0]);
    }
  return 0;
}
