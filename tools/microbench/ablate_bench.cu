// Marginal cost of each component of the headline kernel under real contention: times stft_w32x2p_kernel<u8, 12, 8, ABL>
// with one component removed at a time (kernel_w32x2p.cuh lists the ABL bits).  Outputs are wrong by construction.
// Build: nvcc -O3 -std=c++17 --expt-relaxed-constexpr -gencode arch=compute_100a,code=sm_100a \
//        -I../../spectrogram_b200/csrc -o ablate_bench ablate_bench.cu
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "kernel_w32x2p.cuh"

using namespace sg;

struct Ctx { FrameGeom g; W32Plan pl; Epilogue ep; uint8_t* out; long long frames; };

template <int ABL>
void run(const Ctx& c, const char* what) {
  constexpr int NW = 12, smem = XpShape<NW>::kSmemBytes;
  cudaFuncSetAttribute(stft_w32x2p_kernel<kOutU8, NW, 8, ABL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e9f;
  for (int rep = 0; rep < 6; ++rep) {
    cudaEventRecord(e0);
    stft_w32x2p_kernel<kOutU8, NW, 8, ABL><<<148, NW * 32, smem>>>(c.g, c.pl, c.ep, c.out);
    cudaEventRecord(e1);
    if (cudaDeviceSynchronize() != cudaSuccess) { printf("ABL %d failed: %s\n", ABL, cudaGetErrorString(cudaGetLastError())); return; }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    if (rep >= 2 && ms < best) best = ms;
  }
  printf("ABL %3d  %-44s %.4f ms  %.1f M frames/s\n", ABL, what, best, c.frames / best * 1e-3);
}

int main() {
  const int n_clips = 512;
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
  Ctx c{FrameGeom{pcm, clip_len, clip_len, fpc, (long long)n_clips * fpc, 0, 2048, 512}, W32Plan{d_win, d_tw2, d_ut},
        Epilogue{3.0103f, -72.f, 10.97f, 100.f, 364.f, 1.f / 4096, nullptr}, out, (long long)n_clips * fpc};
  run<0>(c, "full kernel");
  run<128>(c, "full kernel, lane-0 selects as PRMT");
  run<256>(c, "full kernel, mirrors through shared memory");
  run<0>(c, "full kernel (again)");
  run<1>(c, "- exchange (STS/bar/LDS)");
  run<2>(c, "- mirror shuffles");
  run<64>(c, "- lane-0 selects");
  run<2 | 64>(c, "- shuffles and selects");
  run<4>(c, "- MUFU.LG2 / F2IP");
  run<16>(c, "- byte stage + row stores");
  run<4 | 16>(c, "- MUFU/F2IP, byte stage, stores");
  run<8>(c, "- next-pair loads");
  run<32>(c, "- window table reads");
  run<1 | 2 | 64>(c, "- exchange, shuffles, selects");
  run<1 | 2 | 4 | 8 | 16 | 32 | 64>(c, "FMA work only");
  return 0;
}
