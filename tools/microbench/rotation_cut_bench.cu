// Where the rotation's three group barriers should sit: times stft_w32x2p_kernel at every cut placement xp_cut(ab, bc, ca)
// (kernel_w32x2p.cuh) on each shape the product runs it at, alternating the placements round by round in one process, and
// checks that every placement writes the same rows (moving a barrier changes no arithmetic).
// 512 x 10 s clips: the 903 MB of input do not fit the 126 MB L2.  Table values do not influence timing (no data-dependent
// branch), so the plan is filled with finite placeholders.
// Build: nvcc -O3 -std=c++17 --expt-relaxed-constexpr -gencode arch=compute_100a,code=sm_100a \
//        -I../../spectrogram_b200/csrc -o rotation_cut_bench rotation_cut_bench.cu
// usage: rotation_cut_bench [rounds]
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <vector>

#include "kernel_w32x2p.cuh"

using namespace sg;

struct Ctx { const float* pcm; long long clip_len; int n_clips; W32Plan pl; Epilogue ep; };

__global__ void count_mismatches(const uint32_t* a, const uint32_t* b, size_t n, unsigned long long* bad) {
  unsigned long long m = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) m += a[i] != b[i];
  if (m) atomicAdd(bad, m);
}

struct Variant { int cut; void (*launch)(const FrameGeom&, const Ctx&, void*); std::vector<float> ms; };

template <int OUT, int NW, int HOPJ, int CUT>
void launch(const FrameGeom& g, const Ctx& c, void* out) {
  constexpr int smem = XpShape<NW>::kSmemBytes;
  stft_w32x2p_kernel<OUT, NW, HOPJ, 0, CUT><<<148, NW * 32, smem>>>(g, c.pl, c.ep, (typename OutElem<OUT>::type*)out);
}

// round 3's placement first: every other placement is compared against its rows and times.  The first nine keep C | A at
// the end of the pair, the only choice for float rows.
constexpr int kCuts[] = {xp_cut(0, 2, 1), xp_cut(0, 1, 1), xp_cut(0, 0, 1), xp_cut(1, 2, 1), xp_cut(1, 1, 1),
                         xp_cut(1, 0, 1), xp_cut(2, 2, 1), xp_cut(2, 1, 1), xp_cut(2, 0, 1), xp_cut(0, 2, 0),
                         xp_cut(0, 1, 0), xp_cut(0, 0, 0), xp_cut(1, 2, 0), xp_cut(1, 1, 0), xp_cut(1, 0, 0),
                         xp_cut(2, 2, 0), xp_cut(2, 1, 0), xp_cut(2, 0, 0)};

template <int OUT, int NW, int HOPJ, size_t... I>
std::vector<Variant> variants(std::index_sequence<I...>) {
  constexpr int smem = XpShape<NW>::kSmemBytes;
  (cudaFuncSetAttribute(stft_w32x2p_kernel<OUT, NW, HOPJ, 0, kCuts[I]>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), ...);
  return {Variant{kCuts[I], &launch<OUT, NW, HOPJ, kCuts[I]>, {}}...};
}

template <int OUT, int NW, int HOPJ>
void sweep(const char* name, const Ctx& c, int rounds) {
  std::vector<Variant> v;
  if constexpr (OUT == kOutU8) v = variants<OUT, NW, HOPJ>(std::make_index_sequence<18>());
  else v = variants<OUT, NW, HOPJ>(std::make_index_sequence<9>());
  const int hop = 64 * HOPJ;
  const long long fpc = 1 + (c.clip_len - 2048) / hop, frames = (long long)c.n_clips * fpc;
  const FrameGeom g{c.pcm, c.clip_len, c.clip_len, fpc, frames, 0, 2048, hop};
  const size_t bytes = (size_t)frames * 1024 * sizeof(typename OutElem<OUT>::type);
  void *ref, *out;
  cudaMalloc(&ref, bytes); cudaMalloc(&out, bytes);
  unsigned long long* bad; cudaMalloc(&bad, 8);
  // warm-up, and the rows of every placement against the first
  std::vector<unsigned long long> mism(v.size());
  for (size_t i = 0; i < v.size(); ++i) {
    cudaMemset(out, 0xff, bytes);
    v[i].launch(g, c, i == 0 ? ref : out);
    v[i].launch(g, c, i == 0 ? ref : out);
    if (i) {
      cudaMemset(bad, 0, 8);
      count_mismatches<<<1184, 256>>>((const uint32_t*)ref, (const uint32_t*)out, bytes / 4, bad);
      cudaMemcpy(&mism[i], bad, 8, cudaMemcpyDeviceToHost);
    }
  }
  if (cudaDeviceSynchronize() != cudaSuccess) { printf("%s failed: %s\n", name, cudaGetErrorString(cudaGetLastError())); exit(1); }
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  constexpr int kLaunches = 10;
  for (int r = 0; r < rounds; ++r)
    for (size_t j = 0; j < v.size(); ++j) {   // the order rotates every round
      Variant& x = v[(j + r) % v.size()];
      cudaEventRecord(e0);
      for (int l = 0; l < kLaunches; ++l) x.launch(g, c, out);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      x.ms.push_back(ms / kLaunches);
    }
  printf("# %s: %lld frames, %d rounds x %d launches per placement, M frames/s (median of rounds; min..max)\n", name,
         frames, rounds, kLaunches);
  double base = 0;
  for (size_t i = 0; i < v.size(); ++i) {
    std::vector<float> s = v[i].ms;
    std::sort(s.begin(), s.end());
    const double med = frames / s[s.size() / 2] * 1e-3;
    if (i == 0) base = med;
    printf("%-14s ab %d bc %d ca %d  %7.1f  (%6.1f .. %6.1f)  %+6.2f %%  rows differing from the first: %llu words\n", name,
           v[i].cut / 100, v[i].cut / 10 % 10, v[i].cut % 10, med, frames / s.back() * 1e-3, frames / s.front() * 1e-3,
           100. * (med / base - 1), mism[i]);
  }
  fflush(stdout);
  cudaFree(ref); cudaFree(out); cudaFree(bad);
}

int main(int argc, char** argv) {
  const int rounds = argc > 1 ? atoi(argv[1]) : 9;
  const int n_clips = 512;
  const long long clip_len = 441000;
  cudaDeviceProp prop; cudaGetDeviceProperties(&prop, 0);
  printf("# %s, %d SMs\n", prop.name, prop.multiProcessorCount);
  float* pcm; cudaMalloc(&pcm, (size_t)n_clips * clip_len * 4);
  std::vector<float> h(clip_len);
  for (long long i = 0; i < clip_len; ++i) h[i] = 0.5f * sinf(0.001f * i * (1.f + 1e-5f * i));
  for (int c = 0; c < n_clips; ++c) cudaMemcpy(pcm + (size_t)c * clip_len, h.data(), clip_len * 4, cudaMemcpyHostToDevice);
  std::vector<float> win(4096, 0.5f);
  std::vector<float2> tw2(31 * 32, make_float2(0.8f, -0.6f)), ut(16 * 32, make_float2(0.6f, -0.8f));
  float* d_win; float2 *d_tw2, *d_ut;
  cudaMalloc(&d_win, win.size() * 4); cudaMalloc(&d_tw2, tw2.size() * 8); cudaMalloc(&d_ut, ut.size() * 8);
  cudaMemcpy(d_win, win.data(), win.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(d_tw2, tw2.data(), tw2.size() * 8, cudaMemcpyHostToDevice);
  cudaMemcpy(d_ut, ut.data(), ut.size() * 8, cudaMemcpyHostToDevice);
  const Ctx c{pcm, clip_len, n_clips, W32Plan{d_win, d_tw2, d_ut}, Epilogue{3.0103f, -72.f, 10.97f, 100.f, 364.f, 1.f / 4096, nullptr}};
  sweep<kOutU8, 12, 8>("u8 hop512", c, rounds);   // the headline
  sweep<kOutU8, 12, 4>("u8 hop256", c, rounds);
  sweep<kOutF32Db, 12, 8>("dB hop512", c, rounds);
  sweep<kOutF32Db, 12, 4>("dB hop256", c, rounds);
  sweep<kOutF32Mag, 12, 8>("mag hop512", c, rounds);
  sweep<kOutU8, 8, 8>("u8 hop512 8w", c, rounds);
  sweep<kOutF32Db, 8, 8>("dB hop512 8w", c, rounds);
  return 0;
}
