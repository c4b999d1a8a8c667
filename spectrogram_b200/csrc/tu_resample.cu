// Translation unit: PCM ingestion with rational polyphase resampling (kernel_resample.cuh).
#include "kernel_resample.cuh"
#include "plans.cuh"
#include <algorithm>

namespace sg {

namespace {
template <int FMT, bool REG, bool SMEM>
int launch_one(const RsGeom& g, unsigned blocks, const PcmMix& m, size_t smem, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(pcm_resample_kernel<FMT, REG, SMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  pcm_resample_kernel<FMT, REG, SMEM><<<blocks, kRsThreads, smem, st>>>(g, m);
  return (int)cudaGetLastError();
}

template <bool REG, bool SMEM>
int launch_fmt(int format, const RsGeom& g, unsigned blocks, const PcmMix& m, size_t smem, cudaStream_t st) {
  switch (format) {
    case kPcmU8: return launch_one<kPcmU8, REG, SMEM>(g, blocks, m, smem, st);
    case kPcmS16: return launch_one<kPcmS16, REG, SMEM>(g, blocks, m, smem, st);
    case kPcmS24: return launch_one<kPcmS24, REG, SMEM>(g, blocks, m, smem, st);
    case kPcmS32: return launch_one<kPcmS32, REG, SMEM>(g, blocks, m, smem, st);
    case kPcmF32: return launch_one<kPcmF32, REG, SMEM>(g, blocks, m, smem, st);
    default: return (int)cudaErrorInvalidValue;
  }
}

bool taps_in_registers(int J) { return J <= kRsRegTaps; }
bool taps_in_smem(int up, int J) { return (long long)up * J * 4 <= kRsSmemTapBytes; }

int resample_tile_out(int up, int down, int J) {
  // the largest tile whose span, floor((r0 + (nt-1)*down)/up) + J with r0 < up, fits kRsSpan frames
  const long long fit = (long long)(kRsSpan - J - 1) * up / down + 1;
  if (taps_in_registers(J) && fit >= up)                          // whole rounds of phases
    return (int)(up * std::max<long long>(1, std::min<long long>(fit, std::max(up, 8192)) / up));
  return (int)std::min<long long>(fit, 8192);
}
}  // namespace

int launch_pcm_resample(int format, RsGeom g, long long n_clips, const PcmMix& m, cudaStream_t st) {
  if (n_clips <= 0 || g.n_out <= 0) return 0;
  g.tile_out = resample_tile_out(g.up, g.down, g.J);
  g.tiles = (g.n_out + g.tile_out - 1) / g.tile_out;
  const long long blocks = n_clips * g.planes * g.tiles;
  if (blocks > 0x7fffffffLL) return (int)cudaErrorInvalidConfiguration;
  const unsigned b = (unsigned)blocks;
  const size_t with_taps = kRsSmemFixed + (size_t)g.up * g.J * 4;
  if (taps_in_registers(g.J))
    return taps_in_smem(g.up, g.J) ? launch_fmt<true, true>(format, g, b, m, with_taps, st)
                                   : launch_fmt<true, false>(format, g, b, m, kRsSmemFixed, st);
  return taps_in_smem(g.up, g.J) ? launch_fmt<false, true>(format, g, b, m, with_taps, st)
                                 : launch_fmt<false, false>(format, g, b, m, kRsSmemFixed, st);
}

}  // namespace sg
