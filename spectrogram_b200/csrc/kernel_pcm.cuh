// PCM ingestion (SURVEY 8(f) rank 4): interleaved integer/float samples -> float32 planes, the uncompressed
// part of what context.decodeAudioData does for the reference (util/util.js:9-17), plus the mono down-mix the
// AnalyserNode applies to a multi-channel input ([SPEC] channelInterpretation "speakers").
//
// HBM-bound byte work: one CTA converts a tile of sample frames.  The tile's byte span is staged into shared
// memory with 16-byte coalesced loads from the aligned-down address (sample frames of 3, 6, 18 ... bytes have
// no useful global alignment), every thread then picks its samples out of two adjacent 32-bit shared words with
// a funnel shift, and stores float32 coalesced.  Algorithmic bytes per sample frame: channels*sample_bytes read
// + 4*planes written.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sg {

constexpr int kPcmU8 = 0, kPcmS16 = 1, kPcmS24 = 2, kPcmS32 = 3, kPcmF32 = 4;
constexpr int kPcmThreads = 256;
constexpr int kPcmTileBytes = 32768;       // staged span per CTA (plus up to 15 bytes of alignment slack)
constexpr int kPcmMaxChannels = 32;

struct PcmMix { float w[kPcmMaxChannels]; };   // mono = sum_c w[c] * x[c], accumulated in channel order with FMAs

struct PcmGeom {
  const unsigned char* src;    // first sample of clip 0
  long long src_bytes;         // bytes readable from src (guards the 16-byte staging loads)
  long long clip_bytes;        // bytes between clip starts
  long long frames;            // sample frames per clip
  float* out;                  // plane p of clip c at out + (c*planes + p)*out_stride
  long long out_stride;
  long long tiles_per_clip;
  int tile_frames;
  int channels;
  int planes;                  // 1 = mono mix, channels = planar
};

template <int FMT> struct PcmFmt;
template <> struct PcmFmt<kPcmU8>  { static constexpr int kBytes = 1;
  static __device__ __forceinline__ float cvt(uint32_t v) { return (float)((int)(v & 0xffu) - 128) * (1.f / 128.f); } };
template <> struct PcmFmt<kPcmS16> { static constexpr int kBytes = 2;
  static __device__ __forceinline__ float cvt(uint32_t v) { return (float)(short)(v & 0xffffu) * (1.f / 32768.f); } };
template <> struct PcmFmt<kPcmS24> { static constexpr int kBytes = 3;
  static __device__ __forceinline__ float cvt(uint32_t v) { return (float)(((int)(v << 8)) >> 8) * (1.f / 8388608.f); } };
template <> struct PcmFmt<kPcmS32> { static constexpr int kBytes = 4;
  static __device__ __forceinline__ float cvt(uint32_t v) { return __int2float_rn((int)v) * (1.f / 2147483648.f); } };
template <> struct PcmFmt<kPcmF32> { static constexpr int kBytes = 4;
  static __device__ __forceinline__ float cvt(uint32_t v) { return __uint_as_float(v); } };

// Stages bytes [b0, b0 + n) of src into s_q with 16-byte loads from the aligned-down address (bytes outside
// [0, src_bytes) read as 0) and returns b0's offset inside the first staged word.  The caller synchronises.
template <int THREADS>
__device__ __forceinline__ int pcm_stage(uint4* s_q, const unsigned char* src, long long src_bytes, long long b0, int n) {
  const int skew = (int)(((uintptr_t)src + (uintptr_t)b0) & 15);
  const long long a0 = b0 - skew;                                 // 16-byte aligned (as an address), may be < 0
  const int nq = (skew + n + 15) >> 4;
  for (int i = threadIdx.x; i < nq; i += THREADS) {
    const long long o = a0 + 16LL * i;
    uint4 q;
    if (o >= 0 && o + 16 <= src_bytes) {
      q = __ldg(reinterpret_cast<const uint4*>(src + o));
    } else {                                                      // first/last chunk of the buffer: byte by byte
      uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int b = 0; b < 16; ++b)
        if (o + b >= 0 && o + b < src_bytes) w[b >> 2] |= (uint32_t)src[o + b] << (8 * (b & 3));
      q = make_uint4(w[0], w[1], w[2], w[3]);
    }
    s_q[i] = q;
  }
  return skew;
}

// the sample starting at byte_off of the staged words: two adjacent 32-bit words and a funnel shift
template <int FMT>
__device__ __forceinline__ float pcm_pick(const uint32_t* __restrict__ sw, int byte_off) {
  const int wi = byte_off >> 2;
  return PcmFmt<FMT>::cvt(__funnelshift_r(sw[wi], sw[wi + 1], 8 * (byte_off & 3)));
}

// speakers down-mix of the sample frame at byte_off: w[0] x[0], then one FMA per further channel in channel order
template <int FMT>
__device__ __forceinline__ float pcm_mono(const uint32_t* __restrict__ sw, int byte_off, int channels, const PcmMix& m) {
  float acc = m.w[0] * pcm_pick<FMT>(sw, byte_off);
  for (int c = 1; c < channels; ++c) acc = fmaf(m.w[c], pcm_pick<FMT>(sw, byte_off + c * PcmFmt<FMT>::kBytes), acc);
  return acc;
}

template <int FMT>
__global__ void __launch_bounds__(kPcmThreads)
pcm_ingest_kernel(const __grid_constant__ PcmGeom g, const __grid_constant__ PcmMix m) {
  constexpr int SB = PcmFmt<FMT>::kBytes;
  __shared__ uint4 s_q[kPcmTileBytes / 16 + 2];
  const long long clip = blockIdx.x / g.tiles_per_clip;
  const long long tile = blockIdx.x - clip * g.tiles_per_clip;
  const long long f0 = tile * g.tile_frames;
  const int tf = (int)min((long long)g.tile_frames, g.frames - f0);
  const int bpf = g.channels * SB;
  const long long b0 = clip * g.clip_bytes + f0 * bpf;           // first byte of the tile, relative to src
  const int skew = pcm_stage<kPcmThreads>(s_q, g.src, g.src_bytes, b0, tf * bpf);
  __syncthreads();
  const uint32_t* __restrict__ sw = reinterpret_cast<const uint32_t*>(s_q);
  auto sample = [&](int byte_off) { return pcm_pick<FMT>(sw, byte_off); };
  if (g.planes == 1) {
    float* __restrict__ dst = g.out + clip * g.out_stride + f0;
    for (int f = threadIdx.x; f < tf; f += kPcmThreads) {
      dst[f] = pcm_mono<FMT>(sw, skew + f * bpf, g.channels, m);
    }
  } else {
    float* __restrict__ dst = g.out + clip * g.planes * g.out_stride + f0;
    for (int f = threadIdx.x; f < tf; f += kPcmThreads) {
      const int o = skew + f * bpf;
      for (int c = 0; c < g.channels; ++c) dst[c * g.out_stride + f] = sample(o + c * SB);
    }
  }
}

// ---- 16-bit fast path (the common case): when source rows, destination rows and the frame count are 16-byte
// friendly, every thread converts one 16-byte word (8 samples) straight from global memory: no shared-memory stage.
//   MODE 0: mono -> 1 plane (8 frames per word);  1: stereo -> mono mix 0.5(L+R) (4 frames);  2: stereo -> 2 planes
template <int MODE>
__global__ void __launch_bounds__(256)
pcm_s16_vec_kernel(const uint4* __restrict__ src, long long words_per_clip, long long n_clips, float* __restrict__ out,
                   long long out_stride) {
  constexpr float k = 1.f / 32768.f;
  const long long total = words_per_clip * n_clips;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long clip = i / words_per_clip, w = i - clip * words_per_clip;
    const uint4 q = __ldg(src + i);
    auto lo = [](uint32_t v) { return (float)(short)(v & 0xffffu); };
    auto hi = [](uint32_t v) { return (float)((int)v >> 16); };
    if constexpr (MODE == 0) {
      float4* d = reinterpret_cast<float4*>(out + clip * out_stride) + 2 * w;
      d[0] = make_float4(lo(q.x) * k, hi(q.x) * k, lo(q.y) * k, hi(q.y) * k);
      d[1] = make_float4(lo(q.z) * k, hi(q.z) * k, lo(q.w) * k, hi(q.w) * k);
    } else if constexpr (MODE == 1) {
      auto mix = [&](uint32_t v) { return fmaf(0.5f, hi(v) * k, 0.5f * (lo(v) * k)); };   // as the generic kernel: w0 x0, then FMA
      reinterpret_cast<float4*>(out + clip * out_stride)[w] = make_float4(mix(q.x), mix(q.y), mix(q.z), mix(q.w));
    } else {
      float* base = out + 2 * clip * out_stride;
      reinterpret_cast<float4*>(base)[w] = make_float4(lo(q.x) * k, lo(q.y) * k, lo(q.z) * k, lo(q.w) * k);
      reinterpret_cast<float4*>(base + out_stride)[w] = make_float4(hi(q.x) * k, hi(q.y) * k, hi(q.z) * k, hi(q.w) * k);
    }
  }
}

}  // namespace sg
