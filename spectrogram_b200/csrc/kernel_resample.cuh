// Rational polyphase resampling fused into PCM ingestion: interleaved integer/float samples at the file's rate ->
// float32 planes at the context's rate, the sample-rate conversion decodeAudioData applies before the AnalyserNode
// sees the audio ([SPEC] BaseAudioContext.decodeAudioData: "resampled to the sample-rate of the BaseAudioContext").
//
// y[k] = sum_n x[n] h[k*down + half - n*up] over the n with 0 <= k*down + half - n*up <= 2*half (scipy's
// resample_poly with its default Kaiser(5) filter).  With t = k*down + half, n_max = floor(t/up) and r = t mod up,
// the terms are h[r + j*up] x[n_max - j] for j = 0 .. jr-1, jr = floor((2*half - r)/up) + 1: the filter is stored
// phase-major, `up` rows of J = ceil((2*half+1)/up) taps (zero past 2*half).  Every output sums its jr terms in
// ascending j with float32 FMAs, whichever path computes it and however the work is tiled.
//
// One CTA owns a tile of outputs of one plane of one clip.  It stages the input span the tile needs (PCM bytes
// through pcm_stage, converted and mixed by pcm_pick / pcm_mono exactly as the ingest kernel does) into a float32
// span in shared memory, then computes its outputs from that span.  Two choices, both fixed by the ratio:
//   REG   a thread keeps one phase's taps in registers (J <= kRsRegTaps; every upsampling ratio has J = 21) and
//         computes the outputs k, k+up, ... of that phase, so the only shared-memory load per FMA is the sample;
//         otherwise one thread per output reads tap and sample for every FMA
//   SMEM  the whole table (up*J*4 <= kRsSmemTapBytes) is copied into shared memory; larger tables are read
//         through L1/L2.  (The REG path needs this too: lanes hold different phases, so a warp's load of tap j
//         from the global table touches up to 32 cache lines; rows of odd J are bank-conflict free.)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernel_pcm.cuh"

namespace sg {

constexpr int kRsThreads = 256;
constexpr int kRsStageBytes = 16384;         // PCM bytes staged per pass (a span larger than this is staged in passes)
constexpr int kRsSpan = 8192;                // input frames a tile may need (float32 span in shared memory)
constexpr int kRsRegTaps = 24;               // REG holds up to this many taps per phase in registers
constexpr int kRsOutPerItem = 8;             // REG: outputs of one phase per work item
constexpr int kRsSmemTapBytes = 48 * 1024;   // SMEM up to this table size
constexpr int kRsSmemFixed = (kRsStageBytes / 16 + 2) * 16 + kRsSpan * 4;

struct RsGeom {
  const unsigned char* src;    // first uploaded sample frame of clip 0
  long long src_bytes;         // bytes readable from src
  long long clip_bytes;        // bytes between clip starts in src
  long long in_f0;             // index, within the clip, of the first frame at src
  long long in_n;              // frames present per clip; frames outside [in_f0, in_f0 + in_n) read as 0
  long long k0;                // index, within the clip, of the first output computed
  long long n_out;             // outputs per plane
  float* out;                  // output k of plane p of clip c at out + (c*planes + p)*out_stride + (k - k0)
  long long out_stride;
  const float* taps;           // [up][J], phase-major
  long long tiles;             // tiles per plane
  int tile_out;                // outputs per tile
  int up, down, half, J;
  int channels;
  int planes;                  // 1 = mono mix, channels = planar
};

template <int FMT, bool REG, bool SMEM>
__global__ void __launch_bounds__(kRsThreads)
pcm_resample_kernel(const __grid_constant__ RsGeom g, const __grid_constant__ PcmMix m) {
  constexpr int SB = PcmFmt<FMT>::kBytes;
  extern __shared__ uint4 s_dyn[];
  uint4* s_q = s_dyn;
  float* xs = reinterpret_cast<float*>(s_dyn + kRsStageBytes / 16 + 2);
  float* s_taps = xs + kRsSpan;
  const long long row = blockIdx.x / g.tiles;                     // clip * planes + plane
  const long long tile = blockIdx.x - row * g.tiles;
  const long long clip = row / g.planes;
  const int plane = (int)(row - clip * g.planes);
  const long long k_t = g.k0 + tile * g.tile_out;                 // first output of the tile
  const int nt = (int)min((long long)g.tile_out, g.k0 + g.n_out - k_t);
  const long long t0 = k_t * g.down + g.half;
  const long long q0 = t0 / g.up;
  const int r0 = (int)(t0 - q0 * g.up);                           // output o of the tile: t = q0*up + r0 + o*down
  const long long n_first = q0 - (g.J - 1);                       // input frame held in xs[0]
  const int span = (int)((r0 + (long long)(nt - 1) * g.down) / g.up) + g.J;
  const long long v_lo = max(n_first, g.in_f0), v_hi = min(n_first + span, g.in_f0 + g.in_n);
  for (int i = threadIdx.x; i < span; i += kRsThreads)
    if (n_first + i < v_lo || n_first + i >= v_hi) xs[i] = 0.f;   // outside the clip (or the uploaded range)
  if constexpr (SMEM)
    for (int i = threadIdx.x; i < g.up * g.J; i += kRsThreads) s_taps[i] = __ldg(g.taps + i);
  // ---- the span, converted: staged in passes of whole sample frames
  const int bpf = g.channels * SB;
  const int pass = kRsStageBytes / bpf;
  const uint32_t* __restrict__ sw = reinterpret_cast<const uint32_t*>(s_q);
  for (long long f = v_lo; f < v_hi; f += pass) {
    const int nf = (int)min((long long)pass, v_hi - f);
    __syncthreads();                                              // the previous pass has been read
    const int skew = pcm_stage<kRsThreads>(s_q, g.src, g.src_bytes, clip * g.clip_bytes + (f - g.in_f0) * bpf, nf * bpf);
    __syncthreads();
    float* dst = xs + (f - n_first);
    if (g.planes == 1) {
      for (int i = threadIdx.x; i < nf; i += kRsThreads) dst[i] = pcm_mono<FMT>(sw, skew + i * bpf, g.channels, m);
    } else {
      for (int i = threadIdx.x; i < nf; i += kRsThreads) dst[i] = pcm_pick<FMT>(sw, skew + i * bpf + plane * SB);
    }
  }
  __syncthreads();
  // ---- outputs
  float* __restrict__ out = g.out + row * g.out_stride + (k_t - g.k0);
  const int two_half = 2 * g.half;
  const float* __restrict__ tp = SMEM ? s_taps : g.taps;
  auto tap_at = [&](int i) { return SMEM ? tp[i] : __ldg(tp + i); };
  if constexpr (REG) {
    const int P = min(g.up, nt);                                  // phases present in the tile
    const int per_phase = (nt + g.up - 1) / g.up;
    const int items = P * ((per_phase + kRsOutPerItem - 1) / kRsOutPerItem);
    for (int it = threadIdx.x; it < items; it += kRsThreads) {
      const int p = it % P, m0 = (it / P) * kRsOutPerItem;
      const int r = (r0 + p * g.down) % g.up;                     // the phase of outputs p, p + up, p + 2 up, ...
      const int jr = (two_half - r) / g.up + 1;
      float tap[kRsRegTaps];
#pragma unroll
      for (int j = 0; j < kRsRegTaps; ++j) tap[j] = j < jr ? tap_at(r * g.J + j) : 0.f;
      const float* x0 = xs + (r0 + p * g.down) / g.up + g.J - 1 + m0 * g.down;   // x[n_max] of output p + m0 up
#pragma unroll
      for (int mm = 0; mm < kRsOutPerItem; ++mm) {
        const int o = p + (m0 + mm) * g.up;
        if (o < nt) {
          const float* xr = x0 + mm * g.down;                           // n_max grows by down per round of phases
          float acc = 0.f;
#pragma unroll
          for (int j = 0; j < kRsRegTaps; ++j)
            if (j < jr) acc = fmaf(tap[j], xr[-j], acc);
          out[o] = acc;
        }
      }
    }
  } else {
    for (int o = threadIdx.x; o < nt; o += kRsThreads) {
      const int t = r0 + o * g.down;
      const int qn = t / g.up, r = t - qn * g.up;
      const int jr = (two_half - r) / g.up + 1;
      const float* hr = tp + r * g.J;
      const float* xr = xs + qn + g.J - 1;
      float acc = 0.f;
      for (int j = 0; j < jr; ++j) acc = fmaf(SMEM ? hr[j] : __ldg(hr + j), xr[-j], acc);
      out[o] = acc;
    }
  }
}

}  // namespace sg
