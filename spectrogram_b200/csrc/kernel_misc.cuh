// Small kernels around the frame kernels: the smoothing recurrence along frames (AnalyserNode
// step 4, 3D/visualizer.js:351,357,362 set tau per mode), the byte -> colour LUT
// (bin/shaders/sonogram-*.shader) and the byte time-domain getter (3D/visualizer.js:363).
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace sg {

// X^_t[k] = tau*X^_{t-1}[k] + (1-tau)*|X_t[k]|, per (clip, bin), sequential along frames.
// mags: [n_clips][frames][bins] linear magnitudes (already /N).  state: [n_clips][bins], read as
// the initial X^ and written back with the final one (so chunks of one clip can be chained, and
// the streaming objects keep it across calls).  Arithmetic as Chromium: double, stored as float.
// HBM-bound: 4 B read + elem B written per (frame, bin); coalesced across bins.
// [SPEC] "non-finite X^ -> 0": the frame kernels write the magnitudes of a frame with a NaN / Inf sample as 0, which
// the recurrence cannot tell from silence, so `poison` ([n_clips][frames], poison_flags_kernel) names those frames and
// the state restarts from 0 there, as in the fused kernels.  poison == nullptr: no frame is poisoned (the AnalyserNode
// object, whose non-finite magnitudes enter the recurrence as 0).  A magnitude that is itself non-finite (|X|^2
// overflowing float) enters as 0.
template <int OUT>
__global__ void __launch_bounds__(256)
smooth_emit_kernel(const float* __restrict__ mags, typename OutElem<OUT>::type* __restrict__ out,
                   float* __restrict__ state, long long n_clips, long long frames, int bins, double tau,
                   Epilogue ep, const uint8_t* __restrict__ poison) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_clips * bins) return;
  const long long clip = idx / bins;
  const int b = (int)(idx - clip * bins);
  const float* __restrict__ m = mags + clip * frames * bins + b;
  typename OutElem<OUT>::type* __restrict__ o = out + clip * frames * bins + b;
  const uint8_t* __restrict__ pz = poison ? poison + clip * frames : nullptr;
  float s = state[idx];
  const double k1 = 1.0 - tau;
  long long t = 0;
  for (; t + 4 <= frames; t += 4) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = finite_or_zero(__ldg(m + (t + u) * bins));
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      s = finite_or_zero((float)(tau * (double)s + k1 * (double)v[u]));
      if (pz && __ldg(pz + t + u)) s = 0.f;
      o[(t + u) * bins] = emit_mag<OUT>(s, ep);
    }
  }
  for (; t < frames; ++t) {
    s = finite_or_zero((float)(tau * (double)s + k1 * (double)finite_or_zero(__ldg(m + t * bins))));
    if (pz && __ldg(pz + t)) s = 0.f;
    o[t * bins] = emit_mag<OUT>(s, ep);
  }
  state[idx] = s;
}

// poison[clip][t] = 1 when frame t of the clip holds a NaN / Inf sample (samples outside the clip are the zero
// history): what smooth_emit_kernel and smooth_scan_kernel restart the state on.  One warp per frame, coalesced loads
// (a sample is read by n_fft / hop frames; the overlap comes from L2).
__global__ void __launch_bounds__(256) poison_flags_kernel(FrameGeom g, uint8_t* __restrict__ poison) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= g.total_frames) return;     // (whole warps)
  const long long clip = w / g.frames_per_clip, t = w - clip * g.frames_per_clip;
  const float* __restrict__ x = g.pcm + clip * g.clip_stride;
  const long long s0 = g.start0 + t * g.hop;
  const long long lo = s0 > 0 ? s0 : 0, hi = s0 + g.n_fft < g.clip_len ? s0 + g.n_fft : g.clip_len;
  bool bad = false;
  for (long long i = lo + lane; i < hi; i += 32) bad |= !(fabsf(__ldg(x + i)) <= 3.4028235e38f);
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) poison[w] = bad ? 1 : 0;
}

// ---- time-parallel form of the same recurrence for long clips with few (clip, bin) pairs, ONE kernel ---------------
// The recurrence is linear with a constant coefficient, so a clip's frames are cut into chunks of `chunk` frames:
//   (A) each chunk's zero-state response at its last frame (thread per (clip, chunk, bin), bins coalesced),
//   (B) the same recurrence one level up (s' = dec * s + local) turns those into the true state at every chunk start:
//       one warp per (clip, bin) scans 32 chunks at a time with a shuffle prefix scan of decayed sums, so a
//       45 000-frame clip needs ~45 warp steps instead of ~1400 sequential ones,
//   (C) the chunks re-run in parallel from their true initial state, emitting dB / bytes (the magnitudes are still
//       in L1/L2).
// The three phases are grid-stride loops of one cooperative launch separated by grid barriers (the grid is sized to
// be co-resident), so a two-channel clip costs one launch after its frame kernel instead of three.
// A poisoned frame (see smooth_emit_kernel) restarts the state: (A) restarts its local sum there and records the
// restart in the sign bit of the chunk's carry (the sums are never negative, so -0.0 still says so), (B) gives such a
// chunk decay 0 -- its scan composes affine steps s' = d_j s + l_j with d_j = dec or 0 -- and (C) restarts per frame
// like the sequential kernel.  The carried state differs from the sequential kernel's by float rounding of the chunk
// sums (a few ulp): tests/test_gpu_parity.py compares the two.
// carry: [n_clips][bins][n_chunks] float (chunk fastest: phase B reads a bin's chunks coalesced).
struct ScanGeom {
  long long n_clips, frames, n_chunks;
  int bins, chunk;
  double tau;
};

template <int OUT>
__global__ void __launch_bounds__(256)
smooth_scan_kernel(const float* __restrict__ mags, typename OutElem<OUT>::type* __restrict__ out,
                   float* __restrict__ state, float* __restrict__ carry, ScanGeom sg_, Epilogue ep,
                   const uint8_t* __restrict__ poison) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  const long long n_clips = sg_.n_clips, frames = sg_.frames, n_chunks = sg_.n_chunks;
  const int bins = sg_.bins, chunk = sg_.chunk;
  const double tau = sg_.tau, k1 = 1.0 - tau;
  const long long nthreads = (long long)gridDim.x * blockDim.x, tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = n_clips * n_chunks * bins;
  // ---- (A)
  for (long long idx = tid; idx < total; idx += nthreads) {
    const int b = (int)(idx % bins);
    const long long cj = idx / bins, clip = cj / n_chunks, j = cj - clip * n_chunks;
    if (j + 1 == n_chunks) continue;          // the last chunk is nobody's predecessor
    const long long t0 = j * chunk, t1 = min(frames, t0 + (long long)chunk);
    const float* __restrict__ m = mags + clip * frames * bins + b;
    const uint8_t* __restrict__ pz = poison ? poison + clip * frames : nullptr;
    double s = 0.0;
    bool restart = false;
    long long t = t0;
    // the loads do not depend on the recurrence: eight in flight per thread, then eight dependent updates
    for (; t + 8 <= t1; t += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = finite_or_zero(__ldg(m + (t + u) * bins));
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        s = tau * s + k1 * (double)v[u];
        if (pz && __ldg(pz + t + u)) { s = 0.0; restart = true; }
      }
    }
    for (; t < t1; ++t) {
      s = tau * s + k1 * (double)finite_or_zero(__ldg(m + t * bins));
      if (pz && __ldg(pz + t)) { s = 0.0; restart = true; }
    }
    const float local = (float)s;
    carry[(clip * bins + b) * n_chunks + j] = restart ? -local : local;
  }
  grid.sync();
  // ---- (B) carry[j] <- state at the START of chunk j (in place); state[clip][bin] holds the clip's initial state
  {
    const int lane = threadIdx.x & 31;
    const double dec = pow(tau, (double)chunk);   // every chunk but the last is full, and the last one's decay is unused
    for (long long w = tid >> 5; w < n_clips * bins; w += nthreads >> 5) {
      float* __restrict__ c = carry + w * n_chunks;
      double s = (double)state[w];               // state at the start of the current 32-chunk segment
      for (long long j0 = 0; j0 < n_chunks; j0 += 32) {
        const long long j = j0 + lane;
        // chunk j maps the state at its start to d * s + y; the last chunk (nobody's predecessor) and lanes past the
        // end are the identity.  Inclusive scan of the composition (d, y) then (d', y') = (d d', d' y + y').
        double d = 1.0, y = 0.0;
        if (j + 1 < n_chunks) {
          const float v = __ldcg(c + j);
          d = signbit(v) ? 0.0 : dec;
          y = (double)fabsf(v);
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          const double up_d = __shfl_up_sync(0xffffffffu, d, 1 << k), up_y = __shfl_up_sync(0xffffffffu, y, 1 << k);
          if (lane >= (1 << k)) { y = fma(d, up_y, y); d *= up_d; }
        }
        const double prev_d = __shfl_up_sync(0xffffffffu, d, 1), prev_y = __shfl_up_sync(0xffffffffu, y, 1);
        if (j < n_chunks) c[j] = (float)(lane ? fma(prev_d, s, prev_y) : s);   // the state at the start of chunk j
        s = fma(__shfl_sync(0xffffffffu, d, 31), s, __shfl_sync(0xffffffffu, y, 31));
      }
    }
  }
  grid.sync();
  // ---- (C)
  for (long long idx = tid; idx < total; idx += nthreads) {
    const int b = (int)(idx % bins);
    const long long cj = idx / bins, clip = cj / n_chunks, j = cj - clip * n_chunks;
    const long long t0 = j * chunk, t1 = min(frames, t0 + (long long)chunk);
    const float* __restrict__ m = mags + clip * frames * bins + b;
    typename OutElem<OUT>::type* __restrict__ o = out + clip * frames * bins + b;
    const uint8_t* __restrict__ pz = poison ? poison + clip * frames : nullptr;
    float s = __ldcg(carry + (clip * bins + b) * n_chunks + j);
    long long t = t0;
    for (; t + 8 <= t1; t += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = finite_or_zero(__ldg(m + (t + u) * bins));
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        s = finite_or_zero((float)(tau * (double)s + k1 * (double)v[u]));
        if (pz && __ldg(pz + t + u)) s = 0.f;
        o[(t + u) * bins] = emit_mag<OUT>(s, ep);
      }
    }
    for (; t < t1; ++t) {
      s = finite_or_zero((float)(tau * (double)s + k1 * (double)finite_or_zero(__ldg(m + t * bins))));
      if (pz && __ldg(pz + t)) s = 0.f;
      o[t * bins] = emit_mag<OUT>(s, ep);
    }
    if (j == n_chunks - 1) state[clip * bins + b] = s;
  }
}

// re-emit a stored state vector (getByte/FloatFrequencyData called twice in one render quantum)
template <int OUT>
__global__ void emit_state_kernel(const float* __restrict__ state, typename OutElem<OUT>::type* __restrict__ out,
                                  long long n, Epilogue ep) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = emit_mag<OUT>(state[i], ep);
}

__global__ void lut_kernel(const uint8_t* __restrict__ in, uint32_t* __restrict__ out, long long n,
                           const uint32_t* __restrict__ lut) {
  __shared__ uint32_t s_lut[256];
  if (threadIdx.x < 256) s_lut[threadIdx.x] = lut[threadIdx.x];
  __syncthreads();
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if ((n & 3) == 0 && ((reinterpret_cast<uintptr_t>(in) & 3) | (reinterpret_cast<uintptr_t>(out) & 15)) == 0) {
    // four pixels per thread: 16-byte stores (the destination may be page-locked host memory: wide PCIe writes)
    const uchar4* in4 = reinterpret_cast<const uchar4*>(in);
    uint4* out4 = reinterpret_cast<uint4*>(out);
    for (long long i = first; i < n / 4; i += stride) {
      const uchar4 b = in4[i];
      out4[i] = make_uint4(s_lut[b.x], s_lut[b.y], s_lut[b.z], s_lut[b.w]);
    }
    return;
  }
  for (long long i = first; i < n; i += stride) out[i] = s_lut[in[i]];
}

// b = (unsigned char) clamp(128 * (x + 1), 0, 255)   [SPEC getByteTimeDomainData]
__global__ void time_domain_byte_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (uint8_t)byte_from_scaled(128.f * (x[i] + 1.f));
}

// ---- sonogram view (SURVEY 8(f) rank 2/3): the picture the reference draws from its byte texture, headless.
// ring: [rows][bins] u8, the bins x rows ALPHA texture of 3D/visualizer.js:301-329 written row by row at yoffset
// (:399-416).  One thread per output pixel (px, py), texCoord u = (px+.5)/W, v = (py+.5)/H:
//   s = 256^(u-1)                         log-frequency axis, sonogram-fragment.shader:16 / sonogram-vertex.shader:51
//   t = v + yoffset/(rows-1)              fragment:17 with the uniform of visualizer.js:460
//   a = LINEAR sample of alpha (byte/255), CLAMP_TO_EDGE in s, REPEAT in t      visualizer.js:312-315
//   rgb = HSV(360 - 360 a, 1, 1)          sonogram-vertex.shader:19-58 (evaluated per pixel here, per vertex there)
//   fade = sqrt(cos((1-v) pi/2))          fragment:24
//   out = clamp(0.08 + a*fade*rgb), alpha 1, 8-bit round-to-nearest            fragment:26, visualizer.js:69
// One pixel of that picture, from a [rows][bins] texture.  Shared by the single view and the batched one below so the
// two stay bit-identical: every term is evaluated in the same order on both paths.
__device__ __forceinline__ uint32_t sonogram_pixel(const uint8_t* __restrict__ ring, int bins, int rows, int yoffset,
                                                   int px, int py, int width, int height, float background) {
  const float u = (px + 0.5f) / width, v = (py + 0.5f) / height;
  const float sc = exp2f(8.f * (u - 1.f));                       // 256^(u-1)
  float tc = v + (float)yoffset / (float)(rows - 1);
  tc -= floorf(tc);                                              // REPEAT
  const float x = sc * bins - 0.5f, y = tc * rows - 0.5f;
  const float xf = floorf(x), yf = floorf(y);
  const float fx = x - xf, fy = y - yf;
  const int x0 = min(max((int)xf, 0), bins - 1), x1 = min(max((int)xf + 1, 0), bins - 1);     // CLAMP_TO_EDGE
  const int y0 = (((int)yf % rows) + rows) % rows, y1 = (y0 + 1) % rows;                      // REPEAT
  const float a00 = ring[(long long)y0 * bins + x0], a01 = ring[(long long)y0 * bins + x1];
  const float a10 = ring[(long long)y1 * bins + x0], a11 = ring[(long long)y1 * bins + x1];
  const float top = fmaf(fx, a01 - a00, a00), bot = fmaf(fx, a11 - a10, a10);
  const float a = fmaf(fy, bot - top, top) * (1.f / 255.f);
  // HSV(hue, 1, 1) with the shader's branch ladder (hue/60 == 6, i.e. a == 0, matches no branch: black)
  const float hd = (360.f - 360.f * a) * (1.f / 60.f);
  const float xx = 1.f - fabsf(fmodf(hd, 2.f) - 1.f);
  float r = 0.f, g = 0.f, b = 0.f;
  if (hd < 1.f) { r = 1.f; g = xx; }
  else if (hd < 2.f) { r = xx; g = 1.f; }
  else if (hd < 3.f) { g = 1.f; b = xx; }
  else if (hd < 4.f) { g = xx; b = 1.f; }
  else if (hd < 5.f) { r = xx; b = 1.f; }
  else if (hd < 6.f) { r = 1.f; b = xx; }
  const float k = a * sqrtf(fmaxf(cospif((1.f - v) * 0.5f), 0.f));
  auto q = [&](float c) { return (uint32_t)floorf(fminf(fmaxf(fmaf(k, c, background), 0.f), 1.f) * 255.f + 0.5f); };
  return q(r) | (q(g) << 8) | (q(b) << 16) | 0xFF000000u;
}

__global__ void __launch_bounds__(256)
sonogram_view_kernel(const uint8_t* __restrict__ ring, int bins, int rows, int yoffset, int width, int height,
                     float background, uint32_t* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)width * height) return;
  const int py = (int)(idx / width), px = (int)(idx - (long long)py * width);
  out[idx] = sonogram_pixel(ring, bins, rows, yoffset, px, py, width, height, background);
}

// The same picture for `count` textures that share rows and yoffset (a streaming bank's channels), in one launch.
// tex: [count][rows][bins] u8; out: [count][height][width] RGBA8, from cudaMalloc (16-byte aligned).
// A thread owns four neighbouring pixels of one image row and walks channels [blockIdx.y*per, +per): everything in
// sonogram_pixel but the four texel loads and what follows them is the same for every channel, so the compiler hoists
// it out of the channel loop, and each pixel's arithmetic is still exactly sonogram_view_kernel's.
// Stores are one 16-byte store per thread and channel when width % 4 == 0 (each image row then starts 16-byte aligned).
__global__ void __launch_bounds__(256)
sonogram_views_kernel(const uint8_t* __restrict__ tex, int count, int per, int bins, int rows, int yoffset, int width,
                      int height, float background, uint32_t* __restrict__ out) {
  const int qw = (width + 3) >> 2;
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (long long)qw * height) return;
  const int py = (int)(q / qw), px = (int)(q - (long long)py * qw) * 4;
  const int c0 = blockIdx.y * per, c1 = min(count, c0 + per);
  const long long plane = (long long)rows * bins, img = (long long)width * height, o0 = (long long)py * width + px;
  if ((width & 3) == 0) {
    for (int c = c0; c < c1; ++c) {
      const uint8_t* t = tex + c * plane;
      const uint4 v = make_uint4(sonogram_pixel(t, bins, rows, yoffset, px, py, width, height, background),
                                 sonogram_pixel(t, bins, rows, yoffset, px + 1, py, width, height, background),
                                 sonogram_pixel(t, bins, rows, yoffset, px + 2, py, width, height, background),
                                 sonogram_pixel(t, bins, rows, yoffset, px + 3, py, width, height, background));
      *reinterpret_cast<uint4*>(out + c * img + o0) = v;
    }
  } else {
    const int n = min(4, width - px);
    for (int c = c0; c < c1; ++c) {
      const uint8_t* t = tex + c * plane;
      for (int i = 0; i < n; ++i)
        out[c * img + o0 + i] = sonogram_pixel(t, bins, rows, yoffset, px + i, py, width, height, background);
    }
  }
}

}  // namespace sg
