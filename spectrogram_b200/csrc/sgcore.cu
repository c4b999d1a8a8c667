// libsgcore.so -- host core + C ABI (include/sgcore.h) of the B200 spectrogram engine.
//
// Replaces the browser AnalyserNode the reference configures at src/javascripts/UI/player.js:7-11
// and polls at src/javascripts/3D/visualizer.js:346-368.  No CPU fallback: every compute entry
// point runs CUDA kernels (kernel_w32.cuh, kernel_smem.cuh, kernel_misc.cuh) or fails.
#include "../../include/sgcore.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "kernel_misc.cuh"
#include "kernel_w32x2s.cuh"
#include "kernel_pcm.cuh"
#include "kernel_resample.cuh"
#include "kernel_biquad.cuh"
#include "plans.cuh"
using sg::PcmMix; using sg::PcmGeom; using sg::kPcmMaxChannels; using sg::pcm_tile_frames; using sg::launch_pcm_ingest;
using sg::RsGeom; using sg::launch_pcm_resample;

namespace {

thread_local std::string g_err = "";

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define SG_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return fail(_e == cudaErrorMemoryAllocation ? SG_ERR_OOM : SG_ERR_CUDA,              \
                  std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
  } while (0)

#define SG_TRY(expr)              \
  do {                            \
    int _rc = (expr);             \
    if (_rc != SG_OK) return _rc; \
  } while (0)

constexpr double kPi = 3.14159265358979323846264338327950288;

// ------------------------------------------------------------------------------------------
// plans: device tables for one (n_fft, window)
// ------------------------------------------------------------------------------------------
struct PlanKey {
  int n_fft, window;
  uint64_t custom_hash;
  bool operator<(const PlanKey& o) const {
    if (n_fft != o.n_fft) return n_fft < o.n_fft;
    if (window != o.window) return window < o.window;
    return custom_hash < o.custom_hash;
  }
};

struct Plan {
  int n_fft = 0, m = 0;
  std::vector<int> radix;
  float* win = nullptr;
  float2* tw = nullptr;
  float2* ut = nullptr;
  int* pos = nullptr;
  float2* w32_tw2 = nullptr;  // lane-major stage 6-10 twiddles (powers of two, 256 <= n_fft <= 8192)
  float2* w32_ut = nullptr;   // only n_fft == 2048
  float2* eo_tab = nullptr;   // only n_fft == 4096: W_2048^lane, then W_4096^{lane + 32 i}
  float2* wreg_tw3 = nullptr; // lane-major stage 11-12 twiddles (n_fft 4096, 8192)
  float2* pair_twb = nullptr; // n_fft 1024 / 512: pass-2 base twiddles of the part-warp pair kernels [log2 L][32]
  float2* w16_tw = nullptr;   // n_fft == 512: pass-2 twiddles of the 16 x 16 kernel [15][16]
  float2* r400_tw = nullptr;  // n_fft == 400: W_200^{b k1} [5][41]
  float2* r400_ut = nullptr;  // n_fft == 400: W_400^k [200]
  int log2m = 0;              // log2(n_fft/2) when n_fft is a power of two, else 0
  void release() {
    cudaFree(win); cudaFree(tw); cudaFree(ut); cudaFree(pos); cudaFree(w32_tw2); cudaFree(w32_ut); cudaFree(eo_tab); cudaFree(wreg_tw3); cudaFree(pair_twb); cudaFree(w16_tw); cudaFree(r400_tw); cudaFree(r400_ut);
  }
};

bool factorize(int m, std::vector<int>& radix) {
  radix.clear();
  while (m % 4 == 0) { radix.push_back(4); m /= 4; }
  while (m % 2 == 0) { radix.push_back(2); m /= 2; }
  while (m % 5 == 0) { radix.push_back(5); m /= 5; }
  while (m % 3 == 0) { radix.push_back(3); m /= 3; }
  return m == 1 && radix.size() <= 16;
}

void window_table(int kind, int n, const float* custom, std::vector<float>& w) {
  w.resize(n);
  for (int i = 0; i < n; ++i) {
    const double x = (double)i / (double)n;
    double v;
    switch (kind) {
      case SG_WINDOW_BLACKMAN: {
        const double alpha = 0.16, a0 = 0.5 * (1 - alpha), a1 = 0.5, a2 = 0.5 * alpha;
        v = a0 - a1 * std::cos(2 * kPi * x) + a2 * std::cos(4 * kPi * x);
        break;
      }
      case SG_WINDOW_HANN: v = 0.5 - 0.5 * std::cos(2 * kPi * x); break;
      case SG_WINDOW_CUSTOM: v = custom[i]; break;
      default: v = 1.0;
    }
    w[i] = (float)v;  // computed in double, cast to float (as Chromium's ApplyWindow)
  }
}

uint64_t fnv1a(const void* p, size_t n) {
  const unsigned char* b = (const unsigned char*)p;
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
  return h;
}

float2 expi(double turns) {  // exp(-2 pi i turns)
  return make_float2((float)std::cos(-2 * kPi * turns), (float)std::sin(-2 * kPi * turns));
}

template <class T>
int upload(T** dst, const std::vector<T>& src) {
  SG_CUDA(cudaMalloc((void**)dst, std::max<size_t>(src.size(), 1) * sizeof(T)));
  SG_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
  return SG_OK;
}

int build_plan(const sg_stft_config& cfg, Plan& p) {
  p.n_fft = cfg.n_fft;
  p.m = cfg.n_fft / 2;
  if (!factorize(p.m, p.radix)) return fail(SG_ERR_INDEX_SIZE, "n_fft/2 must factor into 2, 3, 5");
  const int m = p.m, n = p.n_fft;
  std::vector<float> win;
  window_table(cfg.window, n, cfg.custom_window, win);
  // the frame-pair kernel parks its idle prefetch loads on this table: keep 4096 readable floats behind it
  if (n == sg::kW32N) win.resize(2 * sg::kW32N, 0.f);
  if (n == 1024 || n == 512 || n == 256) win.resize(2 * n, 0.f);
  std::vector<float2> tw(m), ut(m / 2 + 1);
  for (int k = 0; k < m; ++k) tw[k] = expi((double)k / m);
  for (int k = 0; k <= m / 2; ++k) ut[k] = expi((double)k / n);
  // digit reversal of the in-place DIF: k = q1 + R1*(q2 + R2*(...)) sits at sum q_i * m/(R1..Ri)
  std::vector<int> pos(m);
  for (int k = 0; k < m; ++k) {
    int rem = k, span = m, at = 0;
    for (int r : p.radix) { span /= r; at += (rem % r) * span; rem /= r; }
    pos[k] = at;
  }
  SG_TRY(upload(&p.win, win));
  SG_TRY(upload(&p.tw, tw));
  SG_TRY(upload(&p.ut, ut));
  SG_TRY(upload(&p.pos, pos));
  if ((m & (m - 1)) == 0) {
    while ((1 << p.log2m) < m) ++p.log2m;
  }
  if (p.log2m >= 7 && p.log2m <= 12) {
    std::vector<float2> tw2(31 * 32);
    for (int u = 1; u <= 5; ++u) {
      const int half = 1 << (u - 1);
      for (int q = 0; q < half; ++q)
        for (int lane = 0; lane < 32; ++lane)
          tw2[(half - 1 + q) * 32 + lane] = expi((double)(q * 32 + lane) / (32.0 * 2 * half));
    }
    SG_TRY(upload(&p.w32_tw2, tw2));
    const int r3 = p.log2m - 10;
    if (r3 > 0) {
      const int s3 = 1 << r3;
      std::vector<float2> tw3((size_t)32 * (s3 - 1) * 32);
      for (int q = 0; q < 32; ++q)
        for (int u = 1; u <= r3; ++u) {
          const int half = 1 << (u - 1);
          for (int pp = 0; pp < half; ++pp)
            for (int ka = 0; ka < 32; ++ka)
              tw3[((size_t)q * (s3 - 1) + half - 1 + pp) * 32 + ka] =
                  expi((double)(pp * 1024 + q * 32 + ka) / (1024.0 * 2 * half));
        }
      SG_TRY(upload(&p.wreg_tw3, tw3));
    }
  }
  if (n == 1024 || n == 512 || n == 256) {
    const int log2l = n == 1024 ? 4 : n == 512 ? 3 : 2;
    std::vector<float2> twb(log2l * 32);
    for (int u = 1; u <= log2l; ++u)
      for (int col = 0; col < 32; ++col) twb[(u - 1) * 32 + col] = expi((double)col / (32.0 * (1 << u)));
    SG_TRY(upload(&p.pair_twb, twb));
  }
  if (n == 512 || n == 256) {
    const int rows = n == 512 ? 15 : 7;     // pass 2 is a 16- or 8-point DIT: half = 1 .. rows/2 + 1
    std::vector<float2> tw16(rows * 16);
    for (int half = 1; half <= (rows + 1) / 2; half *= 2)
      for (int pp = 0; pp < half; ++pp)
        for (int col = 0; col < 16; ++col)
          tw16[(half - 1 + pp) * 16 + col] = expi((double)(16 * pp + col) / (32.0 * half));
    SG_TRY(upload(&p.w16_tw, tw16));
  }
  if (n == 400) {
    std::vector<float2> tw5(5 * 41), ut4(200);
    for (int b = 0; b < 5; ++b)
      for (int k1 = 0; k1 < 41; ++k1) tw5[b * 41 + k1] = expi((double)((b * k1) % 200) / 200.0);
    for (int k = 0; k < 200; ++k) ut4[k] = expi((double)k / 400.0);
    SG_TRY(upload(&p.r400_tw, tw5));
    SG_TRY(upload(&p.r400_ut, ut4));
  }
  if (n == sg::kEoN) {
    std::vector<float2> tab(32 + 16 * 32);
    for (int lane = 0; lane < 32; ++lane) tab[lane] = expi((double)lane / 2048.0);
    for (int i = 0; i < 16; ++i)
      for (int lane = 0; lane < 32; ++lane) tab[32 + i * 32 + lane] = expi((double)(lane + 32 * i) / n);
    SG_TRY(upload(&p.eo_tab, tab));
  }
  if (n == sg::kW32N) {
    std::vector<float2> ut32(16 * 32);
    for (int i = 0; i < 16; ++i)
      for (int lane = 0; lane < 32; ++lane) ut32[i * 32 + lane] = expi((double)(lane + 32 * i) / n);
    SG_TRY(upload(&p.w32_ut, ut32));
  }
  return SG_OK;
}

// ------------------------------------------------------------------------------------------
// colour LUT (bin/shaders/sonogram-vertex.shader:19-58, sonogram-fragment.shader:24-26)
// ------------------------------------------------------------------------------------------
void hsv_to_rgb(double hue, double* rgb) {
  const double chroma = 1.0, hd = hue / 60.0;
  const double x = chroma * (1.0 - std::fabs(std::fmod(hd, 2.0) - 1.0));
  rgb[0] = rgb[1] = rgb[2] = 0.0;
  if (hd < 1.0) { rgb[0] = chroma; rgb[1] = x; }
  else if (hd < 2.0) { rgb[0] = x; rgb[1] = chroma; }
  else if (hd < 3.0) { rgb[1] = chroma; rgb[2] = x; }
  else if (hd < 4.0) { rgb[1] = x; rgb[2] = chroma; }
  else if (hd < 5.0) { rgb[0] = x; rgb[2] = chroma; }
  else if (hd < 6.0) { rgb[0] = chroma; rgb[2] = x; }
  // hd == 6 (byte 0) matches no branch in the shader: black
}

void reference_lut(uint32_t* lut) {
  const double bg = 0.08;  // 3D/visualizer.js:69
  for (int b = 0; b < 256; ++b) {
    const double a = b / 255.0;
    double rgb[3];
    hsv_to_rgb(360.0 - a * 360.0, rgb);
    uint32_t px = 0xFF000000u;
    for (int c = 0; c < 3; ++c) {
      const double v = std::min(std::max(bg + a * rgb[c], 0.0), 1.0);
      px |= (uint32_t)std::floor(v * 255.0 + 0.5) << (8 * c);
    }
    lut[b] = px;
  }
}

int validate_cfg(const sg_stft_config* cfg) {
  if (!cfg) return fail(SG_ERR_INVALID_ARG, "cfg is null");
  if (cfg->n_fft < 4 || cfg->n_fft > 32768 || (cfg->n_fft & 1))
    return fail(SG_ERR_INDEX_SIZE, "n_fft must be even and in [4, 32768]");
  std::vector<int> r;
  if (!factorize(cfg->n_fft / 2, r)) return fail(SG_ERR_INDEX_SIZE, "n_fft/2 must factor into 2, 3, 5");
  if (cfg->hop < 1) return fail(SG_ERR_INDEX_SIZE, "hop must be >= 1");
  if (cfg->window < SG_WINDOW_BLACKMAN || cfg->window > SG_WINDOW_CUSTOM)
    return fail(SG_ERR_INVALID_ARG, "unknown window");
  if (cfg->window == SG_WINDOW_CUSTOM && !cfg->custom_window)
    return fail(SG_ERR_INVALID_ARG, "custom window pointer is null");
  if (cfg->output < SG_OUT_U8 || cfg->output > SG_OUT_F32_MAG) return fail(SG_ERR_INVALID_ARG, "unknown output kind");
  if (cfg->align != SG_ALIGN_VALID && cfg->align != SG_ALIGN_ANALYSER) return fail(SG_ERR_INVALID_ARG, "unknown alignment");
  if (!(cfg->min_db < cfg->max_db)) return fail(SG_ERR_INDEX_SIZE, "minDecibels must be < maxDecibels");
  if (!(cfg->smoothing >= 0.f && cfg->smoothing <= 1.f))
    return fail(SG_ERR_INDEX_SIZE, "smoothingTimeConstant must be in [0, 1]");
  return SG_OK;
}

long long frames_for(const sg_stft_config& c, long long clip_len) {
  if (c.align == SG_ALIGN_VALID) return clip_len < c.n_fft ? 0 : 1 + (clip_len - c.n_fft) / c.hop;
  return clip_len / c.hop;
}

size_t elem_bytes(int output) { return output == SG_OUT_U8 ? 1 : 4; }

sg::Epilogue make_epilogue(const sg_stft_config& c, double norm, const uint32_t* lut_dev) {
  sg::Epilogue e;
  const double db_scale = 10.0 * std::log10(2.0);
  const double db_off = -20.0 * std::log10(norm);
  const double s = 255.0 / ((double)c.max_db - (double)c.min_db);
  e.db_scale = (float)db_scale;
  e.db_off = (float)db_off;
  e.byte_a = (float)(s * db_scale);
  e.byte_b = (float)(s * (db_off - (double)c.min_db));
  e.byte_b0 = (float)(s * (-(double)c.min_db));
  e.mag_scale = (float)(1.0 / norm);
  e.lut = lut_dev;
  return e;
}

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t n) {
    if (n <= cap) return SG_OK;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    SG_CUDA(cudaMalloc(&p, n));
    cap = n;
    return SG_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t n) {
    if (n <= cap) return SG_OK;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    SG_CUDA(cudaHostAlloc(&p, n, cudaHostAllocDefault));
    cap = n;
    return SG_OK;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// Polyphase filter of one reduced ratio up/down (sg_pcm.inl designs it): [up][J] float32 taps, phase-major
struct RsTable {
  int up = 1, down = 1, half = 0, J = 0;
  DevBuf taps;
};

bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// engine
// ------------------------------------------------------------------------------------------
struct sg_engine {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;     // compute
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  std::map<PlanKey, Plan> plans;
  uint32_t* lut_ref = nullptr;       // device, reference colour map
  DevBuf lut_user;                   // device copy of cfg.colormap
  DevBuf scratch_mag, scratch_state, scratch_carry, scratch_poison, d_in, d_out;
  DevBuf xs_carry, xs_flags, xs_state;         // fused-smoothing kernel: per-segment carry vectors and their ready flags
  unsigned xs_epoch = 0;
  DevBuf d_raw[2];                   // interleaved PCM bytes in flight (sg_stft_pcm)
  std::map<std::pair<int, int>, RsTable> rs_tables;   // resampling filters by (up, down)
  DevBuf bq_start, bq_agg, bq_io, bq_state;           // biquad filter: tile records (shared scratch), host-call staging
  PinBuf pin_in[2], pin_out[2];
  int64_t launches = 0;
  int kernel_variant = 0;            // 0 auto, 1 force generic smem kernel
  const char* last_kernel = "none";
  std::mutex mu;
  // The scratch buffers above (smoothing state, magnitude tiles, carry vectors, the custom colour table) are shared by
  // every call on this engine, whatever stream the caller passes.  A call that uses them first makes its stream wait
  // for the previous user's last kernel and records its own end on this event afterwards.
#ifdef SG_DEBUG
  sg::DbgState dbg{};                // epoch-tag buffers of the SG_DEBUG build (common.cuh)
#endif
  cudaEvent_t ev_scratch = nullptr;
  cudaEvent_t ev_ring_in[4] = {}, ev_ring_k[4] = {}, ev_pin_in[2] = {}, ev_pin_out[2] = {};   // sg_stft_batch's pipeline
  bool scratch_busy = false;
  int scratch_acquire(cudaStream_t st) {
    if (scratch_busy) SG_CUDA(cudaStreamWaitEvent(st, ev_scratch, 0));
    return SG_OK;
  }
  int scratch_release(cudaStream_t st) {
    SG_CUDA(cudaEventRecord(ev_scratch, st));
    scratch_busy = true;
    return SG_OK;
  }

  int get_plan(const sg_stft_config& cfg, Plan** out) {
    PlanKey key{cfg.n_fft, cfg.window,
                cfg.window == SG_WINDOW_CUSTOM ? fnv1a(cfg.custom_window, sizeof(float) * cfg.n_fft) : 0};
    auto it = plans.find(key);
    if (it == plans.end()) {
      Plan p;
      int rc = build_plan(cfg, p);
      if (rc != SG_OK) { p.release(); return rc; }
      it = plans.emplace(key, p).first;
    }
    *out = &it->second;
    return SG_OK;
  }

  int lut_for(const sg_stft_config& cfg, cudaStream_t st, const uint32_t** out) {
    if (!cfg.colormap || cfg.output != SG_OUT_RGBA8) { *out = lut_ref; return SG_OK; }
    SG_TRY(lut_user.reserve(256 * sizeof(uint32_t)));
    SG_CUDA(cudaMemcpyAsync(lut_user.p, cfg.colormap, 256 * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    *out = (const uint32_t*)lut_user.p;
    return SG_OK;
  }
};

namespace {

// Picks the kernel family for a launch group and enqueues it (the families live in tu_*.cu).
int launch_frames(sg_engine* e, const Plan& pl, const sg::FrameGeom& g, const sg_stft_config& cfg, int out_kind,
                  const uint32_t* lut, void* out, cudaStream_t st) {
  if (g.total_frames <= 0) return SG_OK;
  const sg::Epilogue ep = make_epilogue(cfg, 2.0 * pl.n_fft, lut);
  const int v = e->kernel_variant == 7 ? 0 : e->kernel_variant;   // 7 only concerns the smoothing path
  // The packed kernels' byte path takes lg2 with subnormal powers flushed to zero (|X|/N < 1e-19, below
  // -380 dB): exact for any minDecibels above that, otherwise the one-frame kernel is used.
  const bool bytes_out = out_kind == SG_OUT_U8 || out_kind == SG_OUT_RGBA8;
  const bool x2_ok = !bytes_out || cfg.min_db >= -300.f;
  int rc;
  // float rows (dB, magnitude) at hop 512 are store-heavy (8 KB per pair): the TMA-staged kernel with 8 warps per SM
  // measured 556 M frames/s (dB) / 549 M (magnitude) against 526 M / 520 M on the register-pipelined one (12 warps),
  // so those outputs take the branch below
  const bool db512 = v == 0 && (out_kind == SG_OUT_F32_DB || out_kind == SG_OUT_F32_MAG) && g.hop == 512;
  if (pl.n_fft == sg::kW32N && (g.hop == 512 || (v == 0 && g.hop == 256)) && (v == 0 || v == 6) && x2_ok && !db512) {
    const sg::W32Plan wp{pl.win, pl.w32_tw2, pl.w32_ut};
    rc = sg::launch_w32x2p(out_kind, v == 6 ? 8 : 12, g, wp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "warp32x32x2p";
  } else if (pl.n_fft == sg::kW32N && (v == 4 || (v == 0 && g.hop <= 1024)) && x2_ok) {
    // (hops above 1024 samples -- two frames no longer fit the stage -- are faster on the one-frame-per-warp kernel
    // than on this kernel's guarded loads; hops that are not a multiple of 4 samples take its unaligned-span form)
    const sg::W32Plan wp{pl.win, pl.w32_tw2, pl.w32_ut};
    rc = sg::launch_w32x2(out_kind, g, wp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "warp32x32x2";
  } else if (pl.n_fft == sg::kW32N && v != 1 && v != 3) {
    const sg::W32Plan wp{pl.win, pl.w32_tw2, pl.w32_ut};
    rc = sg::launch_w32(out_kind, g, wp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "warp32x32";
  } else if (pl.n_fft == sg::kEoN && (v == 0 || v == 6) && x2_ok && (g.hop & 3) == 0) {
    // (hops that are not a multiple of 4 samples leave no frame 16-byte aligned: the register family's 4-byte loads
    // are faster there, 152 vs 121 M frames/s at hop 441)
    const sg::EoPlan eo{pl.win, pl.w32_tw2, pl.eo_tab};
    rc = sg::launch_w32eo(out_kind, v == 6 ? 12 : 8, g, eo, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "eo4096";
  } else if (pl.n_fft == 400 && v != 1) {
    const sg::R400Plan rp{pl.win, pl.r400_tw, pl.r400_ut};
    rc = sg::launch_r400(out_kind, g, rp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "r400";
  } else if (sg::pair_kernel_serves(pl.n_fft, g.hop) && v == 0 && x2_ok && g.frames_per_clip >= 4 &&
             (pl.n_fft >= 512 || bytes_out)) {   // n_fft 256 float outputs: the 16 x 8 kernel is faster (3.67 vs 2.93 G frames/s)
    // (a streaming push has one frame per channel: consecutive frames are different clips and the pair loader
    // cannot share their samples -- those launches stay on the per-frame kernels)
    const sg::PairPlan pp{pl.win, pl.pair_twb, pl.ut};
    rc = pl.n_fft == 1024 ? sg::launch_pair_l4(out_kind, g, pp, ep, out, e->sm_count, e->device, st)
         : pl.n_fft == 512 ? sg::launch_pair_l3(out_kind, g, pp, ep, out, e->sm_count, e->device, st)
                           : sg::launch_pair_l2(out_kind, g, pp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = pl.n_fft == 1024 ? "p16" : pl.n_fft == 512 ? "p8" : "p4";
  } else if (pl.n_fft == 256 && v != 1 && v != 3) {
    const sg::W16Plan wp{pl.win, pl.w16_tw, pl.ut};
    rc = sg::launch_w16x8(out_kind, g, wp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "w16";
  } else if (pl.n_fft == 512 && v != 1 && v != 3) {
    const sg::W16Plan wp{pl.win, pl.w16_tw, pl.ut};
    rc = sg::launch_w16(out_kind, g, wp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "w16";
  } else if (pl.log2m >= 7 && pl.log2m <= 12 && v != 1) {
    const sg::WregPlan wp{pl.win, pl.w32_tw2, pl.wreg_tw3, pl.ut};
    switch (out_kind) {
      case SG_OUT_U8: rc = sg::launch_wreg_out0(pl.log2m, g, wp, ep, out, e->sm_count, e->device, st); break;
      case SG_OUT_F32_DB: rc = sg::launch_wreg_out1(pl.log2m, g, wp, ep, out, e->sm_count, e->device, st); break;
      case SG_OUT_RGBA8: rc = sg::launch_wreg_out2(pl.log2m, g, wp, ep, out, e->sm_count, e->device, st); break;
      default: rc = sg::launch_wreg_out3(pl.log2m, g, wp, ep, out, e->sm_count, e->device, st); break;
    }
    e->last_kernel = "wreg";
  } else {
    sg::SmemPlan sp;
    sp.win = pl.win; sp.tw = pl.tw; sp.ut = pl.ut; sp.pos = pl.pos; sp.m = pl.m;
    sp.nstage = (int)pl.radix.size();
    for (int i = 0; i < sp.nstage; ++i) sp.radix[i] = pl.radix[i];
    rc = sg::launch_smem(out_kind, g, sp, ep, out, e->sm_count, e->device, st);
    e->last_kernel = "smem";
  }
  e->launches++;
  SG_CUDA((cudaError_t)rc);
  return SG_OK;
}

template <int OUT>
int launch_smooth_t(sg_engine* e, const float* mags, void* out, float* state, long long n_clips, long long frames,
                    int bins, double tau, const sg::Epilogue& ep, const uint8_t* poison, cudaStream_t st) {
  using T = typename sg::OutElem<OUT>::type;
  const long long n = n_clips * bins;
  if (n <= 0 || frames <= 0) return SG_OK;
  // few (clip, bin) pairs and many frames: cut time into chunks so the GPU has threads to run (one cooperative
  // kernel: chunk sums, carry scan, emit)
  const long long want_threads = 2048LL * e->sm_count;
  if (n < want_threads && frames >= 256) {
    const int chunk = (int)std::max<long long>(32, std::min<long long>(1024, frames * n / want_threads));
    const long long n_chunks = (frames + chunk - 1) / chunk;
    const long long nt = n * n_chunks, blocks = (nt + 255) / 256;
    SG_TRY(e->scratch_carry.reserve((size_t)nt * sizeof(float)));
    float* carry = (float*)e->scratch_carry.p;
    // cooperative launch: the whole grid must be resident for its two grid barriers
    static int per_sm[sg::kMaxDevices] = {};
    int& occ = per_sm[e->device >= 0 && e->device < sg::kMaxDevices ? e->device : 0];
    if (occ == 0) SG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sg::smooth_scan_kernel<OUT>, 256, 0));
    const unsigned grid = (unsigned)std::min<long long>(blocks, (long long)occ * e->sm_count);
    sg::ScanGeom sgm{n_clips, frames, n_chunks, bins, chunk, tau};
    T* out_t = (T*)out;
    sg::Epilogue ep_c = ep;
    void* args[] = {(void*)&mags, (void*)&out_t, (void*)&state, (void*)&carry, (void*)&sgm, (void*)&ep_c, (void*)&poison};
    SG_CUDA(cudaLaunchCooperativeKernel((const void*)sg::smooth_scan_kernel<OUT>, dim3(grid), dim3(256), args, 0, st));
    e->launches++;
    SG_CUDA(cudaGetLastError());
    return SG_OK;
  }
  sg::smooth_emit_kernel<OUT><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(mags, (T*)out, state, n_clips, frames,
                                                                          bins, tau, ep, poison);
  e->launches++;
  SG_CUDA(cudaGetLastError());
  return SG_OK;
}

int launch_smooth(sg_engine* e, int out_kind, const float* mags, void* out, float* state, long long n_clips,
                  long long frames, int bins, double tau, const sg::Epilogue& ep, const uint8_t* poison, cudaStream_t st) {
  switch (out_kind) {
    case SG_OUT_U8: return launch_smooth_t<sg::kOutU8>(e, mags, out, state, n_clips, frames, bins, tau, ep, poison, st);
    case SG_OUT_F32_DB: return launch_smooth_t<sg::kOutF32Db>(e, mags, out, state, n_clips, frames, bins, tau, ep, poison, st);
    case SG_OUT_RGBA8: return launch_smooth_t<sg::kOutRgba8>(e, mags, out, state, n_clips, frames, bins, tau, ep, poison, st);
    default: return launch_smooth_t<sg::kOutF32Mag>(e, mags, out, state, n_clips, frames, bins, tau, ep, poison, st);
  }
}

// the frames of `g` that hold a NaN / Inf sample, [clip][frame] bytes in the engine's scratch: the two-kernel path's
// recurrence restarts there ([SPEC] "non-finite X^ -> 0"; the frame kernel has already written their magnitudes as 0)
int launch_poison(sg_engine* e, const sg::FrameGeom& g, cudaStream_t st, const uint8_t** out) {
  SG_TRY(e->scratch_poison.reserve((size_t)g.total_frames));
  sg::poison_flags_kernel<<<(unsigned)((g.total_frames * 32 + 255) / 256), 256, 0, st>>>(g, (uint8_t*)e->scratch_poison.p);
  e->launches++;
  SG_CUDA(cudaGetLastError());
  *out = (const uint8_t*)e->scratch_poison.p;
  return SG_OK;
}

// tau > 0 at n_fft 2048 / hop 512 or 256: the recurrence fused into the frame-pair kernel (kernel_w32x2s.cuh), one launch,
// no magnitude scratch.  Returns SG_OK with *done = false when the shape is not served.
int launch_fused_smoothing(sg_engine* e, const Plan& pl, const sg_stft_config& cfg, const float* pcm_dev, long long n_clips,
                           long long clip_len, long long clip_stride, long long start0, long long nframes,
                           long long out_clip_rows, void* out, float* state, const uint32_t* lut, cudaStream_t st,
                           bool* done) {
  *done = false;
  const bool bytes_out = cfg.output == SG_OUT_U8 || cfg.output == SG_OUT_RGBA8;
  // n_fft 2048: kernel_w32x2s.cuh; n_fft 1024 / 512 / 256: kernel_pair_s.cuh (chained segments only); hop n_fft/2, /4 or /8.
  // n_fft 4096: kernel_w32eo_s.cuh (chained segments only)
  const bool part_warp = pl.n_fft == 1024 || pl.n_fft == 512 || pl.n_fft == 256;
  const bool even_odd = pl.n_fft == sg::kEoN;      // kernel_w32eo_s.cuh: any hop that keeps frames 16-byte aligned
  if (e->kernel_variant != 0 && e->kernel_variant != 7) return SG_OK;
  // register family (kernel_wreg_s.cuh): n_fft 8192, and 4096 where the even/odd kernel's 16-byte loader cannot go
  bool reg_family = pl.n_fft == 8192;
  if (even_odd && ((cfg.hop & 3) || (clip_stride & 3) || (reinterpret_cast<uintptr_t>(pcm_dev) & 15))) reg_family = true;
  if (reg_family) {
    if (cfg.hop > pl.n_fft || !pl.wreg_tw3) return SG_OK;
  } else if (even_odd) {
  } else if (pl.n_fft == sg::kW32N) {
    if (cfg.hop > 2048) return SG_OK;        // any hop up to n_fft (kernel_w32x2s.cuh: hop 1024 / 512 / 256 share loads)
  } else if (!part_warp || cfg.hop > pl.n_fft) {
    return SG_OK;        // (part-warp kernels: hop n/2, n/4, n/8 and 160 share loads, every other hop loads directly)
  }
  const int bins = pl.n_fft / 2;
  const int step_frames = reg_family ? 256 / (pl.n_fft / 64) : part_warp ? 2 * (32 / (pl.n_fft / 64)) : even_odd ? 1 : 2;   // frames taken at once
  // Every clip is one chain of segments, so the kernel keeps min(n_clips, SMs) CTAs busy.  Below ~2/3 of the SMs the
  // two-kernel path wins (64 x 60 s clips: 1.57 ms against 3.86 ms here, two clips 0.078 against 0.172 ms); variant 7
  // forces this kernel for any clip count (the tests use it to reach the look-back mode).
  if ((bytes_out && cfg.min_db < -300.f) || nframes <= 0 || n_clips <= 0 || nframes > (1 << 28)) return SG_OK;
  const int grid_max = (reg_family ? 2 : 1) * e->sm_count;                          // co-resident CTAs
  const int nw = reg_family ? step_frames : part_warp ? 8 * (step_frames / 2) : even_odd ? 4 : 12;   // pairs in one round of a CTA
  sg::XsGeom x;
  x.n_clips = n_clips;
  x.out_clip_rows = out_clip_rows;
  x.warm = 0;
  auto even_up = [step_frames](long long v) { return (v + step_frames - 1) / step_frames * step_frames; };   // whole warp steps
  long long segs, seg_frames;
  const bool few = 3 * n_clips < 2 * (long long)grid_max;
  bool warm_up = false;
  if (few && e->kernel_variant != 7) {
    // Too few clips for one chain per CTA to fill the GPU.  Cut every clip into grid_max / n_clips INDEPENDENT segments:
    // each starts `warm` frames early from a zero state and writes no rows until its own first frame.  What a segment
    // misses of the true state has decayed by tau^warm < 2^-149 by then -- below the smallest float32 denormal, so the
    // rows are those of the sequential recurrence (the same argument bounds the state a clip hands back).  The extra
    // frames cost warm / seg_frames of the arithmetic; when that is more than the whole segment (long memories: tau close
    // to 1; or very few frames per CTA) it is not worth it.
    const double tau = (double)cfg.smoothing;
    const long long per_clip = grid_max / n_clips;
    if (tau > 0.0 && tau < 1.0 && per_clip >= 2 && !(part_warp && cfg.hop * 4 != pl.n_fft)) {   // (part-warp kernels: hop n/4 only)
      const long long warm = even_up((long long)std::ceil(103.3 / -std::log(tau)));
      seg_frames = even_up((nframes + per_clip - 1) / per_clip);
      if (seg_frames >= warm && seg_frames >= 8 * nw && warm <= (1 << 24)) {
        warm_up = true;
        x.mode = 2;
        x.warm = (int)warm;
      }
    }
    // otherwise: one chain per clip on n_clips CTAs still beats the two-kernel path from ~45 % of the CTAs up (the
    // two-kernel path runs at ~0.4 of the fused kernels' rate); below that, the two-kernel path
    // (break-even against each family's two-kernel rate: 0.40 of the fused rate at n_fft 2048 and 4096, 0.48 for the
    //  part-warp kernels, 0.65 for the register family)
    const long long min_chain = reg_family ? (2 * (long long)grid_max + 2) / 3 : part_warp ? grid_max / 2 : (9 * (long long)grid_max + 19) / 20;
    if (!warm_up && n_clips < min_chain) return SG_OK;
  }
  if (warm_up) {
  } else if (e->kernel_variant == 7 && 2 * n_clips <= grid_max && pl.n_fft == sg::kW32N) {
    // (tests only: it loses to every alternative) every segment gets a CTA of its own: aggregate pass, look-back, emit pass
    seg_frames = std::max<long long>(2 * nw, even_up((nframes + grid_max / n_clips - 1) / (grid_max / n_clips)));
    x.mode = 1;
  } else {
    // chained segments: pick the split that fills whole waves of CTAs best, segments of at least four rounds of pairs
    // (fewer clips than co-resident CTAs: a clip's second segment would sit beside its first and only wait for it)
    long long best_s = 1;
    double best_eff = 0.0;
    const long long s_max = (n_clips < grid_max && e->kernel_variant != 7) ? 1 : 64;   // (variant 7: the tests want chains)
    for (long long s_try = 1; s_try <= s_max; ++s_try) {
      const long long sf = even_up((nframes + s_try - 1) / s_try);
      if (s_try > 1 && sf < 8 * nw) break;
      const long long tasks = ((nframes + sf - 1) / sf) * n_clips, waves = (tasks + grid_max - 1) / grid_max;
      const double eff = (double)tasks / (double)(waves * grid_max);
      if (eff > best_eff + 0.005) { best_eff = eff; best_s = s_try; }
    }
    seg_frames = even_up((nframes + best_s - 1) / best_s);
    x.mode = 0;
  }
  segs = (nframes + seg_frames - 1) / seg_frames;
  const long long tasks = segs * n_clips;
  if (tasks >= (1LL << 31)) return SG_OK;
  x.seg_frames = (int)seg_frames;
  x.segs = (int)segs;
  x.tau = cfg.smoothing;
  x.mscale = (float)((1.0 - (double)cfg.smoothing) / (2.0 * pl.n_fft));
  x.dec = (float)std::pow((double)cfg.smoothing, (double)seg_frames);
  x.state_in = state;
  x.state_out = state;
  const size_t state_bytes = (size_t)n_clips * bins * sizeof(float);
  if (x.mode != 0) {
    // the segments of a clip run concurrently and every one of them reads the clip's initial state: the final state
    // goes to a buffer of its own and is copied over afterwards
    SG_TRY(e->xs_state.reserve(state_bytes));
    x.state_out = (float*)e->xs_state.p;
  }
  SG_TRY(e->xs_carry.reserve((size_t)tasks * (bins / 2) * sizeof(float2)));
  if ((size_t)tasks * sizeof(unsigned) > e->xs_flags.cap) {
    SG_TRY(e->xs_flags.reserve(std::max<size_t>(4 * (size_t)tasks, 4096) * sizeof(unsigned)));
    SG_CUDA(cudaMemsetAsync(e->xs_flags.p, 0, e->xs_flags.cap, st));   // flags only ever hold epochs of earlier launches
  }
  x.carry = (float2*)e->xs_carry.p;
  x.flags = (unsigned*)e->xs_flags.p;
  x.epoch = ++e->xs_epoch;
  sg::FrameGeom g{pcm_dev, clip_len, clip_stride, nframes, n_clips * nframes, start0, cfg.n_fft, cfg.hop};
  const sg::Epilogue ep = make_epilogue(cfg, 2.0 * pl.n_fft, lut);
  const int grid = (int)std::min<long long>(tasks, grid_max);
  static const bool trace = getenv("SG_TRACE_FUSED") != nullptr;
  if (trace)
    fprintf(stderr, "[sgcore] fused smoothing: n_fft %d hop %d clips %lld frames %lld mode %d segs %lld seg_frames %lld warm %d grid %d\n",
            pl.n_fft, cfg.hop, n_clips, nframes, x.mode, segs, seg_frames, x.warm, grid);
  int rc;
  const char* name;
  if (reg_family) {
    const sg::WregPlan wp{pl.win, pl.w32_tw2, pl.wreg_tw3, pl.ut};
    rc = sg::launch_wreg_s(cfg.output, pl.log2m, g, x, wp, ep, out, grid, e->device, st);
    name = "wregs";
  } else if (even_odd) {
    const sg::EoPlan eo{pl.win, pl.w32_tw2, pl.eo_tab};
    rc = sg::launch_w32eo_s(cfg.output, g, x, eo, ep, out, grid, e->device, st);
    name = "eo4096s";
  } else if (part_warp) {
    const sg::PairPlan pp{pl.win, pl.pair_twb, pl.ut};
    rc = pl.n_fft == 1024 ? sg::launch_pair_s_l4(cfg.output, g, x, pp, ep, out, grid, e->device, st)
         : pl.n_fft == 512 ? sg::launch_pair_s_l3(cfg.output, g, x, pp, ep, out, grid, e->device, st)
                           : sg::launch_pair_s_l2(cfg.output, g, x, pp, ep, out, grid, e->device, st);
    name = pl.n_fft == 1024 ? "p16s" : pl.n_fft == 512 ? "p8s" : "p4s";
  } else {
    const sg::W32Plan wp{pl.win, pl.w32_tw2, pl.w32_ut};
    rc = sg::launch_w32x2s(cfg.output, g, x, wp, ep, out, grid, e->device, st);
    name = "warp32x32x2s";
  }
  if (rc == (int)cudaErrorCooperativeLaunchTooLarge || rc == (int)cudaErrorLaunchOutOfResources) {
    // the grid cannot be made co-resident on this device right now (fewer free SMs than the properties say: a partitioned
    // or shared GPU): nothing was launched -- the two-kernel path takes the call
    cudaGetLastError();
    return SG_OK;
  }
  SG_CUDA((cudaError_t)rc);
  e->last_kernel = name;
  if (x.mode != 0) SG_CUDA(cudaMemcpyAsync(state, x.state_out, state_bytes, cudaMemcpyDeviceToDevice, st));
  e->launches++;
  *done = true;
  return SG_OK;
}

// One launch group over `n_clips` clips x frames [t0, t0+nframes) of each clip.
// tau == 0: a single fused kernel.  tau > 0: a fused smoothing kernel, or the frames' non-finite flags, the frame
// kernel -> linear magnitudes (scratch) and the recurrence + dB/byte kernel, chained through `state` ([n_clips][bins]).
int run_range(sg_engine* e, const Plan& pl, const sg_stft_config& cfg, const float* pcm_dev, long long n_clips,
              long long clip_len, long long clip_stride, long long t0, long long nframes, long long frames_total,
              void* out_dev, float* state, const uint32_t* lut, cudaStream_t st) {
  const int bins = cfg.n_fft / 2;
  const long long start0 = (cfg.align == SG_ALIGN_VALID ? 0 : (long long)cfg.hop - cfg.n_fft) + t0 * cfg.hop;
  const size_t eb = elem_bytes(cfg.output);
  if (cfg.smoothing == 0.f) {
    if (n_clips == 1 || nframes == frames_total) {
      sg::FrameGeom g{pcm_dev, clip_len, clip_stride, nframes, n_clips * nframes, start0, cfg.n_fft, cfg.hop};
      char* o = (char*)out_dev + (size_t)t0 * bins * eb;
      return launch_frames(e, pl, g, cfg, cfg.output, lut, o, st);
    }
    for (long long c = 0; c < n_clips; ++c) {  // partial frame range of several clips: per clip
      sg::FrameGeom g{pcm_dev + c * clip_stride, clip_len, clip_stride, nframes, nframes, start0, cfg.n_fft, cfg.hop};
      char* o = (char*)out_dev + ((size_t)c * frames_total + t0) * bins * eb;
      SG_TRY(launch_frames(e, pl, g, cfg, cfg.output, lut, o, st));
    }
    return SG_OK;
  }
  {
    bool fused = false;
    char* o = (char*)out_dev + (size_t)t0 * bins * eb;
    SG_TRY(launch_fused_smoothing(e, pl, cfg, pcm_dev, n_clips, clip_len, clip_stride, start0, nframes, frames_total, o, state,
                                  lut, st, &fused));
    if (fused) return SG_OK;
  }
  // tau > 0 on a shape without a fused kernel: frame kernel -> linear magnitudes (scratch) -> recurrence kernel, in
  // tiles of whole clips, or frame ranges of one clip chained through `state`.  Tiles small enough to keep the
  // magnitudes in L2 between the two kernels were measured and lose: 64 x 60 s clips at n_fft 2048 take 2.54 ms with
  // 56 MB tiles (64 launches), 2.09 ms with 160 MB, 1.63 ms with one 1.4 GB tile (tools/tau_tile_sweep.py) -- a tile
  // has to fill the GPU several times over before the launch gaps and the pipeline fill stop showing.  So the tile is
  // bounded by memory only (SG_TAU_TILE_MB overrides it for the sweep).
  static const size_t kTileBytes = [] { const char* v = getenv("SG_TAU_TILE_MB"); return (size_t)(v ? atoi(v) : 1024) << 20; }();
  const size_t frame_bytes = (size_t)bins * sizeof(float);
  const sg::Epilogue ep = make_epilogue(cfg, 2.0 * cfg.n_fft, lut);
  const long long tile_frames = std::max<long long>(1, (long long)(kTileBytes / frame_bytes));
  if (nframes <= tile_frames && nframes == frames_total) {
    const long long group = std::max<long long>(1, std::min<long long>(n_clips, tile_frames / nframes));
    SG_TRY(e->scratch_mag.reserve((size_t)group * nframes * frame_bytes));
    for (long long c0 = 0; c0 < n_clips; c0 += group) {
      const long long nc = std::min(group, n_clips - c0);
      sg::FrameGeom g{pcm_dev + c0 * clip_stride, clip_len, clip_stride, nframes, nc * nframes, start0, cfg.n_fft, cfg.hop};
      const uint8_t* poison;
      SG_TRY(launch_poison(e, g, st, &poison));
      SG_TRY(launch_frames(e, pl, g, cfg, SG_OUT_F32_MAG, lut, e->scratch_mag.p, st));
      char* o = (char*)out_dev + (size_t)c0 * frames_total * bins * eb;
      SG_TRY(launch_smooth(e, cfg.output, (const float*)e->scratch_mag.p, o, state + c0 * bins, nc, nframes, bins,
                           cfg.smoothing, ep, poison, st));
    }
    return SG_OK;
  }
  // long clips (or a frame range of several clips): clip by clip, frame tiles chained through the state
  SG_TRY(e->scratch_mag.reserve((size_t)std::min(nframes, tile_frames) * frame_bytes));
  for (long long c = 0; c < n_clips; ++c)
    for (long long tt = 0; tt < nframes; tt += tile_frames) {
      const long long nt = std::min(tile_frames, nframes - tt);
      sg::FrameGeom g{pcm_dev + c * clip_stride, clip_len, clip_stride, nt, nt, start0 + tt * cfg.hop, cfg.n_fft, cfg.hop};
      const uint8_t* poison;
      SG_TRY(launch_poison(e, g, st, &poison));
      SG_TRY(launch_frames(e, pl, g, cfg, SG_OUT_F32_MAG, lut, e->scratch_mag.p, st));
      char* o = (char*)out_dev + ((size_t)c * frames_total + t0 + tt) * bins * eb;
      SG_TRY(launch_smooth(e, cfg.output, (const float*)e->scratch_mag.p, o, state + c * bins, 1, nt, bins, cfg.smoothing,
                           ep, poison, st));
    }
  return SG_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// C ABI: library
// ------------------------------------------------------------------------------------------
extern "C" {

const char* sg_last_error(void) { return g_err.c_str(); }
int sg_version(void) { return SG_VERSION_MAJOR * 100 + SG_VERSION_MINOR; }

int sg_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int sg_stft_config_default(sg_stft_config* cfg) {
  if (!cfg) return fail(SG_ERR_INVALID_ARG, "cfg is null");
  cfg->n_fft = 2048; cfg->hop = 512; cfg->window = SG_WINDOW_BLACKMAN; cfg->output = SG_OUT_U8;
  cfg->align = SG_ALIGN_VALID; cfg->min_db = -100.f; cfg->max_db = -30.f; cfg->smoothing = 0.f;
  cfg->custom_window = nullptr; cfg->colormap = nullptr;
  return SG_OK;
}

int sg_colormap_reference(uint32_t lut[256]) {
  if (!lut) return fail(SG_ERR_INVALID_ARG, "lut is null");
  reference_lut(lut);
  return SG_OK;
}

int sg_stft_num_bins(const sg_stft_config* cfg) { return cfg ? cfg->n_fft / 2 : SG_ERR_INVALID_ARG; }
int64_t sg_stft_num_frames(const sg_stft_config* cfg, int64_t clip_len) {
  if (validate_cfg(cfg) != SG_OK) return -1;
  if (clip_len < 0) return -1;
  return frames_for(*cfg, clip_len);
}
int sg_stft_elem_bytes(const sg_stft_config* cfg) { return cfg ? (int)elem_bytes(cfg->output) : SG_ERR_INVALID_ARG; }

// ------------------------------------------------------------------------------------------
// engine
// ------------------------------------------------------------------------------------------
int sg_engine_create(int device, sg_engine** out) {
  if (!out) return fail(SG_ERR_INVALID_ARG, "out is null");
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(SG_ERR_NO_DEVICE, "no CUDA device visible (this engine has no CPU fallback)");
  }
  if (device < 0 || device >= n) return fail(SG_ERR_INVALID_ARG, "device index out of range");
  SG_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SG_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)     // the library holds sm_100a code only: sm_90 and sm_120 parts have no kernel image
    return fail(SG_ERR_NO_DEVICE, "device is not compute capability 10.x (sm_100a kernels only)");
  sg_engine* e = new sg_engine();
  e->device = device;
  e->sm_count = prop.multiProcessorCount;
  const int rc = [&]() -> int {
    SG_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    SG_CUDA(cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking));
    SG_CUDA(cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking));
    SG_CUDA(cudaEventCreateWithFlags(&e->ev_scratch, cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) {
      SG_CUDA(cudaEventCreateWithFlags(&e->ev_ring_in[i], cudaEventDisableTiming));
      SG_CUDA(cudaEventCreateWithFlags(&e->ev_ring_k[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; ++i) {
      SG_CUDA(cudaEventCreateWithFlags(&e->ev_pin_in[i], cudaEventDisableTiming));
      SG_CUDA(cudaEventCreateWithFlags(&e->ev_pin_out[i], cudaEventDisableTiming));
    }
    uint32_t lut[256];
    reference_lut(lut);
    SG_CUDA(cudaMalloc((void**)&e->lut_ref, sizeof(lut)));
    SG_CUDA(cudaMemcpy(e->lut_ref, lut, sizeof(lut), cudaMemcpyHostToDevice));
#ifdef SG_DEBUG
    {
      const size_t words = (size_t)e->sm_count * (sg::kDbgMaxWarps * sg::kDbgWarpSlots + sg::kDbgCtaSlots);
      SG_CUDA(cudaMalloc((void**)&e->dbg.tags, words * sizeof(unsigned)));
      SG_CUDA(cudaMemset(e->dbg.tags, 0, words * sizeof(unsigned)));
      SG_CUDA(cudaMalloc((void**)&e->dbg.counts, sg::kDbgSites * sizeof(unsigned long long)));
      SG_CUDA(cudaMemset(e->dbg.counts, 0, sg::kDbgSites * sizeof(unsigned long long)));
      e->dbg.ctas = e->sm_count;
      const char* brk = getenv("SG_DEBUG_BREAK_CHAIN");
      e->dbg.break_chain = brk && brk[0] == '1';
      SG_CUDA((cudaError_t)sg::dbg_attach_w32x2p(e->dbg));
      SG_CUDA((cudaError_t)sg::dbg_attach_w32x2s(e->dbg));
      SG_CUDA((cudaError_t)sg::dbg_attach_w32eo_s(e->dbg));
      SG_CUDA((cudaError_t)sg::dbg_attach_psmooth_l2(e->dbg));
      SG_CUDA((cudaError_t)sg::dbg_attach_psmooth_l3(e->dbg));
      SG_CUDA((cudaError_t)sg::dbg_attach_psmooth_l4(e->dbg));
    }
#endif
    return SG_OK;
  }();
  if (rc != SG_OK) {          // nothing half-built is left behind
    const std::string why = g_err;
    sg_engine_destroy(e);
    return fail(rc, why);
  }
  *out = e;
  return SG_OK;
}

int sg_engine_destroy(sg_engine* e) {
  if (!e) return SG_OK;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (auto& kv : e->plans) kv.second.release();
  cudaFree(e->lut_ref);
  e->lut_user.release(); e->scratch_mag.release(); e->scratch_state.release(); e->scratch_carry.release(); e->scratch_poison.release(); e->xs_carry.release(); e->xs_flags.release(); e->xs_state.release(); e->d_in.release(); e->d_out.release();
  e->d_raw[0].release(); e->d_raw[1].release();
  for (auto& kv : e->rs_tables) kv.second.taps.release();
  e->bq_start.release(); e->bq_agg.release(); e->bq_io.release(); e->bq_state.release();
  for (int i = 0; i < 2; ++i) { e->pin_in[i].release(); e->pin_out[i].release(); }
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->s_h2d) cudaStreamDestroy(e->s_h2d);
  if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
  if (e->ev_scratch) cudaEventDestroy(e->ev_scratch);
  for (int i = 0; i < 4; ++i) { if (e->ev_ring_in[i]) cudaEventDestroy(e->ev_ring_in[i]); if (e->ev_ring_k[i]) cudaEventDestroy(e->ev_ring_k[i]); }
  for (int i = 0; i < 2; ++i) { if (e->ev_pin_in[i]) cudaEventDestroy(e->ev_pin_in[i]); if (e->ev_pin_out[i]) cudaEventDestroy(e->ev_pin_out[i]); }
  delete e;
  return SG_OK;
}

int sg_engine_device(const sg_engine* e) { return e ? e->device : SG_ERR_INVALID_ARG; }
int64_t sg_engine_launch_count(const sg_engine* e) { return e ? e->launches : 0; }
const char* sg_engine_last_kernel(const sg_engine* e) { return e ? e->last_kernel : "none"; }
int sg_engine_set_kernel_variant(sg_engine* e, int variant) {
  if (!e || variant < 0 || variant > 7 || variant == 5)
    return fail(SG_ERR_INVALID_ARG,
                "variant must be 0 (auto), 1 (generic smem), 2 (one frame per warp), 3 (register family), "
                "4 (TMA-staged pair kernel), 6 (pair kernel, 8 warps) or 7 (fused smoothing kernel at any clip count)");
  e->kernel_variant = variant;
  return SG_OK;
}
int sg_engine_synchronize(sg_engine* e) {
  if (!e) return fail(SG_ERR_INVALID_ARG, "engine is null");
  SG_CUDA(cudaSetDevice(e->device));
  SG_CUDA(cudaStreamSynchronize(e->stream));
  return SG_OK;
}

int sg_host_alloc(size_t bytes, void** out) {
  if (!out) return fail(SG_ERR_INVALID_ARG, "out is null");
  *out = nullptr;
  SG_CUDA(cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable));
  return SG_OK;
}
int sg_host_free(void* p) {
  if (p) SG_CUDA(cudaFreeHost(p));
  return SG_OK;
}

// ------------------------------------------------------------------------------------------
// batched path
// ------------------------------------------------------------------------------------------
int sg_stft_batch_device(sg_engine* e, const float* pcm_dev, int64_t n_clips, int64_t clip_len, int64_t clip_stride,
                         const sg_stft_config* cfg, void* out_dev, void* cuda_stream) {
  if (!e) return fail(SG_ERR_INVALID_ARG, "engine is null");
  SG_TRY(validate_cfg(cfg));
  if (n_clips < 0 || clip_len < 0 || clip_stride < clip_len) return fail(SG_ERR_INVALID_ARG, "bad clip geometry");
  if (n_clips == 0) return SG_OK;
  if (!pcm_dev || !out_dev) return fail(SG_ERR_INVALID_ARG, "null device buffer");
  if (((uintptr_t)pcm_dev & 15) || ((uintptr_t)out_dev & 15)) return fail(SG_ERR_INVALID_ARG, "device buffers must be 16-byte aligned");
  std::lock_guard<std::mutex> lock(e->mu);
  SG_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
  Plan* pl;
  SG_TRY(e->get_plan(*cfg, &pl));
  const long long frames = frames_for(*cfg, clip_len);
  if (frames == 0) return SG_OK;
  // the engine's scratch (smoothing state / magnitude tiles / carries, the custom colour table) is shared by all
  // streams: order this call after the previous user, whatever stream that was on
  const bool shared = cfg->smoothing != 0.f || (cfg->colormap && cfg->output == SG_OUT_RGBA8);
  if (shared) SG_TRY(e->scratch_acquire(st));
  const uint32_t* lut;
  SG_TRY(e->lut_for(*cfg, st, &lut));
  float* state = nullptr;
  if (cfg->smoothing != 0.f) {
    const size_t sb = (size_t)n_clips * (cfg->n_fft / 2) * sizeof(float);
    SG_TRY(e->scratch_state.reserve(sb));
    SG_CUDA(cudaMemsetAsync(e->scratch_state.p, 0, sb, st));
    state = (float*)e->scratch_state.p;
  }
  SG_TRY(run_range(e, *pl, *cfg, pcm_dev, n_clips, clip_len, clip_stride, 0, frames, frames, out_dev, state, lut, st));
  if (shared) SG_TRY(e->scratch_release(st));
  return SG_OK;
}

// Host buffers.  Work is cut into chunks (groups of whole clips, or frame ranges of one long clip);
// chunk i+1's host->device copy and chunk i-1's device->host copy overlap chunk i's kernels on three
// streams.  Pageable host memory is staged through the engine's pinned bounce buffers.
}  // extern "C"

namespace {
// Interleaved PCM in front of the pipeline (sg_stft_pcm): the raw bytes are what is copied to the device, an
// ingest kernel turns each chunk into float32 planes, and every plane is a clip for the frame kernels.
// With `rs` set the ingest kernel also resamples: clip_len counts output frames, in_frames the source's.
struct RawPcm {
  int format, channels, planes, bytes_per_frame;
  PcmMix mix;
  const RsTable* rs = nullptr;
  long long in_frames = 0;
};

long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// source frames [lo, hi) that outputs [k_lo, k_hi) of a clip of `frames` source frames read (nonzero taps only)
void resample_input_range(const RsTable& t, long long frames, long long k_lo, long long k_hi, long long* lo, long long* hi) {
  *lo = std::max(0LL, -floor_div(t.half - k_lo * t.down, t.up));   // ceil((k_lo*down - half)/up)
  *hi = std::min(frames, floor_div((k_hi - 1) * t.down + t.half, t.up) + 1);
  if (*hi < *lo) *hi = *lo;
}

// enqueues the fused ingest + resample kernel: outputs [k0, k0 + n_out) of every plane from source frames
// [in_f0, in_f0 + in_n) of every clip (clip c's first present frame at src + c*clip_bytes)
int resample_on_device(sg_engine* e, const RsTable& t, const void* src, long long src_bytes, long long clip_bytes, int64_t n_clips,
                       long long in_f0, long long in_n, const RawPcm& raw, long long k0, long long n_out, float* out,
                       long long out_stride, cudaStream_t st) {
  if (n_clips == 0 || n_out == 0) return SG_OK;
  RsGeom g;
  g.src = (const unsigned char*)src;
  g.src_bytes = src_bytes;
  g.clip_bytes = clip_bytes;
  g.in_f0 = in_f0;
  g.in_n = in_n;
  g.k0 = k0;
  g.n_out = n_out;
  g.out = out;
  g.out_stride = out_stride;
  g.taps = (const float*)t.taps.p;
  g.up = t.up; g.down = t.down; g.half = t.half; g.J = t.J;
  g.channels = raw.channels;
  g.planes = raw.planes;
  SG_CUDA((cudaError_t)launch_pcm_resample(raw.format, g, n_clips, raw.mix, st));
  e->launches++;
  return SG_OK;
}

int stft_batch_impl(sg_engine* e, const void* pcm, int64_t n_clips, int64_t clip_len, const sg_stft_config* cfg,
                    void* out, const RawPcm* raw) {
  if (!e) return fail(SG_ERR_INVALID_ARG, "engine is null");
  SG_TRY(validate_cfg(cfg));
  if (n_clips < 0 || clip_len < 0) return fail(SG_ERR_INVALID_ARG, "bad clip geometry");
  if (n_clips == 0) return SG_OK;
  if (!pcm || !out) return fail(SG_ERR_INVALID_ARG, "null host buffer");
  std::lock_guard<std::mutex> lock(e->mu);
  SG_CUDA(cudaSetDevice(e->device));
  Plan* pl;
  SG_TRY(e->get_plan(*cfg, &pl));
  SG_TRY(e->scratch_acquire(e->stream));     // an earlier sg_stft_batch_device call on another stream may still use it
  const uint32_t* lut;
  SG_TRY(e->lut_for(*cfg, e->stream, &lut));
  const long long frames = frames_for(*cfg, clip_len);
  if (frames == 0) return SG_OK;
  const int bins = cfg->n_fft / 2;
  const size_t eb = elem_bytes(cfg->output);
  const int planes = raw ? raw->planes : 1;               // device clips per source clip
  const RsTable* rs = raw ? raw->rs : nullptr;
  // source bytes per sample frame of the clip (with resampling: per output frame, rounded up)
  const size_t unit = rs ? ((size_t)raw->bytes_per_frame * rs->down + rs->up - 1) / rs->up
                         : raw ? (size_t)raw->bytes_per_frame : sizeof(float);
  const size_t out_bytes = (size_t)n_clips * planes * frames * bins * eb;
  // device-resident copies of the whole problem (clip_stride padded to 4 floats for 16-byte rows)
  const long long stride = (clip_len + 3) & ~3LL;
  SG_TRY(e->d_in.reserve((size_t)n_clips * planes * stride * sizeof(float)));
  SG_TRY(e->d_out.reserve(out_bytes));
  float* d_in = (float*)e->d_in.p;
  char* d_out = (char*)e->d_out.p;
  float* state = nullptr;
  if (cfg->smoothing != 0.f) {
    const size_t sb = (size_t)n_clips * planes * bins * sizeof(float);
    SG_TRY(e->scratch_state.reserve(sb));
    SG_CUDA(cudaMemsetAsync(e->scratch_state.p, 0, sb, e->stream));
    state = (float*)e->scratch_state.p;
  }
  const bool in_pinned = is_pinned(pcm), out_pinned = is_pinned(out);
  // target bytes per chunk, whichever side (input or output) is larger: at small hops a frame's output dwarfs its hop
  static const size_t kChunkEnv = [] { const char* v = getenv("SG_CHUNK_MB"); return (size_t)(v ? atoi(v) : 0) << 20; }();
  const size_t kChunk = kChunkEnv ? kChunkEnv : (size_t)32 << 20;
  struct Chunk { long long c0, nc, t0, nt; };
  std::vector<Chunk> chunks;
  const size_t clip_bytes = rs ? (size_t)raw->in_frames * raw->bytes_per_frame : (size_t)clip_len * unit;
  const size_t clip_out_bytes = (size_t)planes * frames * bins * eb;
  if (std::max(clip_bytes, clip_out_bytes) <= kChunk) {
    const long long per = std::max<long long>(1, (long long)(kChunk / std::max<size_t>(std::max(clip_bytes, clip_out_bytes), 1)));
    for (long long c = 0; c < n_clips; c += per) chunks.push_back({c, std::min(per, n_clips - c), 0, frames});
  } else {
    const long long per = std::max<long long>(1, (long long)(kChunk / std::max((size_t)cfg->hop * unit, (size_t)planes * bins * eb)));
    for (long long c = 0; c < n_clips; ++c)
      for (long long t = 0; t < frames; t += per) chunks.push_back({c, 1, t, std::min(per, frames - t)});
  }
  const long long start_base = cfg->align == SG_ALIGN_VALID ? 0 : (long long)cfg->hop - cfg->n_fft;
  // events of the pipeline: the engine's own (created once), chunk i uses slot i & 3
  cudaEvent_t* const ev_in = e->ev_ring_in;
  cudaEvent_t* const ev_k = e->ev_ring_k;
  cudaEvent_t* const ev_pin_in = e->ev_pin_in;
  cudaEvent_t* const ev_pin_out = e->ev_pin_out;
  bool pin_in_used[2] = {false, false};
  // a chunk's output is `rows` runs of `width` bytes, `pitch` apart (one run, or one per plane for a frame range)
  struct Pending { char* dst; size_t width, pitch; int rows; bool live; } pend[2] = {{nullptr, 0, 0, 0, false}, {nullptr, 0, 0, 0, false}};
  int rc = SG_OK;
  auto drain_out = [&](int slot) -> int {  // copy a finished pinned output bounce to the caller
    if (!pend[slot].live) return SG_OK;
    SG_CUDA(cudaEventSynchronize(ev_pin_out[slot]));
    for (int r = 0; r < pend[slot].rows; ++r)
      std::memcpy(pend[slot].dst + r * pend[slot].pitch, (char*)e->pin_out[slot].p + r * pend[slot].width, pend[slot].width);
    pend[slot].live = false;
    return SG_OK;
  };
  auto body = [&]() -> int {
    long long uploaded_to = 0;  // per-clip sample watermark for frame-range chunks
    long long uploaded_clip = -1;
    for (size_t i = 0; i < chunks.size(); ++i) {
      const Chunk& ch = chunks[i];
      const int slot = (int)(i & 1);
      // ---- host -> device
      long long s_lo, s_hi;  // sample range of each clip in this chunk
      if (ch.nt == frames) { s_lo = 0; s_hi = clip_len; }
      else {
        if (uploaded_clip != ch.c0) { uploaded_clip = ch.c0; uploaded_to = 0; }
        s_lo = uploaded_to;
        s_hi = std::min<long long>(clip_len, std::max<long long>(s_lo, start_base + (ch.t0 + ch.nt - 1) * cfg->hop + cfg->n_fft));
        uploaded_to = s_hi;
      }
      long long in_lo = s_lo, in_hi = s_hi;  // source frames uploaded (differ from s_lo, s_hi when resampling)
      if (rs) {
        if (ch.nt == frames) { in_lo = 0; in_hi = raw->in_frames; }
        else resample_input_range(*rs, raw->in_frames, s_lo, s_hi, &in_lo, &in_hi);
      }
      const size_t row = rs ? (size_t)(in_hi - in_lo) * raw->bytes_per_frame : (size_t)(s_hi - s_lo) * unit;
      if (row > 0) {
        const char* src = (const char*)pcm + (size_t)ch.c0 * clip_bytes + (size_t)in_lo * (rs ? raw->bytes_per_frame : unit);
        char* dst = (char*)(d_in + ch.c0 * stride + s_lo);   // float32 source: straight into the clip rows
        size_t dpitch = (size_t)stride * sizeof(float);
        if (raw) {                                            // raw PCM: dense rows in this slot's byte buffer
          SG_TRY(e->d_raw[slot].reserve(row * ch.nc + 32));
          if (i >= 2) SG_CUDA(cudaStreamWaitEvent(e->s_h2d, ev_k[(i - 2) & 3], 0));   // its last reader has finished
          dst = (char*)e->d_raw[slot].p;
          dpitch = row;
        }
        if (!in_pinned) {
          SG_TRY(e->pin_in[slot].reserve(row * ch.nc));
          if (pin_in_used[slot]) SG_CUDA(cudaEventSynchronize(ev_pin_in[slot]));   // previous use of this bounce has been copied
          for (long long c = 0; c < ch.nc; ++c)
            std::memcpy((char*)e->pin_in[slot].p + c * row, src + c * clip_bytes, row);
          // (one clip per chunk: a plain copy -- a 2-D copy's pitch is limited to 2^31 - 1 bytes)
          if (ch.nc == 1) SG_CUDA(cudaMemcpyAsync(dst, e->pin_in[slot].p, row, cudaMemcpyHostToDevice, e->s_h2d));
          else SG_CUDA(cudaMemcpy2DAsync(dst, dpitch, e->pin_in[slot].p, row, row, ch.nc, cudaMemcpyHostToDevice, e->s_h2d));
          SG_CUDA(cudaEventRecord(ev_pin_in[slot], e->s_h2d));
          pin_in_used[slot] = true;
        } else {
          if (ch.nc == 1) SG_CUDA(cudaMemcpyAsync(dst, src, row, cudaMemcpyHostToDevice, e->s_h2d));
          else SG_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, clip_bytes, row, ch.nc, cudaMemcpyHostToDevice, e->s_h2d));
        }
      }
      SG_CUDA(cudaEventRecord(ev_in[i & 3], e->s_h2d));
      // ---- kernels
      SG_CUDA(cudaStreamWaitEvent(e->stream, ev_in[i & 3], 0));
      if (rs && s_hi > s_lo) {
        SG_TRY(resample_on_device(e, *rs, e->d_raw[slot].p, (long long)(row * ch.nc), (long long)row, ch.nc, in_lo, in_hi - in_lo,
                                  *raw, s_lo, s_hi - s_lo, d_in + ch.c0 * planes * stride + s_lo, stride, e->stream));
      } else if (raw && row > 0) {
        PcmGeom pg;
        pg.src = (const unsigned char*)e->d_raw[slot].p;
        pg.src_bytes = (long long)(row * ch.nc);
        pg.clip_bytes = (long long)row;
        pg.frames = s_hi - s_lo;
        pg.out = d_in + ch.c0 * planes * stride + s_lo;
        pg.out_stride = stride;
        pg.tile_frames = pcm_tile_frames(raw->bytes_per_frame);
        pg.tiles_per_clip = (pg.frames + pg.tile_frames - 1) / pg.tile_frames;
        pg.channels = raw->channels;
        pg.planes = planes;
        SG_CUDA((cudaError_t)launch_pcm_ingest(raw->format, pg, ch.nc, raw->mix, e->stream));
        e->launches++;
      }
      SG_TRY(run_range(e, *pl, *cfg, d_in + ch.c0 * planes * stride, ch.nc * planes, clip_len, stride, ch.t0, ch.nt, frames,
                       d_out + (size_t)ch.c0 * planes * frames * bins * eb, state ? state + ch.c0 * planes * bins : nullptr,
                       lut, e->stream));
      SG_CUDA(cudaEventRecord(ev_k[i & 3], e->stream));
      // ---- device -> host
      SG_CUDA(cudaStreamWaitEvent(e->s_d2h, ev_k[i & 3], 0));
      const size_t off = ((size_t)ch.c0 * planes * frames + ch.t0) * bins * eb;
      const bool whole = ch.nt == frames;
      const size_t width = (whole ? (size_t)ch.nc * planes * frames : (size_t)ch.nt) * bins * eb;
      const int rows = whole ? 1 : planes;
      const size_t pitch = (size_t)frames * bins * eb;
      if (!out_pinned) {
        SG_TRY(drain_out(slot));
        SG_TRY(e->pin_out[slot].reserve(width * rows));
        if (rows == 1) SG_CUDA(cudaMemcpyAsync(e->pin_out[slot].p, d_out + off, width, cudaMemcpyDeviceToHost, e->s_d2h));
        else SG_CUDA(cudaMemcpy2DAsync(e->pin_out[slot].p, width, d_out + off, pitch, width, rows, cudaMemcpyDeviceToHost, e->s_d2h));
        SG_CUDA(cudaEventRecord(ev_pin_out[slot], e->s_d2h));
        pend[slot] = {(char*)out + off, width, pitch, rows, true};
      } else {
        if (rows == 1) SG_CUDA(cudaMemcpyAsync((char*)out + off, d_out + off, width, cudaMemcpyDeviceToHost, e->s_d2h));
        else SG_CUDA(cudaMemcpy2DAsync((char*)out + off, pitch, d_out + off, pitch, width, rows, cudaMemcpyDeviceToHost, e->s_d2h));
      }
    }
    SG_TRY(drain_out(0));
    SG_TRY(drain_out(1));
    SG_CUDA(cudaStreamSynchronize(e->s_d2h));
    SG_CUDA(cudaStreamSynchronize(e->stream));
    return SG_OK;
  };
  rc = body();
  if (rc != SG_OK) cudaDeviceSynchronize();
  return rc;
}
}  // namespace

#ifdef SG_DEBUG
// debug build only (not part of include/sgcore.h): mismatches per check site -- 0 exchange planes of the frame-pair
// kernel, 1 its byte stage, 2 the state hand-off of the fused smoothing kernel (n_fft 2048), 3 the same of the part-warp
// kernels (n_fft 1024 / 512 / 256), 4 of the n_fft 4096 kernel -- and, in the last entry, how many
// warp iterations ran with the checks armed
extern "C" int sg_debug_counts(sg_engine* e, unsigned long long out[16]) {
  if (!e || !out) return fail(SG_ERR_INVALID_ARG, "null argument");
  SG_CUDA(cudaSetDevice(e->device));
  SG_CUDA(cudaDeviceSynchronize());
  SG_CUDA(cudaMemcpy(out, e->dbg.counts, sg::kDbgSites * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return SG_OK;
}
#endif

extern "C" {
int sg_stft_batch(sg_engine* e, const float* pcm, int64_t n_clips, int64_t clip_len, const sg_stft_config* cfg,
                  void* out) {
  return stft_batch_impl(e, pcm, n_clips, clip_len, cfg, out, nullptr);
}

// Clips sharded over several engines (one per GPU; SURVEY 8(e)): engine s takes the contiguous block
// [n_clips*s/G, n_clips*(s+1)/G), one host thread per engine runs the three-stream pipeline of sg_stft_batch on its
// block, and every block's results land in its own slice of the caller's `out` -- that host copy is the gather; the
// shards exchange nothing.  Bit-identical to one engine processing all clips.
int sg_stft_batch_multi(sg_engine* const* engines, int n_engines, const float* pcm, int64_t n_clips, int64_t clip_len,
                        const sg_stft_config* cfg, void* out) {
  if (!engines || n_engines < 1) return fail(SG_ERR_INVALID_ARG, "need at least one engine");
  for (int s = 0; s < n_engines; ++s) {
    if (!engines[s]) return fail(SG_ERR_INVALID_ARG, "null engine");
    for (int t = 0; t < s; ++t)
      if (engines[t] == engines[s]) return fail(SG_ERR_INVALID_ARG, "the same engine listed twice");
  }
  SG_TRY(validate_cfg(cfg));
  if (n_clips < 0 || clip_len < 0) return fail(SG_ERR_INVALID_ARG, "bad clip geometry");
  if (n_clips == 0) return SG_OK;
  if (!pcm || !out) return fail(SG_ERR_INVALID_ARG, "null host buffer");
  if (n_engines == 1) return stft_batch_impl(engines[0], pcm, n_clips, clip_len, cfg, out, nullptr);
  const size_t out_clip = (size_t)frames_for(*cfg, clip_len) * (size_t)(cfg->n_fft / 2) * elem_bytes(cfg->output);
  std::vector<int> rc((size_t)n_engines, SG_OK);
  std::vector<std::string> msg((size_t)n_engines);
  std::vector<std::thread> workers;
  for (int s = 0; s < n_engines; ++s) {
    const int64_t lo = n_clips * s / n_engines, hi = n_clips * (s + 1) / n_engines;
    if (hi <= lo) continue;
    workers.emplace_back([=, &rc, &msg] {
      rc[(size_t)s] = stft_batch_impl(engines[s], pcm + (size_t)lo * (size_t)clip_len, hi - lo, clip_len, cfg,
                                      (char*)out + (size_t)lo * out_clip, nullptr);
      if (rc[(size_t)s] != SG_OK) msg[(size_t)s] = g_err;      // g_err is thread local: carry it to the caller's thread
    });
  }
  for (auto& w : workers) w.join();
  for (int s = 0; s < n_engines; ++s)
    if (rc[(size_t)s] != SG_OK) return fail(rc[(size_t)s], "engine " + std::to_string(s) + ": " + msg[(size_t)s]);
  return SG_OK;
}
}  // extern "C"

#include "sg_biquad.inl"
#include "sg_objects.inl"
#include "sg_pcm.inl"
