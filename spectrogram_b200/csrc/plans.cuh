// Device-side plan tables (built once per (n_fft, window) on the host, sgcore.cu build_plan) and the
// host-callable launchers of each kernel family.  Every family lives in its own translation unit
// (tu_*.cu) so a change to one kernel rebuilds only that unit.
#pragma once
#include "common.cuh"

namespace sg {

constexpr int kW32N = 2048;   // the reference's fftSize (UI/player.js:10): the size with dedicated kernels
constexpr int kW32M = 1024;

struct W32Plan {        // n_fft == 2048 kernels
  const float* win;    // [2048]
  const float2* tw2;   // [31][32]: stage u (1..5), p < 2^(u-1): W_{32*2^u}^{32 p + lane}
  const float2* ut;    // [16][32]: W_2048^{lane + 32 i}
};

struct WregPlan {       // register family, n_fft = 256 ... 8192
  const float* win;    // [n_fft]
  const float2* tw2;   // [31][32]  W_{32*2^u}^{32 p + k_a}, row (2^(u-1) - 1 + p)      (any M)
  const float2* tw3;   // [32][2^R3 - 1][32]  W_{1024*2^u}^{1024 p + 32 q + k_a}        (M = 2048, 4096)
  const float2* ut;    // [M/2 + 1] W_n^k
};

struct R400Plan {       // n_fft == 400 kernel (M = 200 = 40 x 5)
  const float* win;    // [400]
  const float2* tw;    // [5][41]  W_200^{b k1}, row stride 41
  const float2* ut;    // [200]    W_400^k
};

struct W16Plan {        // n_fft == 512 kernel (M = 256 = 16 x 16)
  const float* win;    // [512]
  const float2* tw;    // [15][16]  row (h - 1 + p), h = 1, 2, 4, 8: W_{32 h}^{16 p + col}
  const float2* ut;    // [129]     W_512^k
};

struct PairPlan {       // frame-pair kernels for n_fft 1024 (L = 16) and 512 (L = 8), M = 32 x L
  const float* win;    // [n_fft], padded to 2 n_fft readable floats (idle prefetches park here)
  const float2* twb;   // [log2 L][32]  W_{32*2^u}^col, u = 1..log2 L
  const float2* ut;    // [M/2 + 1]     W_n^k
};

struct SmemPlan {       // generic mixed-radix kernel
  const float* win;    // [n_fft]
  const float2* tw;    // [m]      W_m^k
  const float2* ut;    // [m/2+1]  W_n^k
  const int* pos;      // [m]      position of Z[k] after the in-place DIF (digit reversal)
  int m;               // n_fft/2
  int nstage;
  int radix[16];
};

// Launchers: enqueue on `st`, return the cudaError_t of the launch (0 = ok).  `out_kind` is kOut*.
int launch_w32x2p(int out_kind, int warps, const FrameGeom& g, const W32Plan& p, const Epilogue& ep, void* out,
                  int sm_count, int device, cudaStream_t st);
struct XsGeom;   // kernel_w32x2s.cuh
// grid = CTAs to launch (<= sm_count: the chained tasks and the look-back need every CTA resident)
int launch_w32x2s(int out_kind, const FrameGeom& g, const XsGeom& x, const W32Plan& p, const Epilogue& ep, void* out,
                  int grid, int device, cudaStream_t st);
int launch_w32x2(int out_kind, const FrameGeom& g, const W32Plan& p, const Epilogue& ep, void* out, int sm_count,
                 int device, cudaStream_t st);
int launch_w32(int out_kind, const FrameGeom& g, const W32Plan& p, const Epilogue& ep, void* out, int sm_count,
               int device, cudaStream_t st);
int launch_wreg(int out_kind, int log2m, const FrameGeom& g, const WregPlan& p, const Epilogue& ep, void* out,
                int sm_count, int device, cudaStream_t st);
int launch_r400(int out_kind, const FrameGeom& g, const R400Plan& p, const Epilogue& ep, void* out, int sm_count,
                int device, cudaStream_t st);
int launch_w16(int out_kind, const FrameGeom& g, const W16Plan& p, const Epilogue& ep, void* out, int sm_count,
               int device, cudaStream_t st);
int launch_w16x8(int out_kind, const FrameGeom& g, const W16Plan& p, const Epilogue& ep, void* out, int sm_count,
                 int device, cudaStream_t st);   // n_fft 256; W16Plan.tw holds 7 rows
// part-warp frame-pair kernels (tu_pair.cu, one object per lane-group size): return -1 when the hop has no
// instantiation (hop must be 2*L*{4, 8, 16} samples, plus hop 160 for n_fft 1024 and 512)
int launch_pair_l4(int out_kind, const FrameGeom& g, const PairPlan& p, const Epilogue& ep, void* out, int sm_count,
                   int device, cudaStream_t st);   // n_fft 1024
int launch_pair_l3(int out_kind, const FrameGeom& g, const PairPlan& p, const Epilogue& ep, void* out, int sm_count,
                   int device, cudaStream_t st);   // n_fft 512
int launch_pair_l2(int out_kind, const FrameGeom& g, const PairPlan& p, const Epilogue& ep, void* out, int sm_count,
                   int device, cudaStream_t st);
// tau > 0 fused into the part-warp pair kernels (tu_psmooth.cu); XsGeom: kernel_w32x2s.cuh.  -1: no instantiation for the hop
int launch_pair_s_l4(int out_kind, const FrameGeom& g, const XsGeom& x, const PairPlan& p, const Epilogue& ep, void* out,
                     int grid, int device, cudaStream_t st);
int launch_pair_s_l3(int out_kind, const FrameGeom& g, const XsGeom& x, const PairPlan& p, const Epilogue& ep, void* out,
                     int grid, int device, cudaStream_t st);
int launch_pair_s_l2(int out_kind, const FrameGeom& g, const XsGeom& x, const PairPlan& p, const Epilogue& ep, void* out,
                     int grid, int device, cudaStream_t st);   // n_fft 256
inline bool pair_kernel_serves(int n_fft, int hop) {
  const int l = n_fft == 1024 ? 16 : n_fft == 512 ? 8 : n_fft == 256 ? 4 : 0;
  if (!l || hop % (2 * l)) return false;
  const int j = hop / (2 * l);
  // (n_fft 256 at hop 128 is faster on the 16 x 8 kernel: 3364 M vs 2812 M frames/s)
  return j == 4 || j == 8 || (j == 16 && l != 4) || (l == 16 && j == 5) || (l == 8 && j == 10);
}
int launch_smem(int out_kind, const FrameGeom& g, const SmemPlan& p, const Epilogue& ep, void* out, int sm_count,
                int device, cudaStream_t st);

// tu_wreg.cu is compiled once per output kind
int launch_wreg_out0(int log2m, const FrameGeom&, const WregPlan&, const Epilogue&, void*, int, int, cudaStream_t);
int launch_wreg_out1(int log2m, const FrameGeom&, const WregPlan&, const Epilogue&, void*, int, int, cudaStream_t);
int launch_wreg_out2(int log2m, const FrameGeom&, const WregPlan&, const Epilogue&, void*, int, int, cudaStream_t);
int launch_wreg_out3(int log2m, const FrameGeom&, const WregPlan&, const Epilogue&, void*, int, int, cudaStream_t);

// tu_w32eo.cu: n_fft 4096 (kernel_w32eo.cuh)
constexpr int kEoN = 4096;
struct EoPlan {
  const float* win;     // [4096]
  const float2* tw2;    // [31][32] pass-2 twiddles of the 1024-point transform (rows 2^u - 1 are the bases)
  const float2* tab;    // [32] W_2048^lane, then [16][32] W_4096^{lane + 32 i}
};
int launch_w32eo(int out_kind, int warps, const FrameGeom& g, const EoPlan& p, const Epilogue& ep, void* out, int sm_count,
                 int device, cudaStream_t st);
// tau > 0 fused into the n_fft 4096 kernel (tu_w32eo_s.cu); XsGeom: kernel_w32x2s.cuh
int launch_w32eo_s(int out_kind, const FrameGeom& g, const XsGeom& x, const EoPlan& p, const Epilogue& ep, void* out, int grid,
                   int device, cudaStream_t st);
// tau > 0 fused into the register family (tu_regsmooth.cu): log2m 12 (n_fft 8192) or 11 (n_fft 4096)
int launch_wreg_s(int out_kind, int log2m, const FrameGeom& g, const XsGeom& x, const WregPlan& p, const Epilogue& ep, void* out,
                  int grid, int device, cudaStream_t st);

// tu_pcm.cu: PCM ingestion (kernel_pcm.cuh)
struct PcmGeom;
struct PcmMix;
int pcm_tile_frames(int bytes_per_frame);
int launch_pcm_ingest(int format, const PcmGeom& g, long long n_clips, const PcmMix& m, cudaStream_t st);
// tu_resample.cu: PCM ingestion + polyphase resampling (kernel_resample.cuh); tile_out and tiles are set by the launcher
struct RsGeom;
int launch_pcm_resample(int format, RsGeom g, long long n_clips, const PcmMix& m, cudaStream_t st);
// tu_biquad.cu: biquad filter (kernel_biquad.cuh)
struct BqArgs;
int launch_biquad(const BqArgs& a, cudaStream_t st, int* launches);

#ifdef SG_DEBUG
int dbg_attach_w32x2p(const DbgState& st);
int dbg_attach_w32x2s(const DbgState& st);
int dbg_attach_w32eo_s(const DbgState& st);
int dbg_attach_psmooth_l2(const DbgState& st);
int dbg_attach_psmooth_l3(const DbgState& st);
int dbg_attach_psmooth_l4(const DbgState& st);
#endif

constexpr int kMaxDevices = 64;

// one cudaFuncSetAttribute(MaxDynamicSharedMemorySize) per kernel per device
template <auto Kern>
inline cudaError_t ensure_dynamic_smem(int bytes, int device) {
  static int granted[kMaxDevices] = {};
  const int d = (device >= 0 && device < kMaxDevices) ? device : 0;
  if (granted[d] >= bytes) return cudaSuccess;
  const cudaError_t rc = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (rc == cudaSuccess) granted[d] = bytes;
  return rc;
}

// dispatch a functor template on the output kind
template <class F>
inline int dispatch_out(int out_kind, F&& f) {
  switch (out_kind) {
    case kOutU8: return f(std::integral_constant<int, kOutU8>{});
    case kOutF32Db: return f(std::integral_constant<int, kOutF32Db>{});
    case kOutRgba8: return f(std::integral_constant<int, kOutRgba8>{});
    default: return f(std::integral_constant<int, kOutF32Mag>{});
  }
}

}  // namespace sg
