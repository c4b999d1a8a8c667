// Translation unit: register-pipelined frame-pair kernel (n_fft 2048, hop 512).
#include "kernel_w32x2p.cuh"

namespace sg {

template <int OUT, int NW, int HOPJ>
static int launch_xp(const FrameGeom& g, const W32Plan& p, const Epilogue& ep, void* out, int sm_count, int device,
                     cudaStream_t st) {
  using T = typename OutElem<OUT>::type;
  constexpr int smem = XpShape<NW>::kSmemBytes;
  const cudaError_t rc = ensure_dynamic_smem<stft_w32x2p_kernel<OUT, NW, HOPJ>>(smem, device);
  if (rc != cudaSuccess) return (int)rc;
  const long long pairs = (g.total_frames + 1) / 2;
  const int grid = (int)std::min<long long>((pairs + NW - 1) / NW, sm_count);
  stft_w32x2p_kernel<OUT, NW, HOPJ><<<grid, NW * 32, smem, st>>>(g, p, ep, (T*)out);
  return (int)cudaGetLastError();
}

int launch_w32x2p(int out_kind, int warps, const FrameGeom& g, const W32Plan& p, const Epilogue& ep, void* out,
                  int sm_count, int device, cudaStream_t st) {
  return dispatch_out(out_kind, [&](auto tag) {
    constexpr int OUT = decltype(tag)::value;
    if (g.hop == 256) return launch_xp<OUT, 12, 4>(g, p, ep, out, sm_count, device, st);
    if (warps == 12) return launch_xp<OUT, 12, 8>(g, p, ep, out, sm_count, device, st);
    return launch_xp<OUT, 8, 8>(g, p, ep, out, sm_count, device, st);
  });
}

#ifdef SG_DEBUG
int dbg_attach_w32x2p(const DbgState& st) { return (int)dbg_attach(st); }
#endif

}  // namespace sg
