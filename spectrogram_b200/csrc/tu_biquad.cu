// Translation unit: biquad filter (kernel_biquad.cuh).
#include "kernel_biquad.cuh"
#include "plans.cuh"

namespace sg {

// Launch (2): one CTA per channel turns the tile aggregates into every tile's start state, S_(k+1) = M^T S_k + agg_k
// (T = kBqTile), S_0 = the channel's state.  Thread t folds tiles [t c, (t+1) c) (c = carry_per) into its block's end
// state (thread 0 from S_0, the others from zero); an inclusive scan with the host's powers M^(T c 2^k) turns those
// into every block's true end state; each thread then walks its block again from the previous block's end.
__global__ void __launch_bounds__(kBqThreads) biquad_carry_kernel(const BqArgs a) {
  __shared__ BqVec s_v[kBqThreads];
  const int tid = threadIdx.x;
  const long long ch = blockIdx.x, m = a.tiles - 1, c = a.carry_per;
  const long long k0 = min(m, tid * c), k1 = min(m, k0 + c);
  const BqMat mt = a.pw[kBqPowers - 1];
  const BqVec* __restrict__ agg = a.agg + ch * a.tiles;
  double* __restrict__ start = a.start + ch * a.tiles * 4;
  double s0[4] = {0.0, 0.0, 0.0, 0.0};   // {x1, x2, y1, y2}
  if (a.state)
    for (int i = 0; i < 4; ++i) s0[i] = a.state[ch * 4 + i];
  BqVec v = tid == 0 ? BqVec{s0[2], s0[3], 0.0, 0.0} : BqVec{0.0, 0.0, 0.0, 0.0};
  for (long long k = k0; k < k1; ++k) v = bq_apply(mt, v, agg[k]);
  for (int d = 0; (1 << d) < kBqThreads; ++d) {   // a block past the last tile only carries (identity): its end is
    s_v[tid] = v;                                  // M^(T c) times the previous one, unused
    __syncthreads();
    if (tid >= (1 << d)) v = bq_apply(a.carry[d], s_v[tid - (1 << d)], v);
    __syncthreads();
  }
  s_v[tid] = v;
  __syncthreads();
  BqVec s = tid == 0 ? BqVec{s0[2], s0[3], 0.0, 0.0} : s_v[tid - 1];
  if (tid == 0) { start[0] = s0[2]; start[1] = s0[3]; start[2] = s0[0]; start[3] = s0[1]; }
  for (long long k = k0; k < k1; ++k) {
    s = bq_apply(mt, s, agg[k]);
    start[(k + 1) * 4] = s.x;
    start[(k + 1) * 4 + 1] = s.y;
  }
}

// One launch when every channel fits one tile, else three (kernel_biquad.cuh); *launches counts them.  The shape
// depends on (channels, len) alone.
int launch_biquad(const BqArgs& a, cudaStream_t st, int* launches) {
  *launches = 0;
  if (a.channels <= 0 || a.len <= 0) return 0;
  if (a.channels * a.tiles > 0x7fffffffLL) return (int)cudaErrorInvalidConfiguration;
  if (a.tiles > 1) {
    biquad_tile_kernel<false><<<(unsigned)(a.channels * (a.tiles - 1)), kBqThreads, 0, st>>>(a);
    biquad_carry_kernel<<<(unsigned)a.channels, kBqThreads, 0, st>>>(a);
    *launches += 2;
  }
  biquad_tile_kernel<true><<<(unsigned)(a.channels * a.tiles), kBqThreads, 0, st>>>(a);
  *launches += 1;
  return (int)cudaGetLastError();
}

}  // namespace sg
