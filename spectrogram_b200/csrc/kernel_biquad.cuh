// Biquad filter (W3C BiquadFilterNode, include/sgcore.h "biquad filter"): direct form I in float64, run along the
// time axis in parallel.
//
// The recurrence y[n] = u[n] - a1 y[n-1] - a2 y[n-2], u[n] = b0 x[n] + b1 x[n-1] + b2 x[n-2], is linear in the state
// s = (y[n-1], y[n-2]): a run of R samples maps its start state s to M^R s + v, where M = [[-a1, -a2], [1, 0]] and v is
// the run's end state from s = 0.  A channel is cut into tiles of kBqTile samples, one CTA each; a tile into runs of
// kBqRun samples, one thread each, held in registers.
//   tile kernel   each thread runs its run from zero (the tile's first run from the tile's true start state when it is
//                 known), a warp scan and a cross-warp pass combine the run end states with host-computed powers
//                 M^(R 2^k), so every thread learns its run's true start state and runs it again, writing y.
//   Precision: for poles near z = 1, M is far from normal (|M^n| reaches 1/theta, about 880 for an allpass at 10 Hz),
//   the zero-start states the scans combine are ~100 times the true ones, and a rounding error left in a state is
//   amplified by up to 1/theta downstream.  Plain double combinations miss the contract there by 10x (errors ~1e-8).
//   So every combination (warp scan, cross-warp pass, run starts, tile aggregates, carry scan) is double-double:
//   states as hi + lo, powers as hi + lo, products exact through fma, sums through two_sum.  The powers come from the
//   host, built from the impulse response h of 1/A(z) in double-double (M^n = [[h_n, -a2 h_(n-1)], [h_(n-1),
//   -a2 h_(n-2)]]).  The per-sample recurrences stay plain double (2 DFMA each); only the 1/16 of the work that
//   combines runs pays for the extra precision.
//   several tiles per channel (len > kBqTile): three launches.  (1) the tile kernel without output gives each tile's
//                 aggregate from a zero y start and records the tile's last two x; (2) one CTA per channel
//                 (biquad_carry_kernel, tu_biquad.cu) scans the tile aggregates with M^kBqTile into every tile's true
//                 start state; (3) the tile kernel with output.
//                 The carries pass between launches in stream order, never between running CTAs, so the result does
//                 not depend on scheduling, and x is read twice: 12 B per sample instead of 8.
// In place works: launch (1) writes nothing to x, and launch (3) takes x[-1], x[-2] of a tile from the records of
// launch (1), not from memory that the previous tile may already have overwritten with y.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sg {

constexpr int kBqThreads = 256, kBqRun = 16, kBqTile = kBqThreads * kBqRun;   // 4096 samples per tile
constexpr int kBqPitch = kBqRun + 4;   // floats per run in shared memory: the float4 reads of 8 threads hit 32 banks
constexpr int kBqPowers = 9;           // M^(kBqRun 2^k), k = 0..8; k = 5: one warp's runs, k = 8: one tile

struct BqMat { double h[4], l[4]; };   // [[0, 1], [2, 3]], each entry h + l (double-double)
struct BqVec { double x, y, xl, yl; };  // a state (x, y) = (x + xl, y + yl)

struct BqArgs {
  const float* in;
  float* out;
  long long len, in_stride, out_stride;
  long long channels, tiles;           // tiles per channel: ceil(len / kBqTile)
  double b0, b1, b2, na1, na2;         // na1 = -a1, na2 = -a2
  BqMat pw[kBqPowers];
  BqMat lane[32];                      // M^(kBqRun j), j = 0..31
  BqMat carry[8];                      // M^(kBqTile carry_per 2^k): the carry scan's powers (tiles > 1)
  long long carry_per;                 // tiles per thread of the carry scan: ceil((tiles - 1) / kBqThreads)
  double* state;                       // [channels][4] {x1, x2, y1, y2} or null (zero start, no write-back)
  double* start;                       // [channels][tiles][4] {y1, y2, x1, x2} at each tile's start (tiles > 1)
  BqVec* agg;                          // [channels][tiles] tile end state from a zero y start (tiles > 1)
  int vec;                             // in/out pointers and strides allow float4 access
};

__device__ __forceinline__ void bq_two_sum(double a, double b, double& s, double& e) {
  s = a + b;
  const double bb = s - a;
  e = (a - (s - bb)) + (b - bb);
}
// (p0 + q0)(v0 + w0) + (p1 + q1)(v1 + w1) + (ah + al) as hi + lo
__device__ __forceinline__ double bq_row(double p0, double q0, double p1, double q1, double v0, double w0, double v1,
                                         double w1, double ah, double al, double& lo) {
  const double m0 = p0 * v0, m1 = p1 * v1;
  double e = fma(p0, v0, -m0) + fma(p1, v1, -m1);
  e = fma(p0, w0, fma(q0, v0, e));
  e = fma(p1, w1, fma(q1, v1, e));
  double s1, t1, s2, t2;
  bq_two_sum(ah, m0, s1, t1);
  bq_two_sum(s1, m1, s2, t2);
  e += al + t1 + t2;
  const double h = s2 + e;
  lo = e - (h - s2);
  return h;
}
// m v + add in double-double
__device__ __forceinline__ BqVec bq_apply(const BqMat& m, const BqVec& v, const BqVec& add) {
  BqVec r;
  r.x = bq_row(m.h[0], m.l[0], m.h[1], m.l[1], v.x, v.xl, v.y, v.yl, add.x, add.xl, r.xl);
  r.y = bq_row(m.h[2], m.l[2], m.h[3], m.l[3], v.x, v.xl, v.y, v.yl, add.y, add.yl, r.yl);
  return r;
}
__device__ __forceinline__ BqVec shfl_up_vec(const BqVec& v, int d) {
  return BqVec{__shfl_up_sync(0xffffffffu, v.x, d), __shfl_up_sync(0xffffffffu, v.y, d),
               __shfl_up_sync(0xffffffffu, v.xl, d), __shfl_up_sync(0xffffffffu, v.yl, d)};
}
__device__ __forceinline__ int bq_slot(int e) { return (e / kBqRun) * kBqPitch + e % kBqRun; }

// EMIT = false: launch (1), tiles 0 .. tiles-2 of every channel; EMIT = true: every tile, writing y.
template <bool EMIT>
__global__ void __launch_bounds__(kBqThreads, 2) biquad_tile_kernel(const BqArgs a) {
  __shared__ __align__(16) float s_x[kBqThreads * kBqPitch];   // x of the tile by run, then y
  __shared__ BqMat s_lane[32];                                  // M^(kBqRun j), j = 0..31
  __shared__ BqVec s_warp[kBqThreads / 32];                     // warp end states, then the warps' start states
  __shared__ double s_start[4];                                 // the tile's start state {y1, y2, x1, x2}

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long per = EMIT ? a.tiles : a.tiles - 1;
  const long long ch = blockIdx.x / per, tile = blockIdx.x % per, t0 = tile * kBqTile;
  const int n = (int)min((long long)kBqTile, a.len - t0);
  const float* __restrict__ x = a.in + ch * a.in_stride + t0;

  if (warp == 0) {
    s_lane[lane] = a.lane[lane];
  } else if (tid == 32) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    const double* src = a.tiles > 1 && EMIT ? a.start + (ch * a.tiles + tile) * 4 : nullptr;
    if (src) {
      for (int i = 0; i < 4; ++i) s[i] = src[i];
    } else if (tile > 0) {                  // launch (1): x is not written during it
      s[2] = x[-1];
      s[3] = x[-2];
    } else if (a.state) {                   // launch (1) zeroes the y start; the carry launch adds it
      const double* st = a.state + ch * 4;
      if (EMIT) { s[0] = st[2]; s[1] = st[3]; }
      s[2] = st[0];
      s[3] = st[1];
    }
    for (int i = 0; i < 4; ++i) s_start[i] = s[i];
  }
  if (n == kBqTile && a.vec) {
#pragma unroll
    for (int i = 0; i < kBqTile / (4 * kBqThreads); ++i) {
      const int e = (i * kBqThreads + tid) * 4;
      *reinterpret_cast<float4*>(s_x + bq_slot(e)) = *reinterpret_cast<const float4*>(x + e);
    }
  } else {
    for (int e = tid; e < kBqTile; e += kBqThreads) s_x[bq_slot(e)] = e < n ? x[e] : 0.f;
  }
  __syncthreads();

  // ---- u for this thread's run (x[-1], x[-2] from the previous run, or the tile's start state)
  float xr[kBqRun];
#pragma unroll
  for (int j = 0; j < kBqRun; j += 4) {
    const float4 v = *reinterpret_cast<const float4*>(s_x + tid * kBqPitch + j);
    xr[j] = v.x; xr[j + 1] = v.y; xr[j + 2] = v.z; xr[j + 3] = v.w;
  }
  const double xm1 = tid ? (double)s_x[(tid - 1) * kBqPitch + kBqRun - 1] : s_start[2];
  const double xm2 = tid ? (double)s_x[(tid - 1) * kBqPitch + kBqRun - 2] : s_start[3];
  const int jl = (int)(a.len - 1 - t0) - tid * kBqRun;      // this run holds the channel's last sample when in [0, R)
  // u[j] = b0 x[j] + b1 x[j-1] + b2 x[j-2], formed the same way in both passes (x stays in registers as float)
  auto u_at = [&](int j) {
    const double x0 = xr[j], x1 = j >= 1 ? (double)xr[j - 1] : xm1, x2 = j >= 2 ? (double)xr[j - 2] : (j == 1 ? xm1 : xm2);
    return fma(a.b2, x2, fma(a.b1, x1, a.b0 * x0));
  };

  // ---- run end state from a zero start (the tile's first run: from the tile's start state)
  double y1 = 0.0, y2 = 0.0;
  if (tid == 0) { y1 = s_start[0]; y2 = s_start[1]; }
  const double sy1 = y1, sy2 = y2;
#pragma unroll
  for (int j = 0; j < kBqRun; ++j) {
    const double y = fma(a.na2, y2, fma(a.na1, y1, u_at(j)));
    y2 = y1;
    y1 = y;
  }
  BqVec v{y1, y2, 0.0, 0.0};
#pragma unroll
  for (int k = 0; k < 5; ++k) {   // inclusive scan over the warp's runs: v_t += M^(R d) v_(t-d)
    const BqVec o = shfl_up_vec(v, 1 << k);
    if (lane >= (1 << k)) v = bq_apply(a.pw[k], o, v);
  }
  if (lane == 31) s_warp[warp] = v;
  __syncthreads();
  if (tid == 0) {
    BqVec acc{0.0, 0.0, 0.0, 0.0};
    for (int w = 0; w < kBqThreads / 32; ++w) {
      const BqVec t = s_warp[w];
      s_warp[w] = acc;
      acc = bq_apply(a.pw[5], acc, t);
    }
    if (!EMIT) {
      a.agg[ch * a.tiles + tile] = acc;
      double* nx = a.start + (ch * a.tiles + tile + 1) * 4;     // the next tile's x[-1], x[-2]
      nx[2] = s_x[(kBqThreads - 1) * kBqPitch + kBqRun - 1];
      nx[3] = s_x[(kBqThreads - 1) * kBqPitch + kBqRun - 2];
    }
  }
  if constexpr (!EMIT) return;
  __syncthreads();

  // ---- this run's true start state, then the run again with output
  BqVec prev = shfl_up_vec(v, 1);
  if (lane == 0) prev = BqVec{0.0, 0.0, 0.0, 0.0};
  if (tid != 0) {
    const BqVec s = bq_apply(s_lane[lane], s_warp[warp], prev);
    y1 = s.x;
    y2 = s.y;
  } else {
    y1 = sy1;
    y2 = sy2;
  }
  double fx1 = 0.0, fx2 = 0.0, fy1 = 0.0, fy2 = 0.0;
  float yr[kBqRun];
#pragma unroll
  for (int j = 0; j < kBqRun; ++j) {
    const double y = fma(a.na2, y2, fma(a.na1, y1, u_at(j)));
    if (j == jl) {
      fx1 = xr[j];
      fx2 = j >= 1 ? (double)xr[j - 1] : xm1;
      fy1 = y;
      fy2 = y1;
    }
    y2 = y1;
    y1 = y;
    yr[j] = __double2float_rn(y);
  }
#pragma unroll
  for (int j = 0; j < kBqRun; j += 4)
    *reinterpret_cast<float4*>(s_x + tid * kBqPitch + j) = make_float4(yr[j], yr[j + 1], yr[j + 2], yr[j + 3]);
  if (a.state && jl >= 0 && jl < kBqRun) {
    double* st = a.state + ch * 4;
    st[0] = fx1; st[1] = fx2; st[2] = fy1; st[3] = fy2;
  }
  __syncthreads();
  float* __restrict__ y = a.out + ch * a.out_stride + t0;
  if (n == kBqTile && a.vec) {
#pragma unroll
    for (int i = 0; i < kBqTile / (4 * kBqThreads); ++i) {
      const int e = (i * kBqThreads + tid) * 4;
      *reinterpret_cast<float4*>(y + e) = *reinterpret_cast<const float4*>(s_x + bq_slot(e));
    }
  } else {
    for (int e = tid; e < n; e += kBqThreads) y[e] = s_x[bq_slot(e)];
  }
}

}  // namespace sg
