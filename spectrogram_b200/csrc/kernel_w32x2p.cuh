// Headline kernel, register-pipelined form: n_fft = 2048 (the reference's fftSize, UI/player.js:10),
// hop = 512, one warp per PAIR of consecutive frames, packed FP32 arithmetic (FFMA2 / FADD2).
//
// Same arithmetic network as kernel_w32x2.cuh (1024-point complex radix-2 DIT split 5 + 5, real-FFT
// untangle, dB / byte epilogue).  That kernel is bound by the shared-memory data path (~820 wavefronts per
// frame pair against ~2400 FP32-pipe cycles per scheduler); this one moves everything that does not have
// to cross lanes out of shared memory:
//   loader     the 2560 samples a frame pair covers are read straight into registers (40 coalesced
//              8-byte loads per lane, the two frames share 24 of every 32), issued for the NEXT pair
//              during the untangle -- as the FFT registers die -- so the HBM/L2 latency hides behind
//              the untangle and the dB / byte epilogue (an extra L2 bulk prefetch one pair further ahead
//              measured no gain and was removed).  No shared-memory stage at all.
//   exchange   the 32x32 transpose keeps two planes (re, im) of (frame A, frame B) pairs with row pairs
//              interleaved: 64 STS.64 + 32 LDS.128, bank-conflict free both ways, operands already in
//              the register pairs/quads the packed arithmetic uses (no moves)
//   twiddles   pass 2 builds W_{2^u}^p * W_{32*2^u}^lane from five per-lane bases and compile-time
//              constants (scalar FMAs shared by both frames) instead of a 31-row table
//   untangle   Z[1024-k] lives in the partner lane (32 - lane): 64 warp shuffles replace the
//              shared-memory round trip of the upper half
//   non-finite [SPEC] "NaN/Inf -> 0" is decided once per frame (a non-finite sample poisons every bin
//              of its frame), folded into the byte scale, instead of once per bin
// ~550 shared-memory wavefronts per pair.  Frames the fast loader cannot express (clip edges / zero
// history, pairs that straddle clips, odd alignment) take guarded loads.
#pragma once
#include "common.cuh"
#include "ct_math.cuh"
#include "kernel_w32.cuh"
#include "kernel_w32x2.cuh"

namespace sg {

// tools/microbench/trace_bench.cu builds this kernel with SG_XP_TRACE: lane 0 of every warp of CTA 0 records clock64 at
// the top of each of its first kXpTraceIters pairs (point 0) and just before and just after each of the pair's three group
// barriers (points 1 / 2: A | B, 3 / 4: B | C, 5 / 6: C | A), so each section's busy time and each barrier's wait are
// separable (the product build compiles the hooks away)
#ifdef SG_XP_TRACE
constexpr int kXpTraceIters = 40, kXpTracePoints = 8;
__device__ long long* g_xp_trace;
#define XP_TRACE(p)                                                                                              \
  do {                                                                                                           \
    if (blockIdx.x == 0 && trace_iter < kXpTraceIters && lane == 0) {                                            \
      long long t_;                                                                                              \
      asm volatile("mov.u64 %0, %%clock64;" : "=l"(t_)::"memory");                                               \
      g_xp_trace[(warp * kXpTraceIters + trace_iter) * kXpTracePoints + (p)] = t_;                               \
    }                                                                                                            \
  } while (0)
#else
#define XP_TRACE(p) do {} while (0)
#endif

constexpr int kXpStride = 33;                               // 16-byte units per row PAIR of one plane
constexpr int kXpPlaneBytes = 2 * 16 * kXpStride * 16;      // re plane + im plane: 16896 B
constexpr int kXpBytesStage = 2 * kW32M;                    // u8 staging: 1024 (A,B) byte pairs
constexpr int kXpWarpBytes = kXpPlaneBytes;                 // the byte stage reuses the planes after the exchange
constexpr int kXpTableBytes = kW32M * 8 + 5 * 32 * 8 + 16 * 32 * 8;   // window + 5 base twiddles + untangle
// the next pair's loads are spread over the first kXpLoadSteps of the 16 untangle steps.  Byte rows at hop 512: 16 steps
// 595, 14: 600, 13: 604, 12: 604, 10: 594, 8: 591 M frames/s; float dB at hop 256 prefers 16 (576 vs 553 M with 13)
template <int OUT, int HOPJ>
constexpr int xp_load_steps() { return (HOPJ == 8 && (OUT == kOutU8 || OUT == kOutRgba8)) ? 13 : 16; }
template <int NW>
struct XpShape {
  static constexpr int kSmemBytes = kXpTableBytes + NW * kXpWarpBytes;
  static constexpr int kMaxRegs = NW <= 8 ? 255 : (65536 / (NW * 32)) / 8 * 8;
};

// Rotation.  A pair runs as three sections of different non-FMA content (the cuts between them: xp_cuts below).  Round 3's
// placement, which every output but 12-warp bytes keeps:
//   A  window + pass 1 + exchange stores         B  exchange loads + pass 2 + mirror shuffles / selects
//   C  untangle with the next pair's loads + epilogue
// 12-warp bytes move the exchange stores into B and the byte de-interleave (row stores) into the next pair's A.
// The warps of one scheduler (w, w + 4, w + 8: a rotation group) would otherwise reach the exchange, the shuffles and the
// MUFU epilogue together and leave the FP32 pipe idle meanwhile.  Instead the group runs in steps separated by one group
// barrier (ID 1 + group, NW / 4 warps): at step s, rank k (= w / 4) runs section (s + k) mod 3, so the ranks always sit in
// different sections.  Rank k opens with xp_lead(k) barrier-only steps.  Every output but RGBA rotates (kRotate below).
//
// No warp may leave its group early: every warp of a group executes exactly xp_group_steps() barriers on the group's ID.
// A warp's pairs are the frames 2 (block NW + w) + j * 2 grid NW (j >= 0) below total_frames, xp_warp_pairs() of them.
// A warp with pairs spends xp_lead(k) steps before its first pair and 3 steps on each pair, xp_warp_steps() in all; the
// group's count is the largest of its members', and every member spends the steps left over barrier-only (its tail, or
// all of them for a warp without pairs).  Every input of xp_group_steps() is uniform over the CTA, so the members agree
// on the count, and none of them runs short of it.  A group without pairs takes no step.
__host__ __device__ constexpr int xp_lead(int rank) { return (3 - rank % 3) % 3; }
__host__ __device__ inline long long xp_warp_pairs(long long total_frames, int grid, int nw, int block, int warp) {
  const long long fa = 2 * ((long long)block * nw + warp), step = 2LL * grid * nw;
  return fa < total_frames ? (total_frames - fa - 1) / step + 1 : 0;
}
__host__ __device__ inline long long xp_warp_steps(long long total_frames, int grid, int nw, int block, int warp) {
  const long long n = xp_warp_pairs(total_frames, grid, nw, block, warp);
  return n > 0 ? xp_lead(warp / 4) + 3 * n : 0;
}
__host__ __device__ inline long long xp_group_steps(long long total_frames, int grid, int nw, int block, int group) {
  long long n = 0;
  for (int warp = group; warp < nw; warp += 4) {
    const long long s = xp_warp_steps(total_frames, grid, nw, block, warp);
    n = s > n ? s : n;
  }
  return n;
}
__device__ __forceinline__ void xp_step_barrier(int group, int nw) {
  asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "r"(nw / 4 * 32) : "memory");
}

// Where the three group barriers of a pair sit (a pair stays three sections whatever the cuts, so the step counts above
// do not depend on them), packed as xp_cut(ab, bc, ca):
//   ab  A | B   0: before the exchange loads                1: after them          2: before the exchange stores
//   bc  B | C   0: after pass-2 stage 9 (stage 10 in C)     1: after stage 10     2: after the mirror shuffles and selects
//   ca  C | A   0: before the byte de-interleave (u8 only: its loads, PRMTs and row stores open the next section A)
//               1: at the end of the pair
// A cut away from a point where its barrier also ordered the warp's own shared-memory hand-off leaves a __syncwarp()
// there: exchange stores -> exchange loads, and byte stage -> the next pair's exchange stores.
// tools/microbench/rotation_cut_bench.cu times every placement (profiles/r04_cut_sweep.txt).  Byte rows with 12 warps
// take the exchange stores into B and the byte de-interleave into the next A: hop 512 (the headline) 636 -> 660 M frames/s
// with B | C where round 3 put it, hop 256 640 -> 651 M with B | C after stage 9.  Every other instantiation measured no
// gain from moving a cut and keeps round 3's.
__host__ __device__ constexpr int xp_cut(int ab, int bc, int ca) { return ab * 100 + bc * 10 + ca; }
template <int OUT, int NW, int HOPJ>
constexpr int xp_cuts() {
  return OUT != kOutU8 || NW != 12 ? xp_cut(0, 2, 1) : HOPJ == 8 ? xp_cut(2, 2, 0) : xp_cut(2, 0, 0);
}

// stage U (1..5) of pass 2: butterflies (i0, i0 + half), twiddle W_{2 half}^p * base
template <int U>
__device__ __forceinline__ void dit2_stage_gen(C2 (&a)[32], float2 base) {
  constexpr int half = 1 << (U - 1);
  static_for<0, half>([&](auto pp) {
    constexpr int p = decltype(pp)::value;
    const float2 w = twiddle_times<p, 2 * half>(base);
    static_for<0, 16 / half>([&](auto bb) {
      constexpr int i0 = decltype(bb)::value * 2 * half + p;
      bfly2(a[i0], a[i0 + half], w.x, w.y);
    });
  });
}

// sel = 0x3210: x, sel = 0x7654: y -- a select as PRMT with a per-lane selector (the ABL 128 experiment only: FSEL is faster)
__device__ __forceinline__ float pick(float x, float y, unsigned sel) {
  return __uint_as_float(__byte_perm(__float_as_uint(x), __float_as_uint(y), sel));
}

// volatile: the loads stay where they are written (interleaved with the untangle)
__device__ __forceinline__ float2 ldg_nc_f2(const float2* p) {
  float2 v;
  asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  return v;
}

// Loop state is kept small (the FFT needs nearly the whole register file): a pair is (clip, t) of frame A plus
// the running offset of its first sample, advanced incrementally (no 64-bit multiply or divide in the loop).
struct PairP {
  long long fa;    // global index of frame A; frame B = fa + 1
  long long off;   // (clip * clip_stride + start0 + t * 512): first sample of frame A, relative to g.pcm
  int clip, t;     // clip and in-clip index of frame A
};
struct PairStep {
  long long d_off, wrap_off;   // offset advance per step, and its correction when t wraps into the next clip
  int step, step_clip, step_t, fpc;
  int t_lo, t_hi;              // pairs with t in [t_lo, t_hi] lie wholly inside their clip (no zero fill)
  unsigned pcm_lo;             // low address bits of g.pcm (alignment test)
};
__device__ __forceinline__ PairP pair_advance(const PairP& c, const PairStep& st) {
  PairP n;
  n.fa = c.fa + st.step; n.clip = c.clip + st.step_clip; n.t = c.t + st.step_t; n.off = c.off + st.d_off;
  if (n.t >= st.fpc) { n.t -= st.fpc; ++n.clip; n.off += st.wrap_off; }
  return n;
}
// both frames inside one clip, no zero fill, first sample aligned to `align` bytes
__device__ __forceinline__ bool pair_is_fast(const FrameGeom& g, const PairP& p, const PairStep& st, unsigned align = 8) {
  return p.fa + 1 < g.total_frames && p.t >= st.t_lo && p.t <= st.t_hi &&
         ((st.pcm_lo + ((unsigned)p.off << 2)) & (align - 1)) == 0;
}

// ABL (tools/microbench/ablate_bench.cu only; 0 in every product launch) removes one component at a time -- results are
// wrong, the time saved is that component's marginal cost under the real contention: 1 exchange, 2 mirror shuffles,
// 4 MUFU/F2IP, 8 next-pair loads, 16 byte stage + row stores, 32 window table reads, 64 lane-0 selects (128: the
// selects as PRMT instead of FSEL; 256: the mirrors through shared memory instead of shuffles)
// CUT moves the rotation's barriers (xp_cut above); tools/microbench/rotation_cut_bench.cu sets it, product launches take
// the default
template <int OUT, int NW, int HOPJ = 8, int ABL = 0,   // hop = 64 * HOPJ samples: frame B's element j is element j + HOPJ of the lane
          int CUT = xp_cuts<OUT, NW, HOPJ>()>
__global__ void __launch_bounds__(NW * 32, 1) __maxnreg__(XpShape<NW>::kMaxRegs)
stft_w32x2p_kernel(FrameGeom g, W32Plan pl, Epilogue ep, typename OutElem<OUT>::type* __restrict__ out) {
  using T = typename OutElem<OUT>::type;
  constexpr int HOP = 64 * HOPJ, NLOAD = 32 + HOPJ, kLoadSteps = xp_load_steps<OUT, HOPJ>();
  constexpr int kCutAB = CUT / 100, kCutBC = CUT / 10 % 10, kCutCA = CUT % 10;
  static_assert(kCutAB <= 2 && kCutBC <= 2 && kCutCA <= 1 && (kCutCA == 1 || OUT == kOutU8), "no such cut");
  extern __shared__ float4 smem_raw[];
  float4* s_win4 = smem_raw;                                           // [16][32] (w2[l+32j], w2[l+32(j+16)])
  float2* s_twb = reinterpret_cast<float2*>(s_win4 + 16 * 32);         // [5][32]  W_{32*2^u}^lane
  float2* s_ut = s_twb + 5 * 32;                                       // [16][32] W_2048^{lane + 32 i}
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char* wbase = reinterpret_cast<unsigned char*>(s_ut + 16 * 32) + warp * kXpWarpBytes;
  float4* xp = reinterpret_cast<float4*>(wbase);                       // exchange planes
  uint16_t* sb16 = reinterpret_cast<uint16_t*>(wbase);   // aliases the planes: written after the exchange is read

  {
    const float2* w2 = reinterpret_cast<const float2*>(pl.win);
    for (int i = threadIdx.x; i < 16 * 32; i += blockDim.x) {
      const int j = i >> 5, l = i & 31;
      const float2 lo = __ldg(w2 + l + 32 * j), hi = __ldg(w2 + l + 32 * (j + 16));
      s_win4[i] = make_float4(lo.x, lo.y, hi.x, hi.y);
    }
    for (int i = threadIdx.x; i < 5 * 32; i += blockDim.x) {
      const int u = i >> 5, l = i & 31;
      s_twb[i] = __ldg(pl.tw2 + ((1 << u) - 1) * 32 + l);
    }
    for (int i = threadIdx.x; i < 16 * 32; i += blockDim.x) s_ut[i] = __ldg(pl.ut + i);
  }
  __syncthreads();
  const int group = warp & 3, rank = warp >> 2;
  // RGBA rows leave through per-bin colour-map gathers and 4-byte stores; in lock step those stall the whole group and the
  // rotation measured 7 % slower (467 vs 502 M frames/s at hop 512, 485 vs 522 at hop 256), so they keep free-running warps
  constexpr bool kRotate = OUT != kOutRgba8;

  PairStep st;
  st.fpc = (int)g.frames_per_clip;
  st.step = 2 * gridDim.x * NW;                        // frames between a warp's consecutive pairs
  st.step_clip = st.step / st.fpc;
  st.step_t = st.step - st.step_clip * st.fpc;
  st.d_off = (long long)st.step_clip * g.clip_stride + (long long)st.step_t * HOP;
  st.wrap_off = g.clip_stride - (long long)st.fpc * HOP;
  st.pcm_lo = (unsigned)reinterpret_cast<uintptr_t>(g.pcm);
  {
    const long long lo = g.start0 >= 0 ? 0 : (-g.start0 + HOP - 1) / HOP;
    const long long room = g.clip_len - (HOP + kW32N) - g.start0;                 // start0 + HOP t <= room
    const long long hi = room < 0 ? -1 : min((long long)st.fpc - 2, room / HOP);
    st.t_lo = (int)lo;
    st.t_hi = (int)hi;
  }
  const int fpc = st.fpc;
  PairP cur;
  cur.fa = 2 * ((long long)blockIdx.x * NW + warp);
  cur.clip = (int)(cur.fa / fpc);
  cur.t = (int)(cur.fa - (long long)cur.clip * fpc);
  cur.off = cur.clip * g.clip_stride + g.start0 + (long long)cur.t * HOP;
  bool cur_fast = pair_is_fast(g, cur, st);
  const int partner = (32 - lane) & 31;
  const bool lane0 = lane == 0;
  const unsigned lane0_sel = lane0 ? 0x7654u : 0x3210u;   // pick(): lane 0 takes the second operand

  float2 s[NLOAD];   // samples of the current pair (fast path): element m = float2 #(lane + 32 m) of the span
  const float2* idle_src = reinterpret_cast<const float2*>(pl.win) + lane;   // 4096 readable floats (build_plan)
  {
    // loads are unconditional (a pair the fast loader cannot express reads the idle table and ignores it):
    // the destination registers are the loop-carried sample registers themselves, nothing waits on a copy
    const float2* src = cur_fast ? reinterpret_cast<const float2*>(g.pcm + cur.off) + lane : idle_src;
    static_for<0, NLOAD>([&](auto mm) { constexpr int m = decltype(mm)::value; s[m] = ldg_nc_f2(src + 32 * m); });
  }
  if (kRotate && cur.fa < g.total_frames)
    for (int i = xp_lead(rank); i > 0; --i) xp_step_barrier(group, NW);

#ifdef SG_XP_TRACE
  int trace_iter = 0;
#endif
#ifdef SG_DEBUG
  unsigned dbg_epoch = 0;                       // this warp's pair counter
  unsigned* dbg_tags = dbg_warp_tags(warp);     // [0, 1024): exchange elements (writer lane, q); [1024, 2048): byte-stage entries
#endif
  while (cur.fa < g.total_frames) {   // a warp past total_frames has no pair and only runs its group's steps below
#ifdef SG_DEBUG
    ++dbg_epoch;
    if (lane == 0) dbg_count_iteration();
#endif
    XP_TRACE(0);
    // ---- steps 1-2 (+ FFT stage 1): window both frames, bit-reversed into registers
    C2 a[32];
    if (cur_fast) {
      static_for<0, 16>([&](auto jj) {
        constexpr int j = decltype(jj)::value;
        constexpr int r0 = bitrev(j, 5), r1 = bitrev(j + 16, 5);   // r1 == r0 + 1
        const float4 w = (ABL & 32) ? make_float4(0.3f, 0.4f, 0.5f, 0.6f) : s_win4[j * 32 + lane];
        window_stage1(a[r0], a[r1], s[j], s[j + 16], s[j + HOPJ], s[j + 16 + HOPJ], make_float2(w.x, w.y),
                      make_float2(w.z, w.w));
      });
    } else {
      // clip edges / zero history / the last frame of a clip paired with the first of the next
      const bool has_b = cur.fa + 1 < g.total_frames;
      int clip_b = cur.clip, tb = cur.t;
      if (has_b) { if (cur.t + 1 == fpc) { ++clip_b; tb = 0; } else ++tb; }
      const float* __restrict__ xa = g.pcm + cur.clip * g.clip_stride;
      const float* __restrict__ xb = g.pcm + clip_b * g.clip_stride;
      const long long start_a = g.start0 + (long long)cur.t * HOP, start_b = g.start0 + (long long)tb * HOP;
      auto ld = [&](const float* __restrict__ x, long long q) { return (q >= 0 && q < g.clip_len) ? __ldg(x + q) : 0.f; };
      static_for<0, 16>([&](auto jj) {
        constexpr int j = decltype(jj)::value;
        constexpr int r0 = bitrev(j, 5), r1 = bitrev(j + 16, 5);
        const long long o0 = 2 * (lane + 32 * j), o1 = 2 * (lane + 32 * (j + 16));
        const float4 w = s_win4[j * 32 + lane];
        window_stage1(a[r0], a[r1], make_float2(ld(xa, start_a + o0), ld(xa, start_a + o0 + 1)),
                      make_float2(ld(xa, start_a + o1), ld(xa, start_a + o1 + 1)),
                      make_float2(ld(xb, start_b + o0), ld(xb, start_b + o0 + 1)),
                      make_float2(ld(xb, start_b + o1), ld(xb, start_b + o1 + 1)), make_float2(w.x, w.y),
                      make_float2(w.z, w.w));
      });
    }

    // ---- pass 1: stages 2-5 in registers, compile-time twiddles
    dit2_stage_const<2>(a);
    dit2_stage_const<3>(a);
    dit2_stage_const<4>(a);
    dit2_stage_const<5>(a);

    // ---- exchange (32x32 transpose).  Each plane (re, im) keeps rows 2j and 2j+1 interleaved in 16-byte units:
    //      unit (j, col) = [row 2j | row 2j+1].  Lane b stores its element k_a as one 8-byte half (STS.64, the 16
    //      lanes of a half-warp fill 8 whole units: conflict free); lane a then reads column a of a row pair with
    //      one LDS.128 -- rows b = 2j, 2j+1 hold q = bitrev4(j), bitrev4(j) + 16.
    //      The A | B barrier, when it falls between the stores and the loads, also orders this warp's exchange.
    if constexpr (kRotate && kCutAB == 2) { XP_TRACE(1); xp_step_barrier(group, NW); XP_TRACE(2); }   // ---- A | B
    if constexpr (!(ABL & 1)) {
      float2* wre = reinterpret_cast<float2*>(xp) + ((lane >> 1) * kXpStride) * 2 + (lane & 1);
      float2* wim = wre + 16 * kXpStride * 2;
      static_for<0, 32>([&](auto qq) {
        constexpr int q = decltype(qq)::value;
        wre[2 * q] = a[q].re.v;
        wim[2 * q] = a[q].im.v;
#ifdef SG_DEBUG
        dbg_write(dbg_tags, lane * 32 + q, dbg_epoch);
#endif
      });
    }
    if constexpr (!kRotate) asm volatile("bar.sync %0, 32;" ::"r"(warp + 1) : "memory");
    else if constexpr (kCutAB == 0) { XP_TRACE(1); xp_step_barrier(group, NW); XP_TRACE(2); }   // ---- A | B
    else __syncwarp();
    if constexpr (!(ABL & 1)) {
      const float4* rre = xp + lane;
      const float4* rim = rre + 16 * kXpStride;
      static_for<0, 16>([&](auto qq) {   // ascending q0: registers stored last are overwritten last
        constexpr int q0 = decltype(qq)::value;
        constexpr int j = bitrev(q0, 4);
        const float4 vr = rre[j * kXpStride], vi = rim[j * kXpStride];
        a[q0].re = P2(vr.x, vr.y); a[q0 + 16].re = P2(vr.z, vr.w);
        a[q0].im = P2(vi.x, vi.y); a[q0 + 16].im = P2(vi.z, vi.w);
#ifdef SG_DEBUG
        // rows 2j and 2j + 1 of column `lane`: written by lanes 2j, 2j + 1 as their element `lane`, this iteration
        dbg_check(dbg_tags, (2 * j) * 32 + lane, dbg_epoch, 0);
        dbg_check(dbg_tags, (2 * j + 1) * 32 + lane, dbg_epoch, 0);
#endif
      });
      __syncwarp();
    }
    if constexpr (kRotate && kCutAB == 1) { XP_TRACE(1); xp_step_barrier(group, NW); XP_TRACE(2); }   // ---- A | B

    // ---- pass 2: stages 6-10, twiddles from the five per-lane bases
    dit2_stage_gen<1>(a, s_twb[0 * 32 + lane]);
    dit2_stage_gen<2>(a, s_twb[1 * 32 + lane]);
    dit2_stage_gen<3>(a, s_twb[2 * 32 + lane]);
    dit2_stage_gen<4>(a, s_twb[3 * 32 + lane]);
    if constexpr (kRotate && kCutBC == 0) { XP_TRACE(3); xp_step_barrier(group, NW); XP_TRACE(4); }   // ---- B | C
    dit2_stage_gen<5>(a, s_twb[4 * 32 + lane]);
    // now a[i] = Z[lane + 32 i] of both frames
    if constexpr (kRotate && kCutBC == 1) { XP_TRACE(3); xp_step_barrier(group, NW); XP_TRACE(4); }   // ---- B | C

    // a non-finite sample makes every Z of its frame non-finite: one test per frame. byte scale -> NaN -> byte 0
    const P2 poison = fma2(a[0].re, bc(0.f), mul2(a[0].im, bc(0.f)));   // 0 or NaN per frame

    // ---- untangle.  Z[1024 - k] for k = lane + 32 i is the partner lane's a[31 - i] (lane 0: its own a[32 - i]).
    //      First fetch every mirror IN PLACE (a[31 - i] <- partner's a[31 - i]; descending i keeps lane 0's own
    //      a[32 - i] intact until it is read), so the arithmetic below is pure register work with no shuffle in
    //      its dependency chains.  Bin 512 = conj Z[512] (lane 0's a[16]) is taken before a[16] is replaced.
    const P2 p512 = mul2(bc(4.f), fma2(a[16].re, a[16].re, mul2(a[16].im, a[16].im)));
    if constexpr (ABL & 256) {
      // experiment: the mirrors through the (idle) exchange planes instead of shuffles + lane-0 selects: 32 STS.64 +
      // 32 LDS.64 (128 wavefronts) instead of 64 SHFL (64 wavefronts) + 64 FSEL; lane 0's case is just an address
      float2* xre = reinterpret_cast<float2*>(xp);
      float2* xim = xre + 520;
      static_for<16, 32>([&](auto ii) {
        constexpr int i = decltype(ii)::value;
        xre[lane + 32 * (i - 16)] = a[i].re.v;
        xim[lane + 32 * (i - 16)] = a[i].im.v;
      });
      if (lane0) { xre[512] = a[0].re.v; xim[512] = a[0].im.v; }
      __syncwarp();
      static_for<0, 16>([&](auto ii) {
        constexpr int i = decltype(ii)::value;
        a[31 - i].re = P2(xre[512 - lane - 32 * i]);
        a[31 - i].im = P2(xim[512 - lane - 32 * i]);
      });
      __syncwarp();
    } else
    static_for<0, 16>([&](auto ii) {
      constexpr int i = 15 - decltype(ii)::value;
      constexpr int src = 31 - i, own = (32 - i) & 31;
      float mra = a[src].re.v.x, mrb = a[src].re.v.y, mia = a[src].im.v.x, mib = a[src].im.v.y;
      if constexpr (!(ABL & 2)) {
        mra = __shfl_sync(0xffffffffu, mra, partner);
        mrb = __shfl_sync(0xffffffffu, mrb, partner);
        mia = __shfl_sync(0xffffffffu, mia, partner);
        mib = __shfl_sync(0xffffffffu, mib, partner);
      }
      if constexpr (ABL & 64) {
        a[src].re = P2(mra, mrb);
        a[src].im = P2(mia, mib);
      } else {
        // lane 0 keeps its own value: 64 FSELs, 6.7 % of the kernel's time (ablate_bench.cu)
        if constexpr (ABL & 128) {   // the selects as PRMT with a per-lane selector: measured 580 vs 607 M frames/s
          a[src].re = P2(pick(mra, a[own].re.v.x, lane0_sel), pick(mrb, a[own].re.v.y, lane0_sel));
          a[src].im = P2(pick(mia, a[own].im.v.x, lane0_sel), pick(mib, a[own].im.v.y, lane0_sel));
        } else {
          a[src].re = P2(lane0 ? a[own].re.v.x : mra, lane0 ? a[own].re.v.y : mrb);
          a[src].im = P2(lane0 ? a[own].im.v.x : mia, lane0 ? a[own].im.v.y : mib);
        }
      }
    });
    if constexpr (kRotate && kCutBC == 2) { XP_TRACE(3); xp_step_barrier(group, NW); XP_TRACE(4); }   // ---- B | C

    // ---- next pair: geometry now, its 40 loads interleaved with the untangle below (registers free up as the
    //      untangle consumes Z), so HBM/L2 latency hides behind the untangle and the epilogue
    const PairP nxt = pair_advance(cur, st);
    const bool has_next = nxt.fa < g.total_frames;
    const bool nxt_fast = has_next && pair_is_fast(g, nxt, st);
    const float2* nsrc = nxt_fast ? reinterpret_cast<const float2*>(g.pcm + nxt.off) + lane : idle_src;

    P2 pk[16], pm[16];
    static_for<0, 16>([&](auto ii) {
      constexpr int i = decltype(ii)::value;
      const P2 zmr = a[31 - i].re, zmi = a[31 - i].im;
      const float2 w = s_ut[i * 32 + lane];
      const C2 zk = a[i];
      const P2 ex = add2(zk.re, zmr), ey = add2(zk.im, neg(zmi));          // 2E
      const P2 ox = add2(zk.im, zmi), oy = add2(zmr, neg(zk.re));          // 2O
      const P2 xr = fma2(ox, bc(w.x), fma2(oy, bc(-w.y), ex));             // 2X[k]
      const P2 xi = fma2(ox, bc(w.y), fma2(oy, bc(w.x), ey));
      const P2 yr = fma2(ex, bc(2.f), neg(xr));                            // 2 conj X[1024-k]
      const P2 yi = fma2(ey, bc(2.f), neg(xi));
      pk[i] = fma2(xr, xr, mul2(xi, xi));
      pm[i] = fma2(yr, yr, mul2(yi, yi));
      if constexpr (i == 0) {
        // lane 0: the mirror of k = 0 is the Nyquist bin (dropped); its slot carries bin 512
        pm[0] = P2(lane0 ? p512.v.x : pm[0].v.x, lane0 ? p512.v.y : pm[0].v.y);
      }
      // this step's share of the next pair's loads
      if constexpr (i < kLoadSteps && !(ABL & 8)) {
        static_for<(NLOAD * i) / kLoadSteps, (NLOAD * (i + 1)) / kLoadSteps>([&](auto mm) {
          constexpr int m = decltype(mm)::value;
          s[m] = ldg_nc_f2(nsrc + 32 * m);
        });
      }
    });
    // ---- epilogue
    const bool has_b_out = cur.fa + 1 < g.total_frames;
    T* __restrict__ row_a = out + cur.fa * (long long)kW32M;
    T* __restrict__ row_b = row_a + kW32M;   // frame B is the next global frame
    if constexpr (OUT == kOutU8 || OUT == kOutRgba8) {
      const P2 scale = add2(bc(ep.byte_a), poison);
      static_for<0, 16>([&](auto ii) {
        constexpr int i = decltype(ii)::value;
        const int k = lane + 32 * i;
        int mk = kW32M - k;
        if constexpr (i == 0) { if (lane0) mk = 512; }
        const P2 vk = fma2((ABL & 4) ? pk[i] : P2(lg2_ftz(pk[i].v.x), lg2_ftz(pk[i].v.y)), scale, bc(ep.byte_b));
        const P2 vm = fma2((ABL & 4) ? pm[i] : P2(lg2_ftz(pm[i].v.x), lg2_ftz(pm[i].v.y)), scale, bc(ep.byte_b));
        const unsigned ka = (ABL & 4) ? __float_as_uint(vk.v.x) : byte_of_scaled(vk.v.x), kb = (ABL & 4) ? __float_as_uint(vk.v.y) : byte_of_scaled(vk.v.y);
        const unsigned ma = (ABL & 4) ? __float_as_uint(vm.v.x) : byte_of_scaled(vm.v.x), mb = (ABL & 4) ? __float_as_uint(vm.v.y) : byte_of_scaled(vm.v.y);
        if constexpr (ABL & 16) {
          if (((ka ^ kb) + (ma ^ mb)) == 0x12345678u) row_a[k] = (T)ka;   // keeps the values live, never stores
        } else if constexpr (OUT == kOutU8) {
          sb16[k] = (uint16_t)__byte_perm(ka, kb, 0x0040);     // one PRMT instead of SHF + LOP3
          sb16[mk] = (uint16_t)__byte_perm(ma, mb, 0x0040);
#ifdef SG_DEBUG
          dbg_write(dbg_tags, 1024 + k, dbg_epoch);
          dbg_write(dbg_tags, 1024 + mk, dbg_epoch);
#endif
        } else {
          row_a[k] = __ldg(ep.lut + ka); row_a[mk] = __ldg(ep.lut + ma);
          if (has_b_out) { row_b[k] = __ldg(ep.lut + kb); row_b[mk] = __ldg(ep.lut + mb); }
        }
      });
      if constexpr (OUT == kOutU8 && !(ABL & 16)) __syncwarp();
      if constexpr (OUT == kOutU8 && kCutCA == 0) {   // ---- C | A of the next pair
        XP_TRACE(5); xp_step_barrier(group, NW); XP_TRACE(6);
      }
      if constexpr (OUT == kOutU8 && !(ABL & 16)) {
        // de-interleave the (A,B) byte pairs: 8 bins per lane per round, 8-byte coalesced row stores
        const uint4* s16 = reinterpret_cast<const uint4*>(sb16);
        uint2* ra = reinterpret_cast<uint2*>(row_a);
        uint2* rb = reinterpret_cast<uint2*>(row_b);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint4 w = s16[c * 32 + lane];
#ifdef SG_DEBUG
          for (int e8 = 0; e8 < 8; ++e8) dbg_check(dbg_tags, 1024 + 8 * (c * 32 + lane) + e8, dbg_epoch, 1);
#endif
          ra[c * 32 + lane] = make_uint2(__byte_perm(w.x, w.y, 0x6420), __byte_perm(w.z, w.w, 0x6420));
          if (has_b_out) rb[c * 32 + lane] = make_uint2(__byte_perm(w.x, w.y, 0x7531), __byte_perm(w.z, w.w, 0x7531));
        }
      }
    } else {
      // float dB (db_scale * lg2(p) + db_off) or magnitude (sqrt(p) * mag_scale), packed; the non-finite rule is one
      // select per value on the per-frame flag (a poisoned frame reads magnitude 0 / -inf dB).  The approx.ftz forms:
      // powers below 2^-126 read as 0.
      // (Measured slower, 510-511 vs 529 M frames/s in dB: a warp-uniform branch around a select-free copy of this loop,
      //  and select-free stores followed by a cold loop that overwrites a poisoned frame's rows.)
      const bool bad_a = !(poison.v.x == 0.f), bad_b = !(poison.v.y == 0.f);
      const float z = float_of_poisoned<OUT>();
      static_for<0, 16>([&](auto ii) {
        constexpr int i = decltype(ii)::value;
        const int k = lane + 32 * i;
        int mk = kW32M - k;
        if constexpr (i == 0) { if (lane0) mk = 512; }
        const P2 vk = float_of_power<OUT>(pk[i], ep), vm = float_of_power<OUT>(pm[i], ep);
        row_a[k] = bad_a ? z : vk.v.x; row_a[mk] = bad_a ? z : vm.v.x;
        if (has_b_out) { row_b[k] = bad_b ? z : vk.v.y; row_b[mk] = bad_b ? z : vm.v.y; }
      });
    }
    // ---- C | A of the next pair (or, where it does not fall here, the byte stage before the next exchange)
    if constexpr (kRotate && kCutCA == 1) { XP_TRACE(5); xp_step_barrier(group, NW); XP_TRACE(6); }
    else __syncwarp();
#ifdef SG_XP_TRACE
    ++trace_iter;
#endif
    cur = nxt;
    cur_fast = nxt_fast;
  }
  // barrier-only steps up to the group's count: the tail, or every step of a warp without pairs
  if constexpr (kRotate)
  for (long long i = xp_group_steps(g.total_frames, gridDim.x, NW, blockIdx.x, group) -
                     xp_warp_steps(g.total_frames, gridDim.x, NW, blockIdx.x, warp);
       i > 0; --i)
    xp_step_barrier(group, NW);
}

}  // namespace sg
