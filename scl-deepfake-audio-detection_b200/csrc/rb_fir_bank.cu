// rb_fir_bank.cu -- batched bank of ragged-length FIR filters over successive powers of a waveform.
//
// Replaces the arithmetic of filterFIR (/root/reference/datautils/RawBoost.py:51-56) and of the loop body of
// LnL_convolutive_noise (RawBoost.py:61-66):
//
//     y[u][n] = sum_f  sum_k  b_{u,f}[k] * x[u][n + (K_{u,f}+1)/2 - k] ** (pow_base + f*pow_step)
//
// with x == 0 outside [0, len[u]). This is a direct convolution on the FP32 pipe (not a dense contraction, so
// no tensor cores). Design, B200 (sm_100a):
//
//  * One CTA (128 threads) owns a tile of 2560 consecutive outputs of one utterance; each thread owns 20
//    consecutive outputs and keeps 20 x 2 partial accumulators in registers across ALL filters of the bank,
//    so the raw sum is written to HBM exactly once.
//  * The tile plus a 256-sample halo on each side is staged once in shared memory (vectorised, coalesced
//    float4 loads, zero-filled outside the utterance); the power x**p of the current filter is formed once
//    per staged sample (in fp64, rounded once, so it tracks numpy's float32 powf), not once per tap.
//  * Inner loop: register-tiled sliding window. A thread holds a circular window of 24 staged samples in
//    registers; per group of 4 taps it issues ONE LDS.128 for the 4 new window samples and TWO broadcast
//    LDS.128 for the taps, then 40 packed FFMA2 (fma.rn.f32x2, sm_100) = 80 FMAs. The 80-byte stride
//    between threads makes the window LDS.128 bank-conflict-free.
//  * FFMA2 needs both operands as aligned register pairs. Even outputs pair taps (h[i],h[i+1]) with window
//    samples (W[m],W[m+1]), m even. Odd outputs would need misaligned window pairs, so they use a second
//    copy of the taps shifted by one (ho[i] = he[i-1]) against the same aligned window pairs. The two halves
//    of an accumulator pair hold the even-tap and odd-tap partial sums of one output and are added at the end.
//  * Taps are reversed so the window slides upwards and zero-padded to whole 4-tap groups: full 24-tap bodies (the loop
//    is unrolled over two or four of them) are followed by a partial last body that stops after its last useful group.
//    Filters longer than 512 taps are processed as segments with their own staging offset.
//  * Epilogue: per-tile sum / sum of squares / min / max (and min / max over samples not hit by an ISD impulse,
//    from a per-utterance bit mask) via warp shuffles; outputs go through shared memory so the global store is
//    a coalesced STG.128 stream.
//  * Fused tail: the CTA that completes the last tile of an utterance (per-utterance arrival counter) does the whole
//    per-utterance finalisation in place from L2 -- mean removal + normWav [+ ISD scatter + normWav] for LnL, or the
//    norm-matched mix for SSI -- while the other CTAs of the SM keep the FP32 pipe busy. The kernel is a template over
//    the tail so that each variant gets its own register allocation and schedule.
#include "rb_common.cuh"
#include "rb_finalize.cuh"

namespace rb {

namespace {

// Tile geometry as a function of KR, the consecutive outputs per thread. The bank and the SSI kernel use rb_common.cuh's kR
// (20: 40 accumulator + 24 window registers leave room for the tails at four CTAs per SM); the plain single filter
// (TAIL_NONE: rb_filter_fir, the reverb view) has no tail to carry and runs with 28 outputs per thread -- more FFMA2 per window
// and tap LDS, fewer tiles per utterance: +3..5 % from K = 131 to K = 1001 (profiles/r02k_fir_single_filter_kr28.log).
// Strides of 80 B (20) and 112 B (28) both keep the window LDS.128 bank-conflict-free.
template <int KR>
struct Geo {
  static constexpr int kR = KR;
  static constexpr int kTile = kThreads * KR;
  static constexpr int kWarpSpan = 32 * KR;
  static constexpr int kWin = KR + 4;
  static constexpr int kBodyTaps = kWin;
  static constexpr int kTapCap = (3 + kSegTaps + 1 + kBodyTaps - 1) / kBodyTaps * kBodyTaps;
  static constexpr int kXS = kTile + 2 * kHalo + 64;
  static constexpr int kMaxReach = kXS - (kThreads - 1) * KR - kWin - kBodyTaps;
  static_assert(KR % 4 == 0 && (KR * 4) % 32 == 16, "window stride must be an odd multiple of 16 B (conflict-free LDS.128)");
};
static_assert(Geo<kR>::kXS == kXS && Geo<kR>::kMaxReach == kMaxReach && Geo<kR>::kTapCap == kTapCap, "Geo<kR> is rb_common.cuh's tiling");
// the names of rb_common.cuh, rebound to the geometry of the instantiation at hand
#define RB_GEO(KR)                                                     \
  [[maybe_unused]] constexpr int kR = Geo<KR>::kR;                     \
  [[maybe_unused]] constexpr int kTile = Geo<KR>::kTile;               \
  [[maybe_unused]] constexpr int kWarpSpan = Geo<KR>::kWarpSpan;       \
  [[maybe_unused]] constexpr int kWin = Geo<KR>::kWin;                 \
  [[maybe_unused]] constexpr int kBodyTaps = Geo<KR>::kBodyTaps;       \
  [[maybe_unused]] constexpr int kTapCap = Geo<KR>::kTapCap;           \
  [[maybe_unused]] constexpr int kXS = Geo<KR>::kXS;                   \
  [[maybe_unused]] constexpr int kMaxReach = Geo<KR>::kMaxReach

#ifndef RB_STAGE_INLINE
#define RB_STAGE_INLINE __forceinline__
#endif
#ifndef RB_STAGE_BATCHED
#define RB_STAGE_BATCHED(mode) ((mode) != TAIL_AFFINE)
#endif
#ifndef RB_KR_SSI
#define RB_KR_SSI RB_KR
#endif
#ifndef RB_KR_ONE
#define RB_KR_ONE 28
#endif

template <int KR>
struct __align__(16) FirSmem {
  float x1[Geo<KR>::kXS];      // staged samples, x1[j] = x[gbase + j]
  float xp[Geo<KR>::kXS];      // x1 ** power of the current filter (also reused to transpose the outputs)
  float he[Geo<KR>::kTapCap];  // reversed, zero-padded taps for even outputs
  float ho[Geo<KR>::kTapCap];  // the same shifted by one for odd outputs
  float red[4][kStatN];        // per-warp partial statistics
};

__device__ __forceinline__ float pow_round_once(float v, int p) {
  // v**p for small integer p >= 1, evaluated in fp64 and rounded to fp32 once.
#ifdef RB_POW_FP32
  float acc = v;
  for (int i = 1; i < p; ++i) acc *= v;
  return acc;
#else
  double d = (double)v, acc = d;
  for (int i = 1; i < p; ++i) acc *= d;
  return (float)acc;
#endif
}

// xp[j] = x1[j] ** kPow over the whole staged range, four samples per step (LDS.128 / STS.128, the multiply chain unrolled).
// Same arithmetic as pow_round_once: fp64 products in the same order, rounded to fp32 once.
template <int kPow, int KR>
__device__ __forceinline__ void stage_power(float* __restrict__ xp, const float* __restrict__ x1) {
  RB_GEO(KR);
  static_assert(kXS % 4 == 0, "staged range must be whole float4 chunks");
#ifdef RB_POW_FP32
  for (int j = threadIdx.x; j < kXS; j += kThreads) xp[j] = pow_round_once(x1[j], kPow);
#else
  for (int c = threadIdx.x; c < kXS / 4; c += kThreads) {
    const float4 v = reinterpret_cast<const float4*>(x1)[c];
    const double d0 = (double)v.x, d1 = (double)v.y, d2 = (double)v.z, d3 = (double)v.w;
    double a0 = d0, a1 = d1, a2 = d2, a3 = d3;
#pragma unroll
    for (int i = 1; i < kPow; ++i) {
      a0 *= d0;
      a1 *= d1;
      a2 *= d2;
      a3 *= d3;
    }
    reinterpret_cast<float4*>(xp)[c] = make_float4((float)a0, (float)a1, (float)a2, (float)a3);
  }
#endif
}

// Interior tile (all but the first and the last one or two of an utterance): every load of the thread is issued before the
// first store, ONE global round trip for the staging instead of one per chunk (the rolled loop of stage_x waits for each
// LDG.128 before its STS.128: seven / nine serialised round trips at 20 / 28 outputs per thread). Used by the single-filter
// kernels, whose tiles live 5-15 us (SSI +3.6 %, plain K = 51 +27 %, K = 131 +2.6 %); the bank keeps the rolled loop: its
// tiles live ~60 us and the extra registers cost its FFMA2 schedule 0.5 % (profiles/r02l_fir_batched_staging.log; a
// non-inlined copy and batching the edge tiles as well were measured too and are not better).
template <int KR>
__device__ RB_STAGE_INLINE void stage_x_interior(float* __restrict__ dst, const float* __restrict__ src_f) {
  RB_GEO(KR);
  constexpr int kIter = (kXS / 4 + kThreads - 1) / kThreads;
  const float4* src = reinterpret_cast<const float4*>(src_f);
  float4 v[kIter];
#pragma unroll
  for (int i = 0; i < kIter; ++i) {
    const int c = threadIdx.x + i * kThreads;  // the last, partial round re-reads the final chunk instead of branching
    v[i] = __ldg(src + ((i + 1) * kThreads <= kXS / 4 ? c : min(c, kXS / 4 - 1)));
  }
#pragma unroll
  for (int i = 0; i < kIter; ++i) {
    const int c = threadIdx.x + i * kThreads;
    if ((i + 1) * kThreads <= kXS / 4 || c < kXS / 4) reinterpret_cast<float4*>(dst)[c] = v[i];
  }
}

// Stage x[gbase .. gbase+kXS) of one utterance row into smem, zero outside [0, len).
template <int KR, bool kBatched>
__device__ __forceinline__ void stage_x(float* __restrict__ dst, const float* __restrict__ row, int len, int gbase) {
  RB_GEO(KR);
  // gbase is a multiple of 4 and the row is 16-byte aligned, so every chunk is an aligned float4.
#ifndef RB_STAGE_ROLLED
  if (kBatched && gbase >= 0 && gbase + kXS <= len) {
    stage_x_interior<KR>(dst, row + gbase);
    return;
  }
#endif
  for (int c = threadIdx.x; c < kXS / 4; c += kThreads) {
    const int pos = gbase + 4 * c;
    float4 v;
    if (pos >= 0 && pos + 3 < len) {
      v = __ldg(reinterpret_cast<const float4*>(row + pos));
    } else {
      v.x = (pos + 0 >= 0 && pos + 0 < len) ? __ldg(row + pos + 0) : 0.f;
      v.y = (pos + 1 >= 0 && pos + 1 < len) ? __ldg(row + pos + 1) : 0.f;
      v.z = (pos + 2 >= 0 && pos + 2 < len) ? __ldg(row + pos + 2) : 0.f;
      v.w = (pos + 3 >= 0 && pos + 3 < len) ? __ldg(row + pos + 3) : 0.f;
    }
    reinterpret_cast<float4*>(dst)[c] = v;
  }
}

// One filter segment: acc[r] += sum_i h[i] * src[t*kR + r + i + e0], taps already staged in he/ho (nbody*24 each).
// kUnroll = unroll factor of the 24-tap body loop: two or four bodies (480 / 960 FFMA2) per iteration give ptxas room to place
// the LDS of the next body under the FFMA2 stream of the current one (measured against no unrolling: +3.5 % / +4.2 % on the LnL
// bank, +4.4 % / +2.7 % on the single short SSI filter).
// ngroups = number of 4-tap groups that hold non-zero taps: full 24-tap bodies first, then a partial last body that stops
// after its last useful group (uniform branch), so zero padding costs at most 3 taps + alignment instead of up to 23.
template <int kUnroll, int KR>
__device__ __forceinline__ void conv_segment(float2 (&acc)[KR], const float* __restrict__ src, const float* __restrict__ he,
                                             const float* __restrict__ ho, int e0, int ngroups) {
  RB_GEO(KR);
  float2 w[kWin / 2];
#ifdef RB_WIN_LDS64
  // Window loads as 64-bit pairs: leaves ptxas free to keep every window pair in the register bank class the
  // accumulators are not in (an LDS.128 pins its four registers to an aligned quad, i.e. alternating classes).
  const float* xq = src + threadIdx.x * kR + e0;
  auto lds64 = [](const float* p) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"((unsigned)__cvta_generic_to_shared(p)));
    return v;
  };
#pragma unroll
  for (int m = 0; m < kR / 2; ++m) w[m] = lds64(xq + 2 * m);
  xq += kR;
#else
  const float4* xq = reinterpret_cast<const float4*>(src + threadIdx.x * kR + e0);
#pragma unroll
  for (int m = 0; m < kR / 4; ++m) {
    const float4 v = xq[m];
    w[2 * m] = make_float2(v.x, v.y);
    w[2 * m + 1] = make_float2(v.z, v.w);
  }
  xq += kR / 4;
#endif
  const float4* pe = reinterpret_cast<const float4*>(he);
  const float4* po = reinterpret_cast<const float4*>(ho);
  constexpr int kGroups = kWin / 4;  // groups per unrolled body
  const int nfull = ngroups / kGroups, glast = ngroups - nfull * kGroups;
#pragma unroll(kUnroll)
  for (int body = 0; body < nfull; ++body) {
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
      // the chunk that completes the window of this group lands in the slot freed by the previous group
#ifdef RB_WIN_LDS64
      w[((kR + 4 * g) % kWin) / 2] = lds64(xq);
      w[((kR + 4 * g) % kWin) / 2 + 1] = lds64(xq + 2);
      xq += 4;
#else
      const float4 v = *xq++;
      w[((kR + 4 * g) % kWin) / 2] = make_float2(v.x, v.y);
      w[((kR + 4 * g) % kWin) / 2 + 1] = make_float2(v.z, v.w);
#endif
      const float4 e = *pe++;
      const float4 o = *po++;
      const float2 e01 = make_float2(e.x, e.y), e23 = make_float2(e.z, e.w);
      const float2 o01 = make_float2(o.x, o.y), o23 = make_float2(o.z, o.w);
      // Tap-major order: ten consecutive FFMA2 share the tap operand, so it is served by the operand-reuse cache
      // and every FFMA2 reads only two register pairs from the register file (three would halve... cost a third cycle).
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r] = __ffma2_rn(e01, w[((4 * g + r) % kWin) / 2], acc[r]);          // taps 4g+0,1 x W[r],W[r+1]
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r] = __ffma2_rn(e23, w[((4 * g + r + 2) % kWin) / 2], acc[r]);      // taps 4g+2,3 x W[r+2],W[r+3]
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r + 1] = __ffma2_rn(o01, w[((4 * g + r) % kWin) / 2], acc[r + 1]);  // odd outputs: shifted taps,
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r + 1] = __ffma2_rn(o23, w[((4 * g + r + 2) % kWin) / 2], acc[r + 1]);  // same window pairs
    }
  }
  if (glast > 0) {
#pragma unroll
    for (int g = 0; g < kGroups - 1; ++g) {
      if (g >= glast) break;
      // the chunk that completes the window of this group lands in the slot freed by the previous group
#ifdef RB_WIN_LDS64
      w[((kR + 4 * g) % kWin) / 2] = lds64(xq);
      w[((kR + 4 * g) % kWin) / 2 + 1] = lds64(xq + 2);
      xq += 4;
#else
      const float4 v = *xq++;
      w[((kR + 4 * g) % kWin) / 2] = make_float2(v.x, v.y);
      w[((kR + 4 * g) % kWin) / 2 + 1] = make_float2(v.z, v.w);
#endif
      const float4 e = *pe++;
      const float4 o = *po++;
      const float2 e01 = make_float2(e.x, e.y), e23 = make_float2(e.z, e.w);
      const float2 o01 = make_float2(o.x, o.y), o23 = make_float2(o.z, o.w);
      // Tap-major order: ten consecutive FFMA2 share the tap operand, so it is served by the operand-reuse cache
      // and every FFMA2 reads only two register pairs from the register file (three would halve... cost a third cycle).
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r] = __ffma2_rn(e01, w[((4 * g + r) % kWin) / 2], acc[r]);          // taps 4g+0,1 x W[r],W[r+1]
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r] = __ffma2_rn(e23, w[((4 * g + r + 2) % kWin) / 2], acc[r]);      // taps 4g+2,3 x W[r+2],W[r+3]
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r + 1] = __ffma2_rn(o01, w[((4 * g + r) % kWin) / 2], acc[r + 1]);  // odd outputs: shifted taps,
#pragma unroll
      for (int r = 0; r < kR; r += 2) acc[r + 1] = __ffma2_rn(o23, w[((4 * g + r + 2) % kWin) / 2], acc[r + 1]);  // same window pairs
    }
  }
}

#ifndef RB_UNROLL_LNL
#define RB_UNROLL_LNL 4
#endif
#ifndef RB_UNROLL_ONE
#define RB_UNROLL_ONE 2
#endif
#ifndef RB_MIN_BLOCKS
#define RB_MIN_BLOCKS 4
#endif
#ifndef RB_MIN_BLOCKS_SSI
#define RB_MIN_BLOCKS_SSI RB_MIN_BLOCKS
#endif
// kTailMode is a compile-time constant: each tail (none / LnL[->ISD] / SSI) is its own kernel, so the code of one never weighs on
// the register allocation and instruction schedule of another.
template <int kTailMode, int KR>
__global__ void __launch_bounds__(kThreads, kTailMode == TAIL_SSI ? RB_MIN_BLOCKS_SSI : RB_MIN_BLOCKS)
fir_bank_kernel(const float* __restrict__ x, const int32_t* __restrict__ len_arr, int ld, const float* __restrict__ taps,
                const int32_t* __restrict__ tap_off, const int2* __restrict__ support, int n_f, int pow_base, int pow_step,
                float* __restrict__ y, float* __restrict__ stats, const uint32_t* __restrict__ mask, int mask_ld, FirTail tail) {
  RB_GEO(KR);
  constexpr bool kBatchedStaging = RB_STAGE_BATCHED(kTailMode);
  // LnL and SSI run each filter over its effective support (support[u * n_f + f]: kept taps [lo, hi), see launch_tap_support);
  // NULL, and the plain filter of the caller's taps, run every tap.
  constexpr bool kTrim = kTailMode != TAIL_NONE;
  __shared__ FirSmem<KR> sm;
  __shared__ int s_last;
  const int u = blockIdx.y;
  const int tile = blockIdx.x;
  const int ntiles = gridDim.x;
  const int len = len_arr[u];
  const int tile0 = tile * kTile;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  float* st_out = stats ? stats + ((size_t)u * ntiles + tile) * kStatN : nullptr;

  if (tile0 >= len) {  // tile entirely past the end of this utterance: neutral statistics, nothing else
    if (st_out && tid < kStatN) {
      float v = 0.f;
      if (tid == S_MIN || tid == S_MINU) v = INFINITY;
      if (tid == S_MAX || tid == S_MAXU) v = -INFINITY;
      st_out[tid] = v;
    }
    return;
  }
  const float* row = x + (size_t)u * ld;
  const bool warp_active = tile0 + warp * kWarpSpan < len;  // warps whose outputs are all past the end only help staging

  int gbase = tile0 - kHalo;
  // The first filter's taps are requested BEFORE the waveform tile, so that the two global round trips of a tile's start-up
  // overlap instead of following each other (it matters for single short filters: ~1 us of ~5 us of fixed cost per tile).
  // staged0: the first segment's taps are already in he / ho when the filter loop gets there.
  bool staged0 = false;
  // SSI: the signal tile is only needed for its sum of squares. Its loads go out with the start-up round trip as well and are
  // reduced to one register right behind the staging, instead of costing every tile a third, exposed round trip in the epilogue.
  float aux_sq = 0.f;
  float4 av[kTailMode == TAIL_SSI ? kR / 4 : 1];
  if (kTailMode == TAIL_SSI) {
    const float* arow = tail.aux + (size_t)u * ld + tile0;
    const int valid = min(kTile, len - tile0);
#pragma unroll
    for (int k = 0; k < kR / 4; ++k) {
      const int p = 4 * (k * kThreads + tid);
      if (p + 3 < valid) {
        av[k] = __ldg(reinterpret_cast<const float4*>(arow + p));
      } else {
        av[k].x = (p + 0 < valid) ? __ldg(arow + p + 0) : 0.f;
        av[k].y = (p + 1 < valid) ? __ldg(arow + p + 1) : 0.f;
        av[k].z = (p + 2 < valid) ? __ldg(arow + p + 2) : 0.f;
        av[k].w = (p + 3 < valid) ? __ldg(arow + p + 3) : 0.f;
      }
    }
  }
  {
    const int t0 = tap_off[u * n_f];
    const int K = tap_off[u * n_f + 1] - t0;
    int mlo = 0, mhi = K;
    if (kTrim && support) {
      const int2 s = support[u * n_f];
      mlo = K - s.y;
      mhi = K - s.x;
    }
    const int kseg = min(kSegTaps, mhi - mlo);
    const int e = tile0 + ((K + 1) >> 1) - (K - 1) + mlo - gbase;
    if (K > 0 && mhi > mlo && e >= 0 && e + kseg <= kMaxReach) {
      const int z = e & 3;
      const int ngroups = (z + kseg + 1 + 3) >> 2;
      const int nbody = (ngroups + kBodyTaps / 4 - 1) / (kBodyTaps / 4);
      constexpr int kPre = (kTapCap + kThreads - 1) / kThreads;  // taps per thread (5)
      float tp[kPre];
#pragma unroll
      for (int q = 0; q < kPre; ++q) {
        const int i = tid + q * kThreads, m = i - z;
        tp[q] = (i < nbody * kBodyTaps && m >= 0 && m < kseg) ? __ldg(taps + t0 + (K - 1 - (mlo + m))) : 0.f;
      }
      stage_x<KR, kBatchedStaging>(sm.x1, row, len, gbase);
#pragma unroll
      for (int q = 0; q < kPre; ++q) {
        const int i = tid + q * kThreads;
        if (i < nbody * kBodyTaps) {
          sm.he[i] = tp[q];
          if (i + 1 < nbody * kBodyTaps) sm.ho[i + 1] = tp[q];
          if (i == 0) sm.ho[0] = 0.f;
        }
      }
      staged0 = true;
    } else {
      stage_x<KR, kBatchedStaging>(sm.x1, row, len, gbase);
    }
  }

  if (kTailMode == TAIL_SSI) {
#pragma unroll
    for (int k = 0; k < kR / 4; ++k) {
      aux_sq = fmaf(av[k].x, av[k].x, aux_sq);
      aux_sq = fmaf(av[k].y, av[k].y, aux_sq);
      aux_sq = fmaf(av[k].z, av[k].z, aux_sq);
      aux_sq = fmaf(av[k].w, av[k].w, aux_sq);
    }
  }

  float2 acc[kR];
#pragma unroll
  for (int r = 0; r < kR; ++r) acc[r] = make_float2(0.f, 0.f);

  int staged_pow = 1;  // power currently held by sm.xp (1 = none, x1 is used directly)
  for (int f = 0; f < n_f; ++f) {
    const int t0 = tap_off[u * n_f + f];
    const int K = tap_off[u * n_f + f + 1] - t0;
    int mlo = 0, mhi = K;  // reversed taps h[m] = b[K-1-m] that are run: m in [mlo, mhi)
    if (kTrim && support) {
      const int2 s = support[u * n_f + f];  // kept taps b[s.x .. s.y)
      mlo = K - s.y;
      mhi = K - s.x;
    }
    if (K <= 0 || mhi <= mlo) continue;
    const int power = pow_base + f * pow_step;
    const int shift = (K + 1) >> 1;  // reference delay compensation, RawBoost.py:52,55: from the full K, trimmed or not
    const int d0 = shift - (K - 1), tlast = t0 + K - 1;
    for (int i0 = mlo; i0 < mhi; i0 += kSegTaps) {
      const int kseg = min(kSegTaps, mhi - i0);
      // this segment covers m in [i0, i0+kseg):
      //   y[n] += sum_{i<kseg} h[i0+i] * xp[n + i + d],  d = shift - (K-1) + i0
      const int d = d0 + i0;
      int e = tile0 + d - gbase;
      const bool prestaged = staged0;  // the first segment run is filter 0's first one: the one staged with the waveform
      staged0 = false;
      if (!prestaged) __syncthreads();  // previous segment done with he/ho/xp (and x1 staged on first pass)
      if (e < 0 || e + kseg > kMaxReach) {  // uniform: restage the samples around this segment
        gbase = (tile0 + d) & ~3;
        e = tile0 + d - gbase;
        stage_x<KR, kBatchedStaging>(sm.x1, row, len, gbase);
        staged_pow = 1;
        __syncthreads();
      }
      const int z = e & 3;                                      // leading zero taps that align the window to 16 B
      const int ngroups = (z + kseg + 1 + 3) >> 2;              // 4-tap groups holding taps (+1: the odd-output copy is shifted)
      const int nbody = (ngroups + kBodyTaps / 4 - 1) / (kBodyTaps / 4);
      if (!prestaged) {
        for (int i = tid; i < nbody * kBodyTaps; i += kThreads) {
          const int m = i - z;                                    // he[i] = h[i0 + m]
          const float hv = (m >= 0 && m < kseg) ? __ldg(taps + tlast - (i0 + m)) : 0.f;
          sm.he[i] = hv;
          if (i + 1 < nbody * kBodyTaps) sm.ho[i + 1] = hv;
          if (i == 0) sm.ho[0] = 0.f;
        }
      }
      const float* src = sm.x1;
      if (power != 1) {
        if (staged_pow != power) {
          switch (power) {  // uniform; the LnL bank uses 2..N_f
            case 2: stage_power<2, KR>(sm.xp, sm.x1); break;
            case 3: stage_power<3, KR>(sm.xp, sm.x1); break;
            case 4: stage_power<4, KR>(sm.xp, sm.x1); break;
            case 5: stage_power<5, KR>(sm.xp, sm.x1); break;
            default:
              for (int j = tid; j < kXS; j += kThreads) sm.xp[j] = pow_round_once(sm.x1[j], power);
          }
          staged_pow = power;
        }
        src = sm.xp;
      }
      __syncthreads();
      if (warp_active) conv_segment<kTailMode == TAIL_AFFINE ? RB_UNROLL_LNL : RB_UNROLL_ONE, KR>(acc, src, sm.he, sm.ho, e - z, ngroups);
    }
  }
  __syncthreads();  // everyone is done reading xp; reuse it to transpose the outputs

  // ---- epilogue: fold the accumulator halves, statistics, coalesced store ---------------------------
  const int n0 = tile0 + tid * kR;
  float s_sum = 0.f, s_sq = 0.f, s_min = INFINITY, s_max = -INFINITY, s_minu = INFINITY, s_maxu = -INFINITY;
  uint32_t hit = 0;  // bit r set: output n0+r is an ISD impulse position
  if (mask && n0 < len) {
    const uint32_t* mrow = mask + (size_t)u * mask_ld;
    const int wi = n0 >> 5, sh = n0 & 31;
    uint32_t lo = mrow[wi];
    uint32_t hi = (sh > 32 - kR && wi + 1 < mask_ld) ? mrow[wi + 1] : 0u;
    hit = (uint32_t)((((uint64_t)hi << 32) | lo) >> sh);
  }
  float outv[kR];
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    const float v = acc[r].x + acc[r].y;
    outv[r] = v;
    if (kTailMode == TAIL_AFFINE) {
      if (n0 + r < len) {
        s_sum += v;
        s_sq = fmaf(v, v, s_sq);
        s_min = fminf(s_min, v);
        s_max = fmaxf(s_max, v);
        if (!((hit >> r) & 1u)) {
          s_minu = fminf(s_minu, v);
          s_maxu = fmaxf(s_maxu, v);
        }
      }
    } else if (kTailMode == TAIL_SSI) {  // the SSI gain needs the two sums of squares only (rb_finalize.cuh: ssi_scale_block)
      if (n0 + r < len) s_sq = fmaf(v, v, s_sq);
    }
  }
#pragma unroll
  for (int m = 0; m < kR / 4; ++m)
    reinterpret_cast<float4*>(sm.xp + tid * kR)[m] = make_float4(outv[4 * m], outv[4 * m + 1], outv[4 * m + 2], outv[4 * m + 3]);

  if (kTailMode == TAIL_AFFINE) {
    s_sum = warp_sum(s_sum);
    s_sq = warp_sum(s_sq);
    s_min = warp_min(s_min);
    s_max = warp_max(s_max);
    s_minu = warp_min(s_minu);
    s_maxu = warp_max(s_maxu);
    if (lane == 0) {
      sm.red[warp][S_SUM] = s_sum;
      sm.red[warp][S_SUMSQ] = s_sq;
      sm.red[warp][S_MIN] = s_min;
      sm.red[warp][S_MAX] = s_max;
      sm.red[warp][S_MINU] = s_minu;
      sm.red[warp][S_MAXU] = s_maxu;
    }
  } else if (kTailMode == TAIL_SSI) {
    s_sq = warp_sum(s_sq);
    aux_sq = warp_sum(aux_sq);
    if (lane == 0) {
      sm.red[warp][S_SUMSQ] = s_sq;
      sm.red[warp][S_AUXSQ] = aux_sq;
    }
  }
  __syncthreads();
  if (kTailMode == TAIL_AFFINE) {
    if (tid < kStatN) {
      float v;
      if (tid == S_SUM || tid == S_SUMSQ) v = (sm.red[0][tid] + sm.red[1][tid]) + (sm.red[2][tid] + sm.red[3][tid]);
      else if (tid == S_MIN || tid == S_MINU) v = fminf(fminf(sm.red[0][tid], sm.red[1][tid]), fminf(sm.red[2][tid], sm.red[3][tid]));
      else if (tid == S_MAX || tid == S_MAXU) v = fmaxf(fmaxf(sm.red[0][tid], sm.red[1][tid]), fmaxf(sm.red[2][tid], sm.red[3][tid]));
      else v = 0.f;
      st_out[tid] = v;
    }
  } else if (kTailMode == TAIL_SSI) {
    if (tid == S_SUMSQ || tid == S_AUXSQ) st_out[tid] = (sm.red[0][tid] + sm.red[1][tid]) + (sm.red[2][tid] + sm.red[3][tid]);
  }
  float* yrow = y + (size_t)u * ld + tile0;
  const int valid = min(kTile, len - tile0);
#pragma unroll
  for (int k = 0; k < kR / 4; ++k) {
    const int c = k * kThreads + tid;  // float4 chunk within the tile
    const int p = 4 * c;
    if (p + 3 < valid) {
      reinterpret_cast<float4*>(yrow)[c] = reinterpret_cast<const float4*>(sm.xp)[c];
    } else {
      for (int q = 0; q < 4; ++q)
        if (p + q < valid) yrow[p + q] = sm.xp[p + q];
    }
  }
  if (kTailMode == TAIL_NONE) return;

  // ---- fused tail: the CTA that finishes the last tile of an utterance finalises the whole utterance -----------------------
  // (per-utterance reductions need every tile, so this is the one grid-level dependency of the path; the raw tiles were
  // written a moment ago and are read back from L2 while the other CTAs of the SM keep the FP32 pipe busy.)
  const int nact = (len + kTile - 1) / kTile;  // tiles of this utterance that do work (the others returned at once)
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const unsigned prev = atomicAdd(tail.counters + u, 1u);
    s_last = (prev == (unsigned)(nact - 1));
    if (s_last) tail.counters[u] = 0u;  // ready for the next launch
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const float* raw = y + (size_t)u * ld;
  float* orow = tail.out + (size_t)u * ld;
  const float* ust = stats + (size_t)u * ntiles * kStatN;
  const int nchunk = (len + 3) >> 2;
  if (kTailMode == TAIL_AFFINE) {
    const bool with_isd = tail.isd_off != nullptr;
    const int ibeg = with_isd ? tail.isd_off[u] : 0, iend = with_isd ? tail.isd_off[u + 1] : 0;
    // The CTA's shared memory is idle now: x1, xp, he and ho (contiguous) keep the impulses' new values between the gather
    // and the scatter, 7328 of them -- the most P = 10 % gives at L = 64 600 is 6460.
    constexpr int kIsdCap = offsetof(FirSmem<KR>, red) / sizeof(float);
    static_assert(offsetof(FirSmem<KR>, x1) == 0 && kIsdCap == 2 * kXS + 2 * kTapCap, "x1, xp, he, ho must be one run of floats");
    float* isd_v = reinterpret_cast<float*>(&sm);
    const UttParams pr = finalize_block(ust, nact, len, 1, 0, raw, tail.isd_idx, tail.isd_fr, ibeg, iend, with_isd, tail.g_sd,
                                        isd_v, kIsdCap);
    // division by 1 is the identity: skip the idle normalisations (the common case at speech level), bit for bit the same
    const int ndiv = (pr.div1 != 1.f) + (pr.div2 != 1.f);
    const float dv = (pr.div1 != 1.f) ? pr.div1 : pr.div2;
    auto aff = [&](float e) {
      const float d = __fsub_rn(e, pr.sub);
      if (ndiv == 0) return d;
      if (ndiv == 1) return __fdiv_rn(d, dv);
      return __fdiv_rn(__fdiv_rn(d, pr.div1), pr.div2);
    };
    // When the raw sum was written into the output buffer itself (out == y: no intermediate ever reaches HBM) and some
    // impulses did not fit in shared memory, the impulse positions must survive the dense pass untouched, because the scatter
    // gathers those impulses' raw values again.
    const bool keep_hits = with_isd && (orow == raw) && mask != nullptr && iend - ibeg > kIsdCap;
    const uint32_t* mrow = keep_hits ? mask + (size_t)u * mask_ld : nullptr;
    constexpr int kU = 4;  // chunks in flight per thread: the reads come from L2, keep several outstanding
    for (int c0 = tid; c0 < nchunk; c0 += kU * kThreads) {
      float4 v[kU];
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const int p = 4 * (c0 + k * kThreads);
        if (p + 3 < len) {
          v[k] = __ldcg(reinterpret_cast<const float4*>(raw + p));
        } else {
          v[k].x = (p + 0 < len) ? __ldcg(raw + p + 0) : 0.f;
          v[k].y = (p + 1 < len) ? __ldcg(raw + p + 1) : 0.f;
          v[k].z = (p + 2 < len) ? __ldcg(raw + p + 2) : 0.f;
          v[k].w = 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const int p = 4 * (c0 + k * kThreads);
        float4 r = make_float4(aff(v[k].x), aff(v[k].y), aff(v[k].z), aff(v[k].w));
        if (keep_hits && p < len) {  // in place: impulse positions keep the raw value for the scatter below
          const uint32_t hit = (__ldg(mrow + (p >> 5)) >> (p & 31)) & 0xFu;
          if (hit & 1u) r.x = v[k].x;
          if (hit & 2u) r.y = v[k].y;
          if (hit & 4u) r.z = v[k].z;
          if (hit & 8u) r.w = v[k].w;
        }
        if (p + 3 < len) {
          *reinterpret_cast<float4*>(orow + p) = r;
        } else {
          if (p + 0 < len) orow[p + 0] = r.x;
          if (p + 1 < len) orow[p + 1] = r.y;
          if (p + 2 < len) orow[p + 2] = r.z;
        }
      }
    }
    if (with_isd) {
      __syncthreads();  // impulse positions overwrite what the dense pass just stored
      // the positions are a permutation prefix: no two impulses write the same sample, so the order of the writes is free
      for (int i0 = ibeg + tid; i0 < iend; i0 += kIsdInFlight * kThreads) {
        int p[kIsdInFlight];
#pragma unroll
        for (int k = 0; k < kIsdInFlight; ++k) {
          const int i = i0 + k * kThreads;
          p[k] = i < iend ? tail.isd_idx[i] : -1;
        }
#pragma unroll
        for (int k = 0; k < kIsdInFlight; ++k) {
          const int i = i0 + k * kThreads;
          if (p[k] >= 0 && p[k] < len) {
            float v;
            if (i - ibeg < kIsdCap) {
              v = isd_v[i - ibeg];
            } else {  // past the shared-memory capacity (rows much longer than 64 600 samples): gathered again
              v = isd_value(__fdiv_rn(__fsub_rn(__ldcg(raw + p[k]), pr.sub), pr.div1), tail.g_sd, tail.isd_fr[i]);
            }
            orow[p[k]] = __fdiv_rn(v, pr.div2);
          }
        }
      }
    }
  } else {  // TAIL_SSI: out = x + coloured noise * scale  (RawBoost.py:95-96)
    const float scale = ssi_scale_block(ust, S_AUXSQ, ust, nact, tail.snr_db[u]);
    const float* arow = tail.aux + (size_t)u * ld;
    constexpr int kU = 4;  // (eight per array was measured: 1 % slower)
    for (int c0 = tid; c0 < nchunk; c0 += kU * kThreads) {
      float4 v[kU], a[kU];
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const int p = 4 * (c0 + k * kThreads);
        if (p + 3 < len) {
          v[k] = __ldcg(reinterpret_cast<const float4*>(raw + p));
          a[k] = __ldg(reinterpret_cast<const float4*>(arow + p));
        } else {
          v[k].x = (p + 0 < len) ? __ldcg(raw + p + 0) : 0.f;
          v[k].y = (p + 1 < len) ? __ldcg(raw + p + 1) : 0.f;
          v[k].z = (p + 2 < len) ? __ldcg(raw + p + 2) : 0.f;
          v[k].w = 0.f;
          a[k].x = (p + 0 < len) ? __ldg(arow + p + 0) : 0.f;
          a[k].y = (p + 1 < len) ? __ldg(arow + p + 1) : 0.f;
          a[k].z = (p + 2 < len) ? __ldg(arow + p + 2) : 0.f;
          a[k].w = 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < kU; ++k) {
        const int p = 4 * (c0 + k * kThreads);
        const float4 r = make_float4(__fmaf_rn(v[k].x, scale, a[k].x), __fmaf_rn(v[k].y, scale, a[k].y),
                                     __fmaf_rn(v[k].z, scale, a[k].z), __fmaf_rn(v[k].w, scale, a[k].w));
        if (p + 3 < len) {
          *reinterpret_cast<float4*>(orow + p) = r;
        } else {
          if (p + 0 < len) orow[p + 0] = r.x;
          if (p + 1 < len) orow[p + 1] = r.y;
          if (p + 2 < len) orow[p + 2] = r.z;
        }
      }
    }
  }
}

}  // namespace

int launch_fir_bank(const float* x, const int32_t* len, int B, int ld, const float* taps, const int32_t* tap_off,
                    const int2* support, int n_f, int pow_base, int pow_step, float* y, float* stats, const uint32_t* mask,
                    int mask_ld, const FirTail& tail, cudaStream_t st) {
  if (B <= 0 || ld <= 0) return RB_OK;
  if (tail.mode != TAIL_NONE) {
    if (!stats || !tail.counters || !tail.out || (tail.mode == TAIL_SSI && (!tail.aux || !tail.snr_db))) return RB_ERR_INVALID_ARG;
    RB_CUDA(cudaMemsetAsync(tail.counters, 0, (size_t)B * sizeof(uint32_t), st));
  }
  // gridDim.y is limited to 65535: split very large batches over several launches.
  // tiles of the instantiation launched; the statistics (tails only) are laid out [B][tiles_for(ld)][kStatN]
  const int ntiles = tail.mode == TAIL_NONE  ? (ld + Geo<RB_KR_ONE>::kTile - 1) / Geo<RB_KR_ONE>::kTile
                     : tail.mode == TAIL_SSI ? (ld + Geo<RB_KR_SSI>::kTile - 1) / Geo<RB_KR_SSI>::kTile
                                             : tiles_for(ld);
  for (int b0 = 0; b0 < B; b0 += 65535) {
    const int nb = min(65535, B - b0);
    dim3 grid(ntiles, nb);
    profile_begin(st);
    auto kernel = tail.mode == TAIL_AFFINE ? fir_bank_kernel<TAIL_AFFINE, kR>
                  : tail.mode == TAIL_SSI  ? fir_bank_kernel<TAIL_SSI, RB_KR_SSI>
                                           : fir_bank_kernel<TAIL_NONE, RB_KR_ONE>;
    // Largest shared-memory carve-out: the kernel itself needs little L1, and the device planner's kernels (up to ~100 KB of
    // shared memory per CTA) can then run in what the four FIR CTAs of an SM leave free instead of waiting for them.
    RB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    kernel<<<grid, kThreads, 0, st>>>(x + (size_t)b0 * ld, len + b0, ld, taps, tap_off + (size_t)b0 * n_f,
                                       support ? support + (size_t)b0 * n_f : nullptr, n_f, pow_base, pow_step, y + (size_t)b0 * ld,
                                       stats ? stats + (size_t)b0 * ntiles * kStatN : nullptr,
                                       mask ? mask + (size_t)b0 * mask_ld : nullptr, mask_ld, tail.shifted(b0, ld));
    profile_end(st);
    RB_LAUNCH_CHECK();
  }
  return RB_OK;
}

}  // namespace rb
