// rb_dense.cu -- the HBM-bound operators: normWav, the stand-alone impulsive noise (ISD) and the two-branch sum of algo 8.
//
// Reference arithmetic being restated (file:line under /root/reference/datautils/RawBoost.py):
//   normWav 20-25:  m = max|x|;  x / m  if (always or m > 1) else x
//   ISD     76-84:  y = copy(x); y[p] = x[p] + g_sd * x[p] * f_r;  normWav(y, 0)          (x itself is NOT normalised first)
//   algo 8  (asvspoof_2019_augall_3.py:425-432):  normWav(LnL(x) + ISD(x), 0)
//
// Design: normWav is the identity unless the peak exceeds 1 (or `always`), so nothing has to wait for the peak. One launch
// holds, per utterance, a few TILE CTAs that copy 32768 samples each to the output at streaming speed while taking the tile's
// peak, followed by one FINISHER CTA that waits for its row's tiles (they were dispatched before it) and then owns the row:
//   * applies the utterance's impulses (gathering x[p] and scattering y[p] through L2, where the row was streamed a moment ago),
//   * folds their magnitudes into the peak, and
//   * only if the reference would divide (peak > 1 or `always`) rescales the row in place while it is still L2-resident.
// HBM therefore sees each sample once in and once out. All reductions are maxima of |.|, taken on the bit patterns (for
// non-negative floats the unsigned order is the numeric order and every NaN sorts above +inf), so the result is independent
// of the reduction order, bit-exact against numpy, and NaN propagates like np.amax. DESIGN.md 4.2 has the measurements and the
// designs this one replaced.
#include <stdlib.h>

#include "rb_common.cuh"
#include "rb_dense.cuh"
#include "rb_finalize.cuh"

namespace rb {

namespace {

// ---- effective support of a notch cascade (launch_tap_support) --------------------------------------------------------------
// Filter b[0..K) keeps taps [lo, hi): lo is the largest count whose |b| sum to at most t = 2^-31 sum|b| (eps / 2, eps = 2^-30),
// hi the same rule from the other end. The sums are float64 and taken strictly in tap order -- sum|b| and lo from the left, hi
// from the right -- so the result equals plans.tap_support's cumulative sums bit for bit. Every lane of the warp runs the same
// sequential sum; the taps reach it 32 at a time by shuffle. An all-zero filter keeps nothing (0, 0); a non-finite sum keeps
// every tap.
constexpr double kTrimHalfEps = 0x1p-31;

__device__ __forceinline__ float abs_tap(const float* __restrict__ b, int K, int k) { return k < K ? fabsf(__ldg(b + k)) : 0.f; }

__device__ void tap_support_warp(const float* __restrict__ taps, int t0, int K, int lane, int2* __restrict__ out) {
  const float* b = taps + t0;
  double total = 0.0;
  for (int k0 = 0; k0 < K; k0 += 32) {
    const float v = abs_tap(b, K, k0 + lane);
    const int n = min(32, K - k0);
    for (int j = 0; j < n; ++j) total += (double)__shfl_sync(0xffffffffu, v, j);
  }
  int lo = 0, hi = K;
  if (isfinite(total)) {
    const double t = total * kTrimHalfEps;
    double c = 0.0;
    bool more = true;
    for (int k0 = 0; k0 < K && more; k0 += 32) {  // from the left (uniform: every lane holds the same sum)
      const float v = abs_tap(b, K, k0 + lane);
      const int n = min(32, K - k0);
      for (int j = 0; j < n && more; ++j) {
        c += (double)__shfl_sync(0xffffffffu, v, j);
        if (c <= t) lo = k0 + j + 1;
        else more = false;
      }
    }
    c = 0.0;
    more = true;
    for (int k0 = 0; k0 < K && more; k0 += 32) {  // from the right: lane l holds b[K-1-(k0+l)]
      const float v = k0 + lane < K ? fabsf(__ldg(b + K - 1 - (k0 + lane))) : 0.f;
      const int n = min(32, K - k0);
      for (int j = 0; j < n && more; ++j) {
        c += (double)__shfl_sync(0xffffffffu, v, j);
        if (c <= t) hi = K - (k0 + j + 1);
        else more = false;
      }
    }
    if (lo >= hi) lo = hi = 0;
  }
  if (lane == 0) *out = make_int2(lo, hi);
}

// the supports of filters f = first, first + step, ... < n_f of utterance u, one warp each
__device__ __forceinline__ void utt_tap_support(const float* __restrict__ taps, const int32_t* __restrict__ tap_off, int n_f, int u,
                                                int first, int step, int2* __restrict__ support) {
  for (int f = first; f < n_f; f += step) {
    const int i = u * n_f + f;
    const int t0 = tap_off[i];
    tap_support_warp(taps, t0, tap_off[i + 1] - t0, threadIdx.x & 31, support + i);
  }
}

constexpr int kSupportWarps = 4;

__global__ void __launch_bounds__(32 * kSupportWarps)
tap_support_kernel(const float* __restrict__ taps, const int32_t* __restrict__ tap_off, int nfilt, int2* __restrict__ support) {
  const int i = blockIdx.x * kSupportWarps + (threadIdx.x >> 5);
  if (i >= nfilt) return;
  const int t0 = tap_off[i];
  tap_support_warp(taps, t0, tap_off[i + 1] - t0, threadIdx.x & 31, support + i);
}

// ---- ISD impulse bit mask: bit p of row u set iff p is an impulse position of utterance u ---------
// One CTA per utterance assembles the row in shared memory (no global atomics, no memset) and writes it out once. With
// `support`, the same CTAs also derive the supports of the utterance's LnL filters (one launch for both).
constexpr int kMaskThreads = 256;
constexpr int kMaskSmemWords = 12 * 1024;  // rows of up to 393216 samples; longer ones take the global-atomic kernel

__global__ void __launch_bounds__(kMaskThreads)
mask_build_kernel(const int32_t* __restrict__ isd_off, const int32_t* __restrict__ isd_idx, const int32_t* __restrict__ len_arr,
                  uint32_t* __restrict__ mask, int mask_ld, const float* __restrict__ taps, const int32_t* __restrict__ tap_off,
                  int n_f, int2* __restrict__ support) {
  extern __shared__ uint32_t smask[];
  const int u = blockIdx.x, tid = threadIdx.x;
  const int beg = isd_off[u], end = isd_off[u + 1], len = len_arr[u];
  for (int w = tid; w < mask_ld; w += kMaskThreads) smask[w] = 0u;
  __syncthreads();
  constexpr int kU = 4;  // positions in flight per thread
  for (int i0 = beg + tid; i0 < end; i0 += kU * kMaskThreads) {
    int p[kU];
#pragma unroll
    for (int k = 0; k < kU; ++k) {
      const int i = i0 + k * kMaskThreads;
      p[k] = (i < end) ? __ldg(isd_idx + i) : -1;
    }
#pragma unroll
    for (int k = 0; k < kU; ++k)
      if (p[k] >= 0 && p[k] < len) atomicOr(smask + (p[k] >> 5), 1u << (p[k] & 31));
  }
  __syncthreads();
  uint32_t* mrow = mask + (size_t)u * mask_ld;
  for (int w = tid; w < mask_ld; w += kMaskThreads) mrow[w] = smask[w];
  if (support) utt_tap_support(taps, tap_off, n_f, u, tid >> 5, kMaskThreads / 32, support);
}

__global__ void __launch_bounds__(256)
mask_build_global_kernel(const int32_t* __restrict__ isd_off, const int32_t* __restrict__ isd_idx, const int32_t* __restrict__ len_arr,
                         uint32_t* __restrict__ mask, int mask_ld, const float* __restrict__ taps, const int32_t* __restrict__ tap_off,
                         int n_f, int2* __restrict__ support) {
  const int u = blockIdx.y;
  if (support && blockIdx.x == 0) utt_tap_support(taps, tap_off, n_f, u, threadIdx.x >> 5, 256 / 32, support);
  const int beg = isd_off[u], end = isd_off[u + 1], len = len_arr[u];
  uint32_t* mrow = mask + (size_t)u * mask_ld;
  for (int i = beg + blockIdx.x * 256 + threadIdx.x; i < end; i += gridDim.x * 256) {
    const int p = isd_idx[i];
    if (p >= 0 && p < len) atomicOr(mrow + (p >> 5), 1u << (p & 31));
  }
}

// ---- the streaming pass ---------------------------------------------------------------------------------------------------
// Grid: per utterance `ntiles` tile CTAs followed by ONE finisher CTA (block index u * (ntiles + 1) + j). Tile CTAs never wait:
// load, peak, store, release-increment the utterance's arrival counter, exit. The finisher spins (one thread, acquire loads)
// until all tiles of its utterance have arrived -- they were dispatched before it, so they always make progress -- and then
// owns the row: impulses, exact peak, conditional rescale, all through L2.
#ifndef RB_STREAM_THREADS
#define RB_STREAM_THREADS 512
#endif
#ifndef RB_STREAM_CHUNKS
#define RB_STREAM_CHUNKS 4
#endif
#ifndef RB_STREAM_SUBTILES
#define RB_STREAM_SUBTILES 4
#endif
#ifndef RB_STREAM_MIN_BLOCKS
#define RB_STREAM_MIN_BLOCKS 2
#endif
#ifndef RB_STREAM_IMP_U
#define RB_STREAM_IMP_U 8
#endif
#ifndef RB_STREAM_RESCALE_U
#define RB_STREAM_RESCALE_U 8
#endif
#ifndef RB_STREAM_LAG
#define RB_STREAM_LAG 48
#endif
constexpr int kSThreads = RB_STREAM_THREADS;     // threads per CTA
constexpr int kSU = RB_STREAM_CHUNKS;            // float4 chunks per thread and sub-tile
constexpr int kSub = RB_STREAM_SUBTILES;         // sub-tiles per tile CTA (two of them in flight at any time)
constexpr int kSTile = kSThreads * kSU * kSub * 4;  // samples per tile CTA (32768)
constexpr uint32_t kInfBits = 0x7f800000u;

__device__ __forceinline__ uint32_t abs_bits(float v) { return __float_as_uint(v) & 0x7fffffffu; }

// max over the CTA of a uint32 held by every thread; returned in every thread. `scratch` holds one word per warp.
__device__ __forceinline__ uint32_t block_umax(uint32_t v, uint32_t* scratch) {
  const int tid = threadIdx.x;
  v = __reduce_max_sync(0xffffffffu, v);
  __syncthreads();  // scratch may still be read by a previous call
  if ((tid & 31) == 0) scratch[tid >> 5] = v;
  __syncthreads();
  uint32_t r = scratch[0];
#pragma unroll
  for (int w = 1; w < kSThreads / 32; ++w) r = max(r, scratch[w]);
  return r;
}

__device__ __forceinline__ void red_release_add(uint32_t* addr, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}
// Polling load: relaxed (straight to L2, no cache maintenance). An acquire load invalidates the SM's whole L1 every time it
// is issued (CCTL.IVALL in the SASS); the acquire is done once, by a fence, after the loop.
__device__ __forceinline__ uint32_t ld_relaxed(const uint32_t* addr) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");
  return v;
}

struct StreamArgs {
  const float* a;            // [B][ld] input
  const float* b;            // [B][ld] second addend (kSum) or nullptr
  const int32_t* len;        // [B]
  int ld;
  int ntiles;                // tiles per row = ceil(ld / kSTile)
  int always;                // normWav(., 1)
  const int32_t* isd_off;    // kIsd: impulses of utterance u are [off[u], off[u+1])
  const int32_t* isd_idx;
  const double* isd_fr;
  float g_sd;
  float* out;                // [B][ld]; may equal a when !kSum (in place: the copy is skipped)
  uint2* state;              // [B] {peak bits, tiles arrived}; zero on entry, left zero
  int B;                     // utterances of this launch
  int lag;                   // the finisher of utterance u sits behind the tiles of utterance u + lag in the grid
};

template <bool kIsd, bool kSum>
__global__ void __launch_bounds__(kSThreads, RB_STREAM_MIN_BLOCKS)
norm_stream_kernel(const StreamArgs s) {
  __shared__ uint32_t scratch[kSThreads / 32];
  // Block g * (ntiles + 1) + j: j < ntiles is tile j of utterance g; j == ntiles is the finisher of utterance g - lag. Placing
  // a finisher `lag` utterances behind its tiles in the dispatch order means it is started when its row is (nearly) complete
  // instead of spinning -- and holding one of the SM's two CTA slots -- for as long as its tiles take.
  const int per = s.ntiles + 1;
  const int g = blockIdx.x / per, tile = blockIdx.x - g * per;
  const int u = (kIsd || tile < s.ntiles) ? g : g - s.lag;
  if (u < 0 || u >= s.B) return;
  const int tid = threadIdx.x;
  const int len = min(s.len[u], s.ld);  // (a length beyond the row stride would leave the finisher waiting for tiles that do not exist)
  const float* ra = s.a + (size_t)u * s.ld;
  float* ro = s.out + (size_t)u * s.ld;
  uint32_t* st_peak = &s.state[u].x;
  uint32_t* st_count = &s.state[u].y;

  if (tile < s.ntiles) {
    // ---- tile CTA: copy + peak ------------------------------------------------------------------------------------------
    const int tile0 = tile * kSTile;
    if (tile0 >= len) return;
    const float* rb_ = kSum ? s.b + (size_t)u * s.ld : nullptr;
    const bool copy = kSum || (ro != ra);
    // kSub sub-tiles of kSU chunks per thread, software-pipelined: the loads of sub-tile j+1 are in flight while sub-tile j
    // is reduced and stored, so the CTA keeps requests outstanding for most of its life instead of only at its start.
    auto load_sub = [&](int j, float4 (&v)[kSU]) {
#pragma unroll
      for (int k = 0; k < kSU; ++k) {
        const int p = tile0 + 4 * ((j * kSU + k) * kSThreads + tid);
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p + 3 < len) {
          v[k] = __ldg(reinterpret_cast<const float4*>(ra + p));
          if (kSum) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(rb_ + p));
            v[k] = make_float4(__fadd_rn(v[k].x, w.x), __fadd_rn(v[k].y, w.y), __fadd_rn(v[k].z, w.z), __fadd_rn(v[k].w, w.w));
          }
        } else if (p < len) {  // the ragged last chunk; zeros beyond the end are neutral for the peak
          float e[4] = {0.f, 0.f, 0.f, 0.f};
          for (int q = 0; q < 4; ++q)
            if (p + q < len) e[q] = kSum ? __fadd_rn(__ldg(ra + p + q), __ldg(rb_ + p + q)) : __ldg(ra + p + q);
          v[k] = make_float4(e[0], e[1], e[2], e[3]);
        }
      }
    };
    uint32_t m = 0u;
    auto consume_sub = [&](int j, const float4 (&v)[kSU]) {
#pragma unroll
      for (int k = 0; k < kSU; ++k) {
        const int p = tile0 + 4 * ((j * kSU + k) * kSThreads + tid);
        m = max(max(m, abs_bits(v[k].x)), max(abs_bits(v[k].y), max(abs_bits(v[k].z), abs_bits(v[k].w))));
        if (copy) {
          if (p + 3 < len) {
            *reinterpret_cast<float4*>(ro + p) = v[k];
          } else if (p < len) {
            ro[p] = v[k].x;
            if (p + 1 < len) ro[p + 1] = v[k].y;
            if (p + 2 < len) ro[p + 2] = v[k].z;
          }
        }
      }
    };
    float4 va[kSU], vb[kSU];
    load_sub(0, va);
#pragma unroll
    for (int j = 0; j < kSub; j += 2) {
      if (j + 1 < kSub) load_sub(j + 1, vb);
      consume_sub(j, va);
      if (j + 2 < kSub) load_sub(j + 2, va);
      if (j + 1 < kSub) consume_sub(j + 1, vb);
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((tid & 31) == 0) scratch[tid >> 5] = m;
    __threadfence();  // this thread's stores are visible device-wide before the arrival below
    __syncthreads();
    if (tid == 0) {
      uint32_t r = scratch[0];
#pragma unroll
      for (int w = 1; w < kSThreads / 32; ++w) r = max(r, scratch[w]);
      if (r) atomicMax(st_peak, r);
      red_release_add(st_count, 1u);  // release: the peak update above is ordered before the arrival
    }
    return;
  }

  // ---- finisher CTA: impulses, exact peak, conditional rescale (all through L2) ---------------------------------------------
  const int nact = (len + kSTile - 1) / kSTile;  // tiles of this utterance that do work
  if (nact <= 0) return;
  // The impulse values depend on the INPUT only, so the first round of them (all of them for a typical utterance) is
  // gathered -- from the input row, which the utterance's tiles are pulling through L2 at this very moment -- and evaluated
  // before the row is complete; only their stores have to wait for the tiles. (This is why a finisher with impulses sits
  // right behind its tiles, lag 0: started later it would find neither row in L2, see lag_rows() below.)
  constexpr int kU = RB_STREAM_IMP_U;  // impulses in flight per thread
  const int ibeg = kIsd ? s.isd_off[u] : 0, iend = kIsd ? s.isd_off[u + 1] : 0;
  uint32_t mt = 0u, mx = 0u;  // largest new magnitude / largest magnitude an impulse replaced
  int p0[kU];
  float t0[kU];
  auto impulse_round = [&](int i0, int (&p)[kU], float (&t)[kU]) {
    double fr[kU];
    float xv[kU];
#pragma unroll
    for (int k = 0; k < kU; ++k) {
      const int i = i0 + k * kSThreads;
      p[k] = (i < iend) ? __ldg(s.isd_idx + i) : -1;
      if (p[k] >= len) p[k] = -1;
    }
#pragma unroll
    for (int k = 0; k < kU; ++k) {
      fr[k] = (p[k] >= 0) ? __ldg(s.isd_fr + i0 + k * kSThreads) : 0.0;
      xv[k] = (p[k] >= 0) ? __ldcg(ra + p[k]) : 0.f;
    }
#pragma unroll
    for (int k = 0; k < kU; ++k) {
      t[k] = 0.f;
      if (p[k] >= 0) {
        t[k] = isd_value(xv[k], s.g_sd, fr[k]);  // y[p] = x[p] + g_sd * x[p] * f_r  (RawBoost.py:81-82)
        mx = max(mx, abs_bits(xv[k]));
        mt = max(mt, abs_bits(t[k]));
      }
    }
  };
  if (kIsd) impulse_round(ibeg + tid, p0, t0);
  if (tid == 0) {
    uint32_t spins = 0;
    while (ld_relaxed(st_count) < (uint32_t)nact) {
      __nanosleep(40);
      if (++spins > (1u << 26)) __trap();  // a row that never completes becomes a launch error, not a hung GPU
    }
    __threadfence();  // acquire: what the arriving tiles released is visible from here on (cumulative through the barrier below)
  }
  __syncthreads();
  const uint32_t M = __ldcg(st_peak);  // max |v| over the whole row
  __syncthreads();
  if (tid == 0) {  // ready for the next launch
    *st_peak = 0u;
    *st_count = 0u;
  }
  uint32_t pk = M;
  const int nchunk = (len + 3) >> 2;
  if (kIsd) {
#pragma unroll
    for (int k = 0; k < kU; ++k)
      if (p0[k] >= 0) __stcg(ro + p0[k], t0[k]);
    for (int i0 = ibeg + tid + kU * kSThreads; i0 < iend; i0 += kU * kSThreads) {  // utterances with more impulses
      int p[kU];
      float t[kU];
      impulse_round(i0, p, t);
#pragma unroll
      for (int k = 0; k < kU; ++k)
        if (p[k] >= 0) __stcg(ro + p[k], t[k]);
    }
    mt = block_umax(mt, scratch);
    mx = block_umax(mx, scratch);  // (these barriers also order the impulse stores before any read of the row below)
    // The peak of y = max(peak of the untouched samples, mt). The untouched peak is M unless the row's largest sample was
    // itself replaced (mx == M); even then nothing more is needed when a new value reaches M, or when nothing can exceed 1.
    if (mx < M || mt >= M) {
      pk = max(M, mt);
    } else if (M <= __float_as_uint(1.f)) {
      pk = M;  // some value <= M <= 1: no rescale either way
    } else {   // rare: take the peak of y itself
      uint32_t r = 0u;
      for (int c = tid; c < nchunk; c += kSThreads) {
        const int q = 4 * c;
        if (q + 3 < len) {
          const float4 w = __ldcg(reinterpret_cast<const float4*>(ro + q));
          r = max(max(r, abs_bits(w.x)), max(abs_bits(w.y), max(abs_bits(w.z), abs_bits(w.w))));
        } else {
          for (int e = q; e < len; ++e) r = max(r, abs_bits(__ldcg(ro + e)));
        }
      }
      pk = block_umax(r, scratch);
    }
  }
  const float peak = __uint_as_float(pk);
  if (!(s.always || peak > 1.f)) return;  // a NaN peak: "NaN > 1" is false, like the reference
  constexpr int kRU = RB_STREAM_RESCALE_U;  // chunks in flight per thread: the reads come from L2
  for (int c0 = tid; c0 < nchunk; c0 += kRU * kSThreads) {
    float4 w[kRU];
#pragma unroll
    for (int k = 0; k < kRU; ++k) {
      const int p = 4 * (c0 + k * kSThreads);
      w[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p + 3 < len) {
        w[k] = __ldcg(reinterpret_cast<const float4*>(ro + p));
      } else if (p < len) {
        w[k].x = __ldcg(ro + p);
        if (p + 1 < len) w[k].y = __ldcg(ro + p + 1);
        if (p + 2 < len) w[k].z = __ldcg(ro + p + 2);
      }
    }
#pragma unroll
    for (int k = 0; k < kRU; ++k) {
      const int p = 4 * (c0 + k * kSThreads);
      const float4 r = make_float4(__fdiv_rn(w[k].x, peak), __fdiv_rn(w[k].y, peak), __fdiv_rn(w[k].z, peak), __fdiv_rn(w[k].w, peak));
      if (p + 3 < len) {
        *reinterpret_cast<float4*>(ro + p) = r;
      } else if (p < len) {
        ro[p] = r.x;
        if (p + 1 < len) ro[p + 1] = r.y;
        if (p + 2 < len) ro[p + 2] = r.z;
      }
    }
  }
}

// 16-bit PCM -> float32, the conversion a wav reader applies (sample / 32768: exact in float32). n8 = groups of 8 samples.
__global__ void __launch_bounds__(256)
pcm16_to_f32_kernel(const int4* __restrict__ in, float4* __restrict__ out, size_t n8) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const int4 v = __ldg(in + i);
    const int w[4] = {v.x, v.y, v.z, v.w};
    float f[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      f[2 * k] = (float)(short)(w[k] & 0xffff) * (1.f / 32768.f);
      f[2 * k + 1] = (float)(short)((unsigned)w[k] >> 16) * (1.f / 32768.f);
    }
    out[2 * i] = make_float4(f[0], f[1], f[2], f[3]);
    out[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
  }
}

// ---- packed utterances <-> rows [B, ld] ------------------------------------------------------------------------------
// Row r is packed[off[r] - off[0], off[r + 1] - off[0]). A block covers kPackSpan samples of gridDim.y-strided rows (so any
// row count fits the grid); a thread moves four samples: one float4 on the 16-byte aligned row side, scalars on the packed
// side, whose rows start at any sample.
constexpr int kPackThreads = 256;
constexpr int kPackSpan = 4 * kPackThreads;

__device__ __forceinline__ float sample_f32(float v) { return v; }
__device__ __forceinline__ float sample_f32(int16_t v) { return (float)v * (1.f / 32768.f); }  // as pcm16_to_f32_kernel

__global__ void __launch_bounds__(256) lengths_from_offsets_kernel(const int64_t* __restrict__ off, int B, int32_t* __restrict__ len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) len[i] = (int32_t)(off[i + 1] - off[i]);
}

// rows[r][0, len) = the packed samples (as float32), rows[r][len, ld) = 0: the rows the padded entry's zero-padded input gives
template <typename T>
__global__ void __launch_bounds__(kPackThreads)
unpack_rows_kernel(const T* __restrict__ packed, const int64_t* __restrict__ off, int B, int ld, float* __restrict__ rows) {
  const int64_t p = ((int64_t)blockIdx.x * kPackThreads + threadIdx.x) * 4;
  if (p >= ld) return;
  const int64_t base = off[0];
  for (int r = blockIdx.y; r < B; r += gridDim.y) {
    const int64_t o = off[r] - base, n = off[r + 1] - base - o;
    const T* src = packed + o + p;
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = p + k < n ? sample_f32(src[k]) : 0.f;
    *reinterpret_cast<float4*>(rows + (size_t)r * ld + p) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// packed[off[r] - off[0] + i] = rows[r][i] for i < len; nothing else is written
__global__ void __launch_bounds__(kPackThreads)
pack_rows_kernel(const float* __restrict__ rows, const int64_t* __restrict__ off, int B, int ld, float* __restrict__ packed) {
  const int64_t p = ((int64_t)blockIdx.x * kPackThreads + threadIdx.x) * 4;
  if (p >= ld) return;
  const int64_t base = off[0];
  for (int r = blockIdx.y; r < B; r += gridDim.y) {
    const int64_t o = off[r] - base, n = off[r + 1] - base - o;
    if (p >= n) continue;
    const float4 v = *reinterpret_cast<const float4*>(rows + (size_t)r * ld + p);
    float* dst = packed + o + p;
    dst[0] = v.x;
    if (p + 1 < n) dst[1] = v.y;
    if (p + 2 < n) dst[2] = v.z;
    if (p + 3 < n) dst[3] = v.w;
  }
}

inline dim3 pack_grid(int B, int ld) { return dim3((unsigned)((ld + kPackSpan - 1) / kPackSpan), (unsigned)min(B, 65535)); }

}  // namespace

int launch_lengths_from_offsets(const int64_t* off, int B, int32_t* len, cudaStream_t st) {
  if (B <= 0) return RB_OK;
  lengths_from_offsets_kernel<<<(unsigned)min((B + 255) / 256, 148 * 16), 256, 0, st>>>(off, B, len);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

int launch_unpack_rows(const void* packed, bool pcm16, const int64_t* off, int B, int ld, float* rows, cudaStream_t st) {
  if (B <= 0 || ld <= 0) return RB_OK;
  if (ld % 4 != 0 || ((uintptr_t)rows & 15u)) return RB_ERR_ALIGNMENT;
  if (pcm16) unpack_rows_kernel<int16_t><<<pack_grid(B, ld), kPackThreads, 0, st>>>((const int16_t*)packed, off, B, ld, rows);
  else unpack_rows_kernel<float><<<pack_grid(B, ld), kPackThreads, 0, st>>>((const float*)packed, off, B, ld, rows);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

int launch_pack_rows(const float* rows, const int64_t* off, int B, int ld, float* packed, cudaStream_t st) {
  if (B <= 0 || ld <= 0) return RB_OK;
  if (ld % 4 != 0 || ((uintptr_t)rows & 15u)) return RB_ERR_ALIGNMENT;
  pack_rows_kernel<<<pack_grid(B, ld), kPackThreads, 0, st>>>(rows, off, B, ld, packed);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

int stream_tiles_for(int ld) { return (ld + kSTile - 1) / kSTile; }

int launch_pcm16_to_f32(const int16_t* in, float* out, size_t n, cudaStream_t st) {
  if (n == 0) return RB_OK;
  if (n % 8 != 0 || ((uintptr_t)in & 15u) || ((uintptr_t)out & 15u)) return RB_ERR_ALIGNMENT;
  const size_t n8 = n / 8;
  pcm16_to_f32_kernel<<<(unsigned)min((n8 + 255) / 256, (size_t)148 * 16), 256, 0, st>>>((const int4*)in, (float4*)out, n8);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

int launch_tap_support(const float* taps, const int32_t* tap_off, int nfilt, int2* support, cudaStream_t st) {
  if (nfilt <= 0) return RB_OK;
  tap_support_kernel<<<(nfilt + kSupportWarps - 1) / kSupportWarps, 32 * kSupportWarps, 0, st>>>(taps, tap_off, nfilt, support);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

int launch_mask_build(const int32_t* isd_off, const int32_t* isd_idx, const int32_t* len, int B, uint32_t* mask,
                      int mask_ld, const float* taps, const int32_t* tap_off, int n_f, int2* support, cudaStream_t st) {
  if (B <= 0) return RB_OK;
  if (mask_ld <= kMaskSmemWords) {
    mask_build_kernel<<<B, kMaskThreads, (size_t)mask_ld * sizeof(uint32_t), st>>>(isd_off, isd_idx, len, mask, mask_ld, taps,
                                                                                    tap_off, n_f, support);
    RB_LAUNCH_CHECK();
    return RB_OK;
  }
  RB_CUDA(cudaMemsetAsync(mask, 0, (size_t)B * mask_ld * sizeof(uint32_t), st));
  for (int b0 = 0; b0 < B; b0 += 65535) {
    const int nb = min(65535, B - b0);
    mask_build_global_kernel<<<dim3(8, nb), 256, 0, st>>>(isd_off + b0, isd_idx, len + b0, mask + (size_t)b0 * mask_ld, mask_ld,
                                                          taps, support ? tap_off + (size_t)b0 * n_f : nullptr, n_f,
                                                          support ? support + (size_t)b0 * n_f : nullptr);
    RB_LAUNCH_CHECK();
  }
  return RB_OK;
}

// Rows between an utterance's tiles and its finisher in the dispatch order (RAWBOOST_B200_STREAM_LAG overrides both defaults,
// for measurements). Measured on the B200 (profiles/r02_stream_lag_sweep.log, B = 4096): a finisher that starts later does not
// hold a CTA slot while it waits -- plain normWav goes from 0.388 ms (lag 0) to 0.369 (48) and 0.348 (192), with half the rows
// rescaled from 0.474 to 0.457 (64) -- but the rows it comes back to leave L2 after ~64-96 utterances (0.60 ms and more beyond),
// and with impulses any lag loses more than it gains (the early gather from the in-flight input row is what makes them cheap:
// 0.445 ms at lag 0, 0.51 at 16-64, 0.61 at 192, whether the late gather reads the input or the output row). Hence:
// impulses -> 0 (compiled in), plain normWav -> 48.
static int lag_rows(bool isd) {
  static const int env = [] {
    const char* e = getenv("RAWBOOST_B200_STREAM_LAG");
    return e ? (atoi(e) < 0 ? 0 : atoi(e)) : -1;
  }();
  if (isd) return 0;  // (the sweep with impulses was taken with a build whose finisher could gather late)
  return env >= 0 ? env : RB_STREAM_LAG;
}

int launch_norm_stream(const float* a, const float* b, const int32_t* len, int B, int ld, int always, const int32_t* isd_off,
                       const int32_t* isd_idx, const double* isd_fr, float g_sd, float* out, void* state, cudaStream_t st) {
  if (B <= 0 || ld <= 0) return RB_OK;
  const bool isd = isd_off != nullptr;
  if (isd && (!isd_idx || !isd_fr || b)) return RB_ERR_INVALID_ARG;  // impulses apply to a single input
  if (!a || !len || !out || !state) return RB_ERR_INVALID_ARG;
  RB_CUDA(cudaMemsetAsync(state, 0, (size_t)B * sizeof(uint2), st));
  StreamArgs s;
  s.ld = ld;
  s.ntiles = stream_tiles_for(ld);
  s.always = always;
  s.isd_idx = isd_idx;
  s.isd_fr = isd_fr;
  s.g_sd = g_sd;
  const int per = max(1, (int)(0x7fffffff / (long long)(s.ntiles + 1)) - 4096);  // utterances per launch (grid.x < 2^31)
  for (int b0 = 0; b0 < B; b0 += per) {
    const int nb = min(per, B - b0);
    s.a = a + (size_t)b0 * ld;
    s.b = b ? b + (size_t)b0 * ld : nullptr;
    s.len = len + b0;
    s.isd_off = isd ? isd_off + b0 : nullptr;
    s.out = out + (size_t)b0 * ld;
    s.state = (uint2*)state + b0;
    s.B = nb;
    s.lag = lag_rows(isd);
    const unsigned grid = (unsigned)(nb + s.lag) * (unsigned)(s.ntiles + 1);
    if (isd) norm_stream_kernel<true, false><<<grid, kSThreads, 0, st>>>(s);
    else if (b) norm_stream_kernel<false, true><<<grid, kSThreads, 0, st>>>(s);
    else norm_stream_kernel<false, false><<<grid, kSThreads, 0, st>>>(s);
    RB_LAUNCH_CHECK();
  }
  return RB_OK;
}

}  // namespace rb
