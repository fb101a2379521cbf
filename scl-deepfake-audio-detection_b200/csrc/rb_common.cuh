// Shared constants and small device helpers for the RawBoost sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "rawboost_b200.h"

namespace rb {

// ---- tiling of the FIR-bank kernel (rb_fir_bank.cu) ------------------------------------------------
constexpr int kThreads = 128;               // 4 warps per CTA, up to 4 CTAs per SM
#ifndef RB_KR
#define RB_KR 20
#endif
constexpr int kR = RB_KR;                   // consecutive outputs per thread (20 -> 80 B stride: conflict-free LDS.128)
constexpr int kTile = kThreads * kR;        // 2560 outputs per CTA
constexpr int kWarpSpan = 32 * kR;          // 640 outputs per warp
constexpr int kWin = kR + 4;                // circular register window (floats)
constexpr int kBodyTaps = kWin;             // taps consumed per unrolled loop body (6 groups of 4)
constexpr int kHalo = 256;                  // default staging starts kHalo samples before the tile
constexpr int kSegTaps = 512;               // longest filter segment handled by one staging
constexpr int kTapCap = (3 + kSegTaps + 1 + kBodyTaps - 1) / kBodyTaps * kBodyTaps;  // staged taps per copy (528)
constexpr int kXS = kTile + 2 * kHalo + 64; // staged samples (3136)
constexpr int kMaxReach = kXS - (kThreads - 1) * kR - kWin - kBodyTaps;  // e + Kseg must stay <= this (548)

// ---- per-tile partial statistics written by the FIR-bank and dense-stats kernels --------------------
// [B][ntiles][kStatN] floats: sum, sum of squares, min, max, min/max over samples NOT hit by an ISD impulse.
constexpr int kStatN = 8;
enum { S_SUM = 0, S_SUMSQ = 1, S_MIN = 2, S_MAX = 3, S_MINU = 4, S_MAXU = 5, S_AUXSQ = 6 };  // AUXSQ: sum of squares of FirTail::aux

// ---- per-utterance scalars consumed by the dense apply pass: out = ((in - sub) / div1) / div2 -------
struct __align__(16) UttParams {
  float sub;    // mean removed by LnL (0 otherwise)
  float div1;   // first conditional peak normalisation (1 = idle)
  float div2;   // second one (after ISD)              (1 = idle)
  float scale;  // SSI: noise gain
};

inline int tiles_for(int ld) { return (ld + kTile - 1) / kTile; }

extern std::atomic<uint64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

#define RB_CUDA(expr)                                  \
  do {                                                 \
    cudaError_t e__ = (expr);                          \
    if (e__ != cudaSuccess) return (int)e__;           \
  } while (0)
#define RB_LAUNCH_CHECK()                              \
  do {                                                 \
    cudaError_t e__ = cudaGetLastError();              \
    if (e__ != cudaSuccess) return (int)e__;           \
    ::rb::count_launch();                              \
  } while (0)

// ---- optional per-launch timing of the FIR-bank kernel (bench.py's roofline figure) ------------------
// When enabled through rb_profile_enable(), launch_fir_bank brackets its launch with CUDA events recorded on
// the launching stream; rb_profile_read() synchronises them and returns the accumulated device time.
void profile_begin(cudaStream_t st);
void profile_end(cudaStream_t st);

// ---- warp / block reductions (shuffle tree, deterministic) -----------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// NaN-propagating max|.| helpers: numpy's amax returns NaN if any element is NaN; fmaxf would drop it.
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a) ? a : ((b != b) ? b : fmaxf(a, b)); }
__device__ __forceinline__ float nan_min(float a, float b) { return (a != a) ? a : ((b != b) ? b : fminf(a, b)); }

// ---- fused tail of the FIR-bank kernel ---------------------------------------------------------------------------------
// The per-utterance reductions (mean, peak, norms) need every tile of the utterance. Instead of separate finalise / apply
// passes, the CTA that completes an utterance's last tile (a per-utterance arrival counter) finalises it in place:
//   TAIL_AFFINE  out = normWav(y - mean(y), 0), optionally followed by the ISD scatter and its normWav (LnL, LnL -> ISD)
//   TAIL_SSI     out = aux + y * ||aux|| / (||y|| * 10^(snr/20))                                        (SSI)
enum { TAIL_NONE = 0, TAIL_AFFINE = 1, TAIL_SSI = 2 };
struct FirTail {
  int mode = TAIL_NONE;
  uint32_t* counters = nullptr;      // [B] arrival counters (zeroed by the launcher, left zero by the kernel)
  float* out = nullptr;              // [B][ld] final waveform
  const int32_t* isd_off = nullptr;  // TAIL_AFFINE: impulses (NULL = none); offsets are absolute into isd_idx / isd_fr
  const int32_t* isd_idx = nullptr;
  const double* isd_fr = nullptr;
  float g_sd = 0.f;
  const float* aux = nullptr;        // TAIL_SSI: the signal the noise is added to, [B][ld]
  const float* snr_db = nullptr;     // TAIL_SSI: [B]
  // the same tail for the sub-batch starting at utterance b0
  FirTail shifted(int b0, int ld) const {
    FirTail t = *this;
    if (t.counters) t.counters += b0;
    if (t.out) t.out += (size_t)b0 * ld;
    if (t.isd_off) t.isd_off += b0;
    if (t.aux) t.aux += (size_t)b0 * ld;
    if (t.snr_db) t.snr_db += b0;
    return t;
  }
};

// ---- kernel launchers shared between translation units (all asynchronous on `st`) ------------------
// FIR bank: y[u] = sum_f FIR(x[u] ** (pow_base + f*pow_step), taps of filter (u,f)); optional tile stats + ISD mask + tail.
int launch_fir_bank(const float* x, const int32_t* len, int B, int ld, const float* taps, const int32_t* tap_off,
                    int n_f, int pow_base, int pow_step, float* y, float* stats /*nullable*/,
                    const uint32_t* mask /*nullable*/, int mask_ld, const FirTail& tail, cudaStream_t st);

// Device-side planner, stage by stage (rb_devplan.cu); rb_devplan_draw runs all four for the whole batch. The pipelined host
// entry interleaves stages 2/3 of one chunk with the kernels of the previous chunk. With `snaps` (device, [B][625] words in
// numpy's state form, rb_mt.cuh) utterance u's stream starts at snaps[u] instead of np.random.seed(seeds[u]).
int devplan_begin(const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds, void* storage,
                  size_t storage_bytes, rb_plan* plan, cudaStream_t st, const uint32_t* snaps = nullptr);
int devplan_body(const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds, void* storage, int first,
                 int count, cudaStream_t st, const uint32_t* snaps = nullptr);
int devplan_apply(const rb_args* args, int algo, int B, int ld, const int32_t* len, void* storage, int first, int count,
                  cudaStream_t st);
int devplan_end(const rb_args* args, int algo, int B, int ld, void* storage, cudaStream_t st);
// np.random.permutation(len[u])[:off[u+1]-off[u]] -> out[off[u]...] for B rows of at most ld entries whose streams start at
// snaps[u]; `storage` holds shuffle_prefix_bytes(B, ld) bytes, 256-byte aligned.
size_t shuffle_prefix_bytes(int B, int ld);
int shuffle_prefix(int B, int ld, const int32_t* len, const uint32_t* snaps, const int32_t* off, int32_t* out, void* storage,
                   cudaStream_t st);

}  // namespace rb
