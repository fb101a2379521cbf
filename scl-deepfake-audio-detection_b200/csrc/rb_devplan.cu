// rb_devplan.cu -- device-side plan drawing for batches whose utterances are seeded independently
// (np.random.seed(seeds[u]) before utterance u: the benchmark's convention, SURVEY.md 8d).
//
// The reference draws every random parameter from numpy's legacy MT19937 stream
// (/root/reference/datautils/RawBoost.py:15,79,80,90). plans.py (numpy itself) is the contract and rb_planner.cpp is its
// bit-exact host replica; this file replays the SAME stream on the GPU so that a seeded batch needs no host work and no
// plan upload at all:
//
//   seeding          np.random.seed(int)            Knuth LCG fill of the 624-word state
//   uniform          low + (high-low) * double53    two 32-bit words per double, (a>>5, b>>6)
//   permutation(n)   arange + legacy shuffle        Fisher-Yates from the end, masked rejection on 32-bit words
//   rand(n)          double53
//   normal(0,1,n)    legacy polar Box-Muller
//
// Integer results (tap counts, impulse count, impulse positions) and the float64 impulse gains are bit-identical to
// numpy's: they only involve integer arithmetic and correctly rounded fp64 add/mul/div, issued without FMA contraction.
// Filter taps and SSI noise go through sin/cos/log/pow, where CUDA's fp64 libm and glibc may differ in the last ulp of
// the float64 value; after the float32 cast they agree to 1 ulp(fp32) (tests/test_gpu_parity.py).
//
// Kernels (all on the caller's stream, no host synchronisation):
//   plan_head_kernel     one warp per utterance: the first draws -> per-filter design parameters, tap counts, impulse count
//   scan_kernel          exclusive scan of the counts -> CSR offsets
//   plan_body_kernel     one warp per utterance, many per SM: the swap targets of the sequential shuffle (32 stream words per
//                        round, rejection fix-point by ballot) and its conflict-free groups, then the impulse gains / the SSI
//                        noise and draws
//   perm_apply_kernel    one warp per utterance with the permutation in shared memory (uint16, <= 65536 samples): applies
//                        the swaps group by group and emits the first n positions
//   design_kernel        one CTA per filter: windowed-sinc stages, cascade convolution, 1024-point FFT peak, gain, fp32 taps
#include <math.h>

#include <algorithm>
#include <string.h>

#include "rb_algo.h"
#include "rb_common.cuh"
#include "rb_mt.cuh"

namespace rb {

namespace {

constexpr int kNarrowMax = 65536;  // longest row whose permutation is held as uint16 in shared memory

// Draw one genNotchCoeffs parameter set (RawBoost.py:31-45) from stream words [w0, w0 + 2*(3*nBands+1)): returns K.
__device__ int draw_filter_params(const MtStream& s, int w0, const rb_args& a, double minG, double maxG, double* out) {
  int K = 0;
  for (int b = 0; b < a.nBands; ++b) {
    const double fc = mt_uniform(a.minF, a.maxF, mt_double(s.word(w0), s.word(w0 + 1)));
    const double bw = mt_uniform(a.minBW, a.maxBW, mt_double(s.word(w0 + 2), s.word(w0 + 3)));
    int c = (int)mt_uniform(a.minCoeff, a.maxCoeff, mt_double(s.word(w0 + 4), s.word(w0 + 5)));  // int() truncation
    w0 += 6;
    if (c % 2 == 0) c += 1;
    double f1 = __dsub_rn(fc, __dmul_rn(bw, 0.5)), f2 = __dadd_rn(fc, __dmul_rn(bw, 0.5));
    if (f1 <= 0) f1 = 1.0 / 1000;
    if (f2 >= a.fs / 2) f2 = __dsub_rn(a.fs / 2, 1.0 / 1000);
    out[3 * b + 0] = f1;
    out[3 * b + 1] = f2;
    out[3 * b + 2] = (double)c;
    K += c;
  }
  out[3 * a.nBands] = mt_uniform(minG, maxG, mt_double(s.word(w0), s.word(w0 + 1)));
  return K - (a.nBands - 1);
}

// ---- head: LnL design parameters + tap counts, ISD impulse count ----------------------------------------------------------
constexpr int kHeadWarps = 4;

__global__ void __launch_bounds__(32 * kHeadWarps)
plan_head_kernel(rb_args a, int algo, int B, const int32_t* __restrict__ len_arr, const uint32_t* __restrict__ seeds,
                 const uint32_t* __restrict__ snaps, double* __restrict__ lnl_params, int32_t* __restrict__ lnl_cnt, int32_t* __restrict__ isd_cnt) {
  __shared__ MtSmem sm[kHeadWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int u = blockIdx.x * kHeadWarps + warp;
  if (u >= B) return;
  MtStream s;
  s.sm = &sm[warp];
  if (snaps) s.load(snaps + (size_t)u * kMtSnapWords, lane);
  else s.seed(seeds[u], lane);
  const int per = 2 * filter_stride(a.nBands);  // stream words per filter
  if (algo_uses_lnl(algo)) {
    // filters are consumed in windows that fit the two tempered blocks
    const int fpw = max(1, min(kMtN / per, 32));  // filters per window, one lane each
    for (int f0 = 0; f0 < a.N_f; f0 += fpw) {
      const int nf = min(fpw, a.N_f - f0);
      if (lane < nf) {
        const int f = f0 + lane;
        const double minG = a.minG - (f >= 1 ? a.minBiasLinNonLin : 0.0);
        const double maxG = a.maxG - (f >= 1 ? a.maxBiasLinNonLin : 0.0);
        const size_t fi = (size_t)u * a.N_f + f;
        lnl_cnt[fi] = draw_filter_params(s, lane * per, a, minG, maxG, lnl_params + fi * filter_stride(a.nBands));
      }
      s.advance(nf * per, lane);
    }
  }
  if (algo_uses_isd(algo) && lane == 0) {
    const double beta = mt_uniform(0.0, a.P, mt_double(s.word(0), s.word(1)));
    isd_cnt[u] = (int)__dmul_rn((double)len_arr[u], __ddiv_rn(beta, 100.0));
  }
}

// ---- exclusive scan of n counts into n+1 offsets (single CTA; n is at most a few hundred thousand) -------------------------
__global__ void __launch_bounds__(1024)
scan_kernel(const int32_t* __restrict__ cnt, int n, int32_t* __restrict__ off) {
  __shared__ int32_t wsum[32];
  __shared__ int32_t carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + tid;
    const int32_t v = i < n ? cnt[i] : 0;
    int32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t y = __shfl_up_sync(kFull, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int32_t w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int32_t y = __shfl_up_sync(kFull, w, o);
        if (lane >= o) w += y;
      }
      wsum[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const int32_t before = carry + (warp ? wsum[warp - 1] : 0) + (x - v);
    if (i < n) off[i] = before;
    __syncthreads();
    if (tid == 1023) carry = before + v;
    __syncthreads();
  }
  if (tid == 0) off[n] = carry;
}

// ---- body: everything after the LnL draws -------------------------------------------------------------------------------
// numpy's legacy shuffle of arange(L) is sequential: for i = L-1 .. 1: j = random_interval(i); swap(x[i], x[j]), where
// random_interval rejects masked stream words > i. It is replayed in two kernels.
//
// plan_body_kernel (this one; one warp per utterance, many warps per SM, no permutation array) settles everything that does
// not depend on the array contents:
//   1. the swap targets j_i (shuffle_walk_warp, rb_mt.cuh), into jseq[step], step = L-1-i.
//   2. which consecutive steps may be applied together. Steps are taken in chunks of 32; inside a chunk, step t conflicts
//      with an earlier step s when they share the target (j_t == j_s) or when s targets t's own slot (j_s == i_t). A set bit
//      in cuts[chunk] starts a new conflict-free group.
// perm_apply_kernel (one warp per SM, the permutation as uint16 in shared memory) then only loads, swaps and stores group
// by group.
constexpr int kDupWords = 128;  // 4096-bit duplicate filter per warp (keeps 7 CTAs = 28 utterances per SM)
constexpr int kBodyWarps = 4;  // 30 KB of MT19937 state per CTA: up to 7 CTAs = 28 utterances in flight per SM

template <typename JT>  // uint16_t for rows of at most 65536 samples, uint32_t beyond
__device__ void shuffle_scan_warp(MtStream& s, int L, JT* __restrict__ jseq, uint32_t* __restrict__ cuts, uint32_t* dupset,
                                  int lane) {
  shuffle_walk_warp<true>(s, L, jseq, lane);
  __syncwarp();  // jseq was written by other lanes of this warp
  const uint32_t lt = (1u << lane) - 1u;
  const int nsteps = L - 1;
  // Conflicts are rare (7 % of the chunks) and MATCH.ANY is slow (about a hundred cycles of a per-SM unit each), so every
  // chunk first goes through an exact-negative filter: each step sets the bit of its target in a 4096-bit shared-memory
  // set (atomicOr returns the previous word: a set bit means another step of the chunk hashed to the same place) and a
  // vote tells whether any step targets one of the chunk's own slots. Only chunks that trip either test (hash collisions
  // included, ~12 %) take the exact MATCH / REDUX path. The targets of the next four chunks are already on their way from L2.
  constexpr int kAhead = 4;
  int jn[kAhead];
#pragma unroll
  for (int q = 0; q < kAhead; ++q) {
    const int k = q * 32 + lane;
    jn[q] = k < nsteps ? (int)jseq[k] : 0;
  }
  for (int c0 = 0; c0 * 32 < nsteps; c0 += kAhead) {
    int jj[kAhead];
#pragma unroll
    for (int q = 0; q < kAhead; ++q) {
      jj[q] = jn[q];
      const int k = (c0 + kAhead + q) * 32 + lane;
      jn[q] = k < nsteps ? (int)jseq[k] : 0;
    }
#pragma unroll
    for (int q = 0; q < kAhead; ++q) {
      const int c = c0 + q;
      if (c * 32 >= nsteps) break;
      const bool valid = c * 32 + lane < nsteps;
      const int i0 = (L - 1) - c * 32;  // slot of lane 0; lane t owns slot i0 - t
      const int j = jj[q];
      const bool hits_slot = valid && j > i0 - 32 && j != i0 - lane;  // targets the slot of lane i0 - j of this chunk
      const uint32_t old = valid ? atomicOr(dupset + ((j >> 5) & (kDupWords - 1)), 1u << (j & 31)) : 0u;
      const uint32_t suspicious = __ballot_sync(kFull, hits_slot || (valid && ((old >> (j & 31)) & 1u)));
      if (valid) atomicAnd(dupset + ((j >> 5) & (kDupWords - 1)), ~(1u << (j & 31)));  // leave the set empty again
      uint32_t cut = 0;
      if (suspicious) {
        int start = 0;
        for (;;) {
          const bool active = valid && lane >= start;
          const uint32_t same = __match_any_sync(kFull, active ? (uint32_t)j : (0x80000000u + (uint32_t)lane));
          uint32_t tbit = 0;
          if (active && j > i0 - 32 && j != i0 - lane) tbit = 1u << (i0 - j);
          const uint32_t tmap = __reduce_or_sync(kFull, tbit);
          const uint32_t badmask = __ballot_sync(kFull, active && (((same & lt) != 0u) || ((tmap >> lane) & 1u)));
          if (!badmask) break;
          start = __ffs(badmask) - 1;  // grows every time: the first active lane has nothing before it
          cut |= 1u << start;
        }
      }
      if (lane == 0) cuts[c] = cut;
    }
  }
}

template <typename JT>
__global__ void __launch_bounds__(32 * kBodyWarps)
plan_body_kernel(rb_args a, int algo, int B, int ld, int jld, const int32_t* __restrict__ len_arr,
                 const uint32_t* __restrict__ seeds, const uint32_t* __restrict__ snaps, const int32_t* __restrict__ isd_off, double* __restrict__ isd_fr, JT* __restrict__ jseq_all,
                 uint32_t* __restrict__ cuts_all, int cuts_ld, float* __restrict__ ssi_noise, double* __restrict__ ssi_params,
                 int32_t* __restrict__ ssi_cnt, float* __restrict__ ssi_snr) {
  __shared__ MtSmem msm[kBodyWarps];
  __shared__ uint32_t dupset[kBodyWarps][kDupWords];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int u = blockIdx.x * kBodyWarps + warp;
  if (u >= B) return;
  for (int w = lane; w < kDupWords; w += 32) dupset[warp][w] = 0u;
  __syncwarp();
  const int L = len_arr[u];
  MtStream s;
  s.sm = &msm[warp];
  if (snaps) s.load(snaps + (size_t)u * kMtSnapWords, lane);
  else s.seed(seeds[u], lane);
  if (algo_uses_lnl(algo)) s.skip(a.N_f * 2 * filter_stride(a.nBands), lane);
  if (algo_uses_isd(algo)) {
    s.advance(2, lane);  // beta (the head kernel turned it into the impulse count)
    const int beg = isd_off[u], n = isd_off[u + 1] - beg;
    shuffle_scan_warp(s, L, jseq_all + (size_t)u * jld, cuts_all + (size_t)u * cuts_ld, dupset[warp], lane);
    // f_r = (2*rand(n) - 1) * (2*rand(n) - 1)   (RawBoost.py:80)
    for (int pass = 0; pass < 2; ++pass) {
      for (int base = 0; base < n; base += 32) {
        const int m = min(32, n - base);
        if (lane < m) {
          const double r = __dsub_rn(__dmul_rn(2.0, mt_double(s.word(2 * lane), s.word(2 * lane + 1))), 1.0);
          double* dst = isd_fr + beg + base + lane;
          *dst = pass ? __dmul_rn(*dst, r) : r;
        }
        s.advance(2 * m, lane);
      }
    }
  }
  if (algo_uses_ssi(algo)) {
    // np.random.normal(0, 1, L): legacy polar Box-Muller; every attempt uses four words and yields two values
    float* row = ssi_noise + (size_t)u * ld;
    const uint32_t lt = (1u << lane) - 1u;
    int produced = 0;
    while (produced < L) {
      const double x1 = __dsub_rn(__dmul_rn(2.0, mt_double(s.word(4 * lane), s.word(4 * lane + 1))), 1.0);
      const double x2 = __dsub_rn(__dmul_rn(2.0, mt_double(s.word(4 * lane + 2), s.word(4 * lane + 3))), 1.0);
      const double r2 = __dadd_rn(__dmul_rn(x1, x1), __dmul_rn(x2, x2));
      const bool ok = !(r2 >= 1.0 || r2 == 0.0);
      const uint32_t okmask = __ballot_sync(kFull, ok);
      const int need = (L - produced + 1) >> 1;  // accepted attempts still needed
      const int rank = __popc(okmask & lt);
      const uint32_t last = __ballot_sync(kFull, ok && rank == need - 1);  // the attempt that completes the L values
      const int used = last ? __ffs(last) : 32;
      if (ok && rank < need) {
        const double f = sqrt(__ddiv_rn(__dmul_rn(-2.0, log(r2)), r2));
        const int o = produced + 2 * rank;
        row[o] = (float)__dmul_rn(f, x2);
        if (o + 1 < L) row[o + 1] = (float)__dmul_rn(f, x1);
      }
      produced += 2 * min(__popc(okmask), need);
      s.advance(4 * used, lane);
    }
    for (int k = L + lane; k < ld; k += 32) row[k] = 0.f;
    const int per = 2 * filter_stride(a.nBands);
    if (lane == 0) {
      ssi_cnt[u] = draw_filter_params(s, 0, a, a.minG, a.maxG, ssi_params + (size_t)u * filter_stride(a.nBands));
      ssi_snr[u] = (float)mt_uniform(a.SNRmin, a.SNRmax, mt_double(s.word(per), s.word(per + 1)));
    }
  }
}

// The swap targets and groups of a bare permutation whose stream starts at a snapshot (np.random.choice(..., replace=False)
// of an item, rb_items.cu): one warp per row, as plan_body_kernel.
template <typename JT>
__global__ void __launch_bounds__(32 * kBodyWarps)
shuffle_scan_kernel(int B, int jld, const int32_t* __restrict__ len_arr, const uint32_t* __restrict__ snaps, JT* __restrict__ jseq_all,
                    uint32_t* __restrict__ cuts_all, int cuts_ld) {
  __shared__ MtSmem msm[kBodyWarps];
  __shared__ uint32_t dupset[kBodyWarps][kDupWords];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int u = blockIdx.x * kBodyWarps + warp;
  if (u >= B) return;
  for (int w = lane; w < kDupWords; w += 32) dupset[warp][w] = 0u;
  __syncwarp();
  MtStream s;
  s.sm = &msm[warp];
  s.load(snaps + (size_t)u * kMtSnapWords, lane);
  shuffle_scan_warp(s, len_arr[u], jseq_all + (size_t)u * jld, cuts_all + (size_t)u * cuts_ld, dupset[warp], lane);
}

// ---- the swaps themselves: one warp per utterance, permutation in shared memory ------------------------------------------
// The targets and group boundaries stream in through a double-buffered shared-memory stage (cp.async, 1024 steps ahead), so
// the only latency on the critical path of a group is shared memory: load two slots, store two slots, __syncwarp.
constexpr int kStageSteps = 1024;  // steps per staged piece = 32 chunks

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

// Phases. Step k swaps slot i = L-1-k with a target j <= i and never looks above i again, so the live part of the array
// shrinks as the shuffle proceeds. The steps are therefore applied in up to four launches: phase p handles the steps whose
// slots lie below T_hi (rounded to whole 1024-step staging pieces) and keeps only T_hi entries in shared memory -- 128, 96,
// 64 and 32 KB -- so that 1, 2, 3 and 6 utterances per SM are in flight instead of one throughout (the kernel is bound by
// the latency of a single warp per utterance). The array travels between phases through `state` (global, L2-resident);
// every phase writes back all it holds, so slots finalised in an earlier phase keep their final value there.
constexpr int kJStride = kStageSteps + 32;       // uint16 entries per target staging buffer
constexpr int kCStride = kStageSteps / 32 + 4;   // uint32 entries per group-mask staging buffer
constexpr int kApplyStageBytes = 2 * kJStride * 2 + 2 * kCStride * 4;
static_assert((kJStride * 2) % 16 == 0 && (kCStride * 4) % 16 == 0 && kApplyStageBytes % 16 == 0, "cp.async alignment");

__device__ __forceinline__ int phase_first_step(int L, int T) {  // first step (multiple of 1024) whose slot is below T
  const int k = L - T;
  return k <= 0 ? 0 : (k + kStageSteps - 1) / kStageSteps * kStageSteps;
}

__global__ void __launch_bounds__(32)
perm_apply_kernel(int B, int jld, const int32_t* __restrict__ len_arr, const uint16_t* __restrict__ jseq_all,
                  const uint32_t* __restrict__ cuts_all, int cuts_ld, const int32_t* __restrict__ isd_off,
                  int32_t* __restrict__ isd_idx, uint16_t* __restrict__ state_all, int T_hi, int T_lo) {
  extern __shared__ __align__(16) unsigned char dyn[];
  // two staging buffers for targets and group masks, each with one chunk of padding for the one-ahead reads of the loop below
  uint16_t (*jbuf)[kJStride] = reinterpret_cast<uint16_t (*)[kJStride]>(dyn);
  uint32_t (*cbuf)[kCStride] = reinterpret_cast<uint32_t (*)[kCStride]>(dyn + 2 * kJStride * 2);
  uint16_t* perm = reinterpret_cast<uint16_t*>(dyn + kApplyStageBytes);
  const int u = blockIdx.x, lane = threadIdx.x;
  const int L = len_arr[u];
  const int beg = isd_off[u], n = isd_off[u + 1] - beg;
  if (n <= 0) return;  // no impulse: nothing of the permutation is used
  const bool last = T_lo <= 0;
  const int nsteps = max(L - 1, 0);
  const int kb = min(nsteps, phase_first_step(L, T_hi));                       // steps [kb, ke) belong to this phase
  const int ke = last ? nsteps : min(nsteps, phase_first_step(L, T_lo));
  if (kb >= ke && !last) return;  // nothing to do here; the array is created by the first phase that has steps
  const uint16_t* __restrict__ jseq = jseq_all + (size_t)u * jld;
  const uint32_t* __restrict__ cuts = cuts_all + (size_t)u * cuts_ld;
  uint16_t* __restrict__ state = state_all + (size_t)u * jld;
  const int live = L - kb;  // slots [0, live) are what this phase can touch (<= T_hi)
  const int p_begin = kb / kStageSteps, p_end = (ke + kStageSteps - 1) / kStageSteps;
  auto stage = [&](int piece) {  // rows are padded to whole pieces, so no bounds checks
    const uint16_t* src = jseq + (size_t)piece * kStageSteps;
#pragma unroll
    for (int q = 0; q < kStageSteps * 2 / 16 / 32; ++q) cp_async16(&jbuf[piece & 1][(q * 32 + lane) * 8], src + (q * 32 + lane) * 8);
    if (lane < kStageSteps / 32 / 4) cp_async16(&cbuf[piece & 1][lane * 4], cuts + (size_t)piece * (kStageSteps / 32) + lane * 4);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  if (p_begin < p_end) stage(p_begin);
  if (kb == 0) {  // first phase of this utterance: arange
    for (int k = 2 * lane; k < live; k += 64) *reinterpret_cast<uint32_t*>(perm + k) = (uint32_t)k | ((uint32_t)(k + 1) << 16);
  } else {        // the live slots as the previous phase left them: one cp.async group, all of it in flight at once
    for (int k = 8 * lane; k < live; k += 256) cp_async16(perm + k, state + k);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  const int nch_end = (ke + 31) >> 5;
  if (p_begin >= p_end) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
  }
  for (int piece = p_begin; piece < p_end; ++piece) {
    if (piece + 1 < p_end) {
      stage(piece + 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncwarp();
    const uint16_t* jb = jbuf[piece & 1] + lane;
    const uint32_t* cb = cbuf[piece & 1];
    const int c0 = piece * (kStageSteps / 32);
    const int cend = min(kStageSteps / 32, nch_end - c0);
    const int nfull = min(cend, (ke - c0 * 32) >> 5);  // chunks of this piece with all 32 steps
    uint16_t* slotp = perm + ((L - 1) - (c0 * 32 + lane));  // this lane's own slot; moves down 32 slots per chunk
    int jn = jb[0];
    uint32_t cn = cb[0];
    // Full chunks. The next chunk's target and group mask are fetched one iteration ahead; the common case -- no conflict
    // inside the chunk, 93 % of them -- is two loads and two stores per lane.
#pragma unroll 4
    for (int cc = 0; cc < nfull; ++cc) {
      const int j = jn;
      uint32_t cut = cn;
      jn = jb[(cc + 1) * 32];  // past the piece's last chunk this reads the buffer's own padding (never used)
      cn = cb[cc + 1];
      if (cut == 0u) {
        const uint16_t va = perm[j], vb = *slotp;
        perm[j] = vb;
        *slotp = va;
        __syncwarp();
      } else {
        int s0 = 0;
        for (;;) {
          const int s1 = cut ? __ffs(cut) - 1 : 32;
          const bool doit = lane >= s0 && lane < s1;
          uint16_t va = 0, vb = 0;
          if (doit) {
            va = perm[j];
            vb = *slotp;
          }
          if (doit) {
            perm[j] = vb;
            *slotp = va;
          }
          __syncwarp();
          if (!cut) break;
          cut &= cut - 1;
          s0 = s1;
        }
      }
      slotp -= 32;
    }
    if (nfull < cend) {  // the utterance's last, partial chunk (only the last phase can end inside a chunk)
      const int j = jn;
      uint32_t cut = cn;
      const int nvalid = ke - (c0 + nfull) * 32;
      int s0 = 0;
      for (;;) {
        const int s1 = cut ? min(__ffs(cut) - 1, nvalid) : nvalid;
        const bool doit = lane >= s0 && lane < s1;
        uint16_t va = 0, vb = 0;
        if (doit) {
          va = perm[j];
          vb = *slotp;
        }
        if (doit) {
          perm[j] = vb;
          *slotp = va;
        }
        __syncwarp();
        if (!cut) break;
        cut &= cut - 1;
        s0 = s1;
      }
    }
    __syncwarp();  // everyone is done with this stage buffer before it is refilled two pieces later
  }
  __syncwarp();
  if (!last) {  // hand the array on (whole pieces of 8 entries; the rows are padded)
    for (int k = 8 * lane; k < live; k += 256) *reinterpret_cast<uint4*>(state + k) = *reinterpret_cast<const uint4*>(perm + k);
    return;
  }
  // the first n slots: what this phase holds comes from shared memory, slots finalised earlier from the state array
  for (int k = lane; k < n; k += 32) isd_idx[beg + k] = (int32_t)(k < live ? perm[k] : __ldcg(state + k));
}

// ---- the swaps for rows longer than 65536 samples ------------------------------------------------------------------------
// Un-cropped utterances (the loaders apply RawBoost before the crop, asvspoof_2019_augall_3.py:105-117) run to ~200 k samples:
// the permutation no longer fits shared memory as uint16. It then lives in global memory as uint32 (L2 for the most part) and
// one warp per utterance applies the same conflict-free groups with L2 round trips instead of shared-memory ones. The walk is
// latency-bound (about one L2 round trip per 32 steps) but every utterance has its own warp, 32 warps per SM, so a batch of
// long rows still takes a small fraction of the time the FIR bank needs for them.
constexpr int kWideWarps = 4;

__global__ void __launch_bounds__(32 * kWideWarps)
perm_apply_wide_kernel(int B, int jld, const int32_t* __restrict__ len_arr, const uint32_t* __restrict__ jseq_all,
                       const uint32_t* __restrict__ cuts_all, int cuts_ld, const int32_t* __restrict__ isd_off,
                       int32_t* __restrict__ isd_idx, uint32_t* __restrict__ state_all) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int u = blockIdx.x * kWideWarps + warp;
  if (u >= B) return;
  const int L = len_arr[u];
  const int beg = isd_off[u], n = isd_off[u + 1] - beg;
  if (n <= 0) return;  // no impulse: nothing of the permutation is used
  const uint32_t* __restrict__ jseq = jseq_all + (size_t)u * jld;
  const uint32_t* __restrict__ cuts = cuts_all + (size_t)u * cuts_ld;
  uint32_t* perm = state_all + (size_t)u * jld;
  for (int k = lane; k < L; k += 32) __stcg(perm + k, (uint32_t)k);
  __syncwarp();
  const int nsteps = max(L - 1, 0);
  const int nch = (nsteps + 31) >> 5;
  uint32_t jn = (lane < nsteps) ? __ldcg(jseq + lane) : 0u;
  uint32_t cn = nch > 0 ? __ldcg(cuts) : 0u;
  for (int c = 0; c < nch; ++c) {
    const uint32_t j = jn;
    uint32_t cut = cn;
    const int k = c * 32 + lane;
    const bool valid = k < nsteps;
    if (c + 1 < nch) {  // next chunk's targets and group mask travel while this chunk is applied
      jn = (k + 32 < nsteps) ? __ldcg(jseq + k + 32) : 0u;
      cn = __ldcg(cuts + c + 1);
    }
    uint32_t* slotp = perm + ((L - 1) - k);
    int s0 = 0;
    for (;;) {
      const int s1 = cut ? __ffs(cut) - 1 : 32;
      const bool doit = valid && lane >= s0 && lane < s1;
      uint32_t va = 0u, vb = 0u;
      if (doit) {
        va = __ldcg(perm + j);
        vb = __ldcg(slotp);
      }
      if (doit) {
        __stcg(perm + j, vb);
        __stcg(slotp, va);
      }
      __syncwarp();
      if (!cut) break;
      cut &= cut - 1;
      s0 = s1;
    }
  }
  for (int k = lane; k < n; k += 32) isd_idx[beg + k] = (int32_t)__ldcg(perm + k);
}

// ---- genNotchCoeffs arithmetic (RawBoost.py:37-47), one CTA per filter, float64 -------------------------------------------
constexpr int kDesignThreads = 128;
constexpr int kDesignMaxK = 1024;   // freqz's 1024-point FFT path; longer cascades are refused by the host entry
constexpr int kDesignMaxStage = 256;   // taps of one firwin stage

__device__ __forceinline__ double sinc_pi(double x) {  // numpy.sinc
  if (x == 0.0) return 1.0;
  const double y = M_PI * x;
  return sin(y) / y;
}

__global__ void __launch_bounds__(kDesignThreads)
design_kernel(int nBands, double fs, int n_filters, const double* __restrict__ params, const int32_t* __restrict__ tap_off,
              float* __restrict__ taps) {
  __shared__ double stage[kDesignMaxStage];
  __shared__ double casc[2][kDesignMaxK];
  __shared__ double2 fft[1024];
  __shared__ double2 tw[512];
  __shared__ double red[kDesignThreads / 32];
  __shared__ double bc;
  const int fi = blockIdx.x, tid = threadIdx.x;
  if (fi >= n_filters) return;
  const double* p = params + (size_t)fi * (3 * nBands + 1);
  for (int k = tid; k < 512; k += kDesignThreads) {
    double sn, cs;
    sincospi(-(double)k / 512.0, &sn, &cs);
    tw[k] = make_double2(cs, sn);
  }
  int K = 1, curb = 0;
  if (tid == 0) casc[0][0] = 1.0;
  __syncthreads();
  const double nyq = fs / 2.0;
  for (int b = 0; b < nBands; ++b) {
    const double c1 = p[3 * b] / nyq, c2 = p[3 * b + 1] / nyq;
    const int c = (int)p[3 * b + 2];
    const double alpha = 0.5 * (c - 1);
    // scipy.signal.firwin(c, [f1, f2], window='hamming', fs=fs), pass_zero=True: bands [0, c1] and [c2, 1], DC gain 1
    for (int i = tid; i < c; i += kDesignThreads) {
      const double m = i - alpha;
      double v = c1 * sinc_pi(c1 * m);
      v -= 0.0;
      v += sinc_pi(m);
      v -= c2 * sinc_pi(c2 * m);
      const double win = (c == 1) ? 1.0 : 0.54 - 0.46 * cos(2.0 * M_PI * i / (c - 1));
      stage[i] = v * win;
    }
    __syncthreads();
    if (tid == 0) {
      double dc = 0.0;
      for (int i = 0; i < c; ++i) dc += stage[i];
      bc = dc;
    }
    __syncthreads();
    const double dc = bc;
    for (int i = tid; i < c; i += kDesignThreads) stage[i] /= dc;
    __syncthreads();
    const double* old = casc[curb];
    double* nw = casc[curb ^ 1];
    const int Kn = K + c - 1;
    for (int k = tid; k < Kn; k += kDesignThreads) {
      double acc = 0.0;
      const int i0 = max(0, k - (K - 1)), i1 = min(c - 1, k);
      for (int i = i0; i <= i1; ++i) acc += stage[i] * old[k - i];
      nw[k] = acc;
    }
    __syncthreads();
    K = Kn;
    curb ^= 1;
  }
  const double* bcoef = casc[curb];
  // peak of |H| on freqz's default grid: 512 points on [0, pi) = the first half of a 1024-point FFT
  for (int i = tid; i < 1024; i += kDesignThreads) {
    const int r = (int)(__brev((unsigned)i) >> 22);
    fft[r] = make_double2(i < K ? bcoef[i] : 0.0, 0.0);
  }
  __syncthreads();
  for (int len = 2; len <= 1024; len <<= 1) {
    const int half = len >> 1, step = 1024 / len;
    for (int q = tid; q < 512; q += kDesignThreads) {
      const int grp = q / half, k = q - grp * half;
      const int i0 = grp * len + k, i1 = i0 + half;
      const double2 w = tw[k * step], uu = fft[i0], vv = fft[i1];
      const double2 t = make_double2(vv.x * w.x - vv.y * w.y, vv.x * w.y + vv.y * w.x);
      fft[i0] = make_double2(uu.x + t.x, uu.y + t.y);
      fft[i1] = make_double2(uu.x - t.x, uu.y - t.y);
    }
    __syncthreads();
  }
  double best = 0.0;
  for (int i = tid; i < 512; i += kDesignThreads) best = fmax(best, hypot(fft[i].x, fft[i].y));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(kFull, best, o));
  if ((tid & 31) == 0) red[tid >> 5] = best;
  __syncthreads();
  if (tid == 0) {
    double m = red[0];
    for (int w = 1; w < kDesignThreads / 32; ++w) m = fmax(m, red[w]);
    bc = m;
  }
  __syncthreads();
  const double peak = bc;
  const double g = pow(10.0, p[3 * nBands] / 20.0);
  float* out = taps + tap_off[fi];
  for (int k = tid; k < K; k += kDesignThreads) out[k] = (float)((g * bcoef[k]) / peak);
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// swap targets, group masks and the permutation handed between the phases of perm_apply_kernel, for B rows of at most ld
struct ShuffleLayout {
  size_t jseq, cuts, state, bytes;
  int jld, cuts_ld;
};

ShuffleLayout shuffle_layout(int B, int ld) {
  ShuffleLayout l{};
  l.jld = (int)align_up((size_t)ld, kStageSteps);  // rows padded to whole staging pieces of perm_apply_kernel
  l.cuts_ld = l.jld / 32;
  const size_t jbytes = ld > kNarrowMax ? 4 : 2;   // swap targets / permutation entries: uint16 up to 65536 samples, uint32 beyond
  l.jseq = 0;
  l.cuts = align_up((size_t)B * l.jld * jbytes, 256);
  l.state = l.cuts + align_up((size_t)B * l.cuts_ld * 4, 256);
  l.bytes = l.state + align_up((size_t)B * l.jld * jbytes, 256);
  return l;
}

struct DevPlanLayout {
  size_t lnl_params, lnl_cnt, lnl_off, lnl_taps, isd_cnt, isd_off, isd_idx, isd_fr, isd_jseq, isd_cuts, isd_state, ssi_noise, ssi_params,
      ssi_cnt, ssi_off, ssi_taps, ssi_snr, bytes;
  int jld, cuts_ld;
};

int max_taps(const rb_args& a) { return a.nBands * ((int)ceil(a.maxCoeff > a.minCoeff ? a.maxCoeff : a.minCoeff) + 1); }

DevPlanLayout layout(const rb_args& a, int algo, int B, int ld) {
  DevPlanLayout l{};
  size_t off = 0;
  auto take = [&](size_t n) {
    const size_t r = off;
    off += align_up(n, 256);
    return r;
  };
  const bool lnl = algo_uses_lnl(algo);
  const bool isd = algo_uses_isd(algo);
  const bool ssi = algo_uses_ssi(algo);
  const size_t stride = 3 * (size_t)a.nBands + 1, kmax = (size_t)max_taps(a);
  const size_t nl = lnl ? (size_t)B * a.N_f : 0;
  l.lnl_params = take(nl * stride * 8);
  l.lnl_cnt = take(nl * 4);
  l.lnl_off = take(lnl ? (nl + 1) * 4 : 0);
  l.lnl_taps = take(nl * kmax * 4);
  l.isd_cnt = take(isd ? (size_t)B * 4 : 0);
  l.isd_off = take(isd ? (size_t)(B + 1) * 4 : 0);
  const size_t nmax = isd ? (size_t)B * ((size_t)((double)ld * a.P / 100.0) + 1) : 0;
  l.isd_idx = take(nmax * 4);
  l.isd_fr = take(nmax * 8);
  const ShuffleLayout sl = shuffle_layout(B, ld);
  l.jld = sl.jld;
  l.cuts_ld = sl.cuts_ld;
  const size_t shuffle = take(isd ? sl.bytes : 0);
  l.isd_jseq = shuffle + sl.jseq;
  l.isd_cuts = shuffle + sl.cuts;
  l.isd_state = shuffle + sl.state;
  l.ssi_noise = take(ssi ? (size_t)B * ld * 4 : 0);
  l.ssi_params = take(ssi ? (size_t)B * stride * 8 : 0);
  l.ssi_cnt = take(ssi ? (size_t)B * 4 : 0);
  l.ssi_off = take(ssi ? (size_t)(B + 1) * 4 : 0);
  l.ssi_taps = take(ssi ? (size_t)B * kmax * 4 : 0);
  l.ssi_snr = take(ssi ? (size_t)B * 4 : 0);
  l.bytes = off;
  return l;
}

bool args_ok(const rb_args& a) {
  if (a.N_f < 1 || a.nBands < 1 || a.nBands > 100) return false;
  if (!(a.fs > 0) || !(a.P >= 0) || a.P > 100) return false;
  const double cmax = a.maxCoeff > a.minCoeff ? a.maxCoeff : a.minCoeff, cmin = a.maxCoeff > a.minCoeff ? a.minCoeff : a.maxCoeff;
  if (cmin < 1 || cmax + 1 > kDesignMaxStage) return false;
  if (max_taps(a) > kDesignMaxK) return false;
  return true;
}

}  // namespace

}  // namespace rb

using namespace rb;

extern "C" {

size_t rb_devplan_bytes(const rb_args* args, int algo, int B, int ld) {
  if (!args || B <= 0 || ld <= 0 || !args_ok(*args)) return 0;
  return layout(*args, algo, B, ld).bytes;
}

int rb_devplan_draw(const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds, void* storage,
                    size_t storage_bytes, rb_plan* plan, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int rc = devplan_begin(args, algo, B, ld, len, seeds, storage, storage_bytes, plan, st);
  if (rc != RB_OK || B == 0 || ld == 0) return rc;
  if ((rc = devplan_body(args, algo, B, ld, len, seeds, storage, 0, B, st)) != RB_OK) return rc;
  if ((rc = devplan_apply(args, algo, B, ld, len, storage, 0, B, st)) != RB_OK) return rc;
  return devplan_end(args, algo, B, ld, storage, st);
}

}  // extern "C"

namespace rb {

// Stage 1: validation, first draws of every utterance, CSR offsets of the LnL taps and the impulses, LnL filter design.
// Fills *plan with device pointers into `storage` (their contents are complete once all four stages have run).
int devplan_begin(const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds, void* storage,
                  size_t storage_bytes, rb_plan* plan, cudaStream_t st, const uint32_t* snaps) {
  if (!args || !plan || B < 0 || ld < 0) return RB_ERR_INVALID_ARG;
  memset(plan, 0, sizeof(*plan));
  const bool lnl = algo_uses_lnl(algo);
  const bool isd = algo_uses_isd(algo);
  const bool ssi = algo_uses_ssi(algo);
  plan->n_f = lnl ? args->N_f : 0;
  plan->g_sd = (float)args->g_sd;
  if (B == 0 || ld == 0 || !(lnl || isd || ssi)) return RB_OK;
  if (!len || !(seeds || snaps)) return RB_ERR_INVALID_ARG;
  if (!args_ok(*args)) return RB_ERR_UNSUPPORTED;
  if (isd && ld > (1 << 30)) return RB_ERR_UNSUPPORTED;
  if (ld % 4 != 0) return RB_ERR_ALIGNMENT;
  if (!storage || ((uintptr_t)storage & 255u)) return storage ? RB_ERR_ALIGNMENT : RB_ERR_WORKSPACE;
  const DevPlanLayout l = layout(*args, algo, B, ld);
  if (l.bytes > storage_bytes) return RB_ERR_WORKSPACE;
  char* d = (char*)storage;
  const int nl = lnl ? B * args->N_f : 0;
  plan_head_kernel<<<(B + kHeadWarps - 1) / kHeadWarps, 32 * kHeadWarps, 0, st>>>(
      *args, algo, B, len, seeds, snaps, (double*)(d + l.lnl_params), (int32_t*)(d + l.lnl_cnt), (int32_t*)(d + l.isd_cnt));
  RB_LAUNCH_CHECK();
  if (isd) {
    scan_kernel<<<1, 1024, 0, st>>>((const int32_t*)(d + l.isd_cnt), B, (int32_t*)(d + l.isd_off));
    RB_LAUNCH_CHECK();
    plan->isd_off = (const int32_t*)(d + l.isd_off);
    plan->isd_idx = (const int32_t*)(d + l.isd_idx);
    plan->isd_fr = (const double*)(d + l.isd_fr);
  }
  if (lnl) {
    scan_kernel<<<1, 1024, 0, st>>>((const int32_t*)(d + l.lnl_cnt), nl, (int32_t*)(d + l.lnl_off));
    RB_LAUNCH_CHECK();
    design_kernel<<<nl, kDesignThreads, 0, st>>>(args->nBands, args->fs, nl, (const double*)(d + l.lnl_params),
                                                 (const int32_t*)(d + l.lnl_off), (float*)(d + l.lnl_taps));
    RB_LAUNCH_CHECK();
    plan->lnl_taps = (const float*)(d + l.lnl_taps);
    plan->lnl_tap_off = (const int32_t*)(d + l.lnl_off);
  }
  if (ssi) {
    plan->ssi_noise = (const float*)(d + l.ssi_noise);
    plan->ssi_taps = (const float*)(d + l.ssi_taps);
    plan->ssi_tap_off = (const int32_t*)(d + l.ssi_off);
    plan->ssi_snr_db = (const float*)(d + l.ssi_snr);
  }
  return RB_OK;
}

// Stage 2, utterances [first, first+count): the rest of the stream (swap targets and groups, impulse gains, SSI draws).
int devplan_body(const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds, void* storage, int first,
                 int count, cudaStream_t st, const uint32_t* snaps) {
  if (!(algo_uses_isd(algo) || algo_uses_ssi(algo)) || count <= 0) return RB_OK;
  const DevPlanLayout l = layout(*args, algo, B, ld);
  char* d = (char*)storage;
  const size_t stride = 3 * (size_t)args->nBands + 1;
  const unsigned grid = (count + kBodyWarps - 1) / kBodyWarps;
  const uint32_t* sd = seeds ? seeds + first : nullptr;
  const uint32_t* sn = snaps ? snaps + (size_t)first * kMtSnapWords : nullptr;
  if (ld > kNarrowMax)
    plan_body_kernel<uint32_t><<<grid, 32 * kBodyWarps, 0, st>>>(
        *args, algo, count, ld, l.jld, len + first, sd, sn, (const int32_t*)(d + l.isd_off) + first, (double*)(d + l.isd_fr),
        (uint32_t*)(d + l.isd_jseq) + (size_t)first * l.jld, (uint32_t*)(d + l.isd_cuts) + (size_t)first * l.cuts_ld, l.cuts_ld,
        (float*)(d + l.ssi_noise) + (size_t)first * ld, (double*)(d + l.ssi_params) + (size_t)first * stride,
        (int32_t*)(d + l.ssi_cnt) + first, (float*)(d + l.ssi_snr) + first);
  else
    plan_body_kernel<uint16_t><<<grid, 32 * kBodyWarps, 0, st>>>(
        *args, algo, count, ld, l.jld, len + first, sd, sn, (const int32_t*)(d + l.isd_off) + first, (double*)(d + l.isd_fr),
        (uint16_t*)(d + l.isd_jseq) + (size_t)first * l.jld, (uint32_t*)(d + l.isd_cuts) + (size_t)first * l.cuts_ld, l.cuts_ld,
        (float*)(d + l.ssi_noise) + (size_t)first * ld, (double*)(d + l.ssi_params) + (size_t)first * stride,
        (int32_t*)(d + l.ssi_cnt) + first, (float*)(d + l.ssi_snr) + first);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

// Apply the swaps of `count` rows (stride ld, padded to jld / cuts_ld) and emit the first off[u+1]-off[u] entries of row u's
// permutation to idx[off[u]...].
int launch_perm_apply(int count, int ld, int jld, int cuts_ld, const int32_t* len, const void* jseq, const uint32_t* cuts,
                      const int32_t* off, int32_t* idx, void* state, cudaStream_t st) {
  if (ld > kNarrowMax) {
    perm_apply_wide_kernel<<<(count + kWideWarps - 1) / kWideWarps, 32 * kWideWarps, 0, st>>>(
        count, jld, len, (const uint32_t*)jseq, cuts, cuts_ld, off, idx, (uint32_t*)state);
    RB_LAUNCH_CHECK();
    return RB_OK;
  }
  static const int kPhaseT[5] = {65536, 49152, 32768, 16384, 0};
  RB_CUDA(cudaFuncSetAttribute(perm_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  RB_CUDA(cudaFuncSetAttribute(perm_apply_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  for (int ph = 0; ph < 4; ++ph) {
    const int T_hi = kPhaseT[ph], T_lo = kPhaseT[ph + 1];
    if (T_lo >= ld) continue;  // no utterance of this batch has slots that high
    const size_t entries = (size_t)std::min(T_hi, (ld + 7) / 8 * 8) + 8;  // + the uint4 tail of the state copy
    const size_t smem = kApplyStageBytes + align_up(entries * 2, 16);
    if (smem > 227 * 1024) return RB_ERR_UNSUPPORTED;
    perm_apply_kernel<<<count, 32, smem, st>>>(count, jld, len, (const uint16_t*)jseq, cuts, cuts_ld, off, idx, (uint16_t*)state,
                                              T_hi, T_lo);
    RB_LAUNCH_CHECK();
  }
  return RB_OK;
}

// Stage 3, utterances [first, first+count): apply the swaps, emit the impulse positions.
int devplan_apply(const rb_args* args, int algo, int B, int ld, const int32_t* len, void* storage, int first, int count,
                  cudaStream_t st) {
  if (!algo_uses_isd(algo) || count <= 0) return RB_OK;
  const DevPlanLayout l = layout(*args, algo, B, ld);
  char* d = (char*)storage;
  const size_t jbytes = ld > kNarrowMax ? 4 : 2;
  return launch_perm_apply(count, ld, l.jld, l.cuts_ld, len + first, d + l.isd_jseq + (size_t)first * l.jld * jbytes,
                           (const uint32_t*)(d + l.isd_cuts) + (size_t)first * l.cuts_ld, (const int32_t*)(d + l.isd_off) + first,
                           (int32_t*)(d + l.isd_idx), d + l.isd_state + (size_t)first * l.jld * jbytes, st);
}

size_t shuffle_prefix_bytes(int B, int ld) { return B > 0 && ld > 0 ? shuffle_layout(B, ld).bytes : 0; }

// np.random.permutation(len[u])[:off[u+1]-off[u]] -> out[off[u]...] for B rows whose streams start at snapshots[u].
int shuffle_prefix(int B, int ld, const int32_t* len, const uint32_t* snaps, const int32_t* off, int32_t* out, void* storage,
                   cudaStream_t st) {
  if (B <= 0 || ld <= 0) return RB_OK;
  const ShuffleLayout l = shuffle_layout(B, ld);
  char* d = (char*)storage;
  const unsigned grid = (B + kBodyWarps - 1) / kBodyWarps;
  if (ld > kNarrowMax)
    shuffle_scan_kernel<uint32_t><<<grid, 32 * kBodyWarps, 0, st>>>(B, l.jld, len, snaps, (uint32_t*)(d + l.jseq),
                                                                   (uint32_t*)(d + l.cuts), l.cuts_ld);
  else
    shuffle_scan_kernel<uint16_t><<<grid, 32 * kBodyWarps, 0, st>>>(B, l.jld, len, snaps, (uint16_t*)(d + l.jseq),
                                                                   (uint32_t*)(d + l.cuts), l.cuts_ld);
  RB_LAUNCH_CHECK();
  return launch_perm_apply(B, ld, l.jld, l.cuts_ld, len, d + l.jseq, (const uint32_t*)(d + l.cuts), off, out, d + l.state, st);
}

// Stage 4 (after stage 2 of ALL utterances): CSR offsets and design of the SSI filters.
int devplan_end(const rb_args* args, int algo, int B, int ld, void* storage, cudaStream_t st) {
  if (!algo_uses_ssi(algo) || B <= 0) return RB_OK;
  const DevPlanLayout l = layout(*args, algo, B, ld);
  char* d = (char*)storage;
  scan_kernel<<<1, 1024, 0, st>>>((const int32_t*)(d + l.ssi_cnt), B, (int32_t*)(d + l.ssi_off));
  RB_LAUNCH_CHECK();
  design_kernel<<<B, kDesignThreads, 0, st>>>(args->nBands, args->fs, B, (const double*)(d + l.ssi_params),
                                              (const int32_t*)(d + l.ssi_off), (float*)(d + l.ssi_taps));
  RB_LAUNCH_CHECK();
  return RB_OK;
}

}  // namespace rb
