// rb_mt.cuh -- numpy's legacy MT19937 stream replayed by one warp (shared by the device planner and the item walk).
//
//   seeding          np.random.seed(int)            Knuth LCG fill of the 624-word state
//   uniform          low + (high-low) * double53    two 32-bit words per double, (a>>5, b>>6)
//   permutation(n)   arange + legacy shuffle        Fisher-Yates from the end, masked rejection on 32-bit words
//
// A stream can also start from, and be saved to, numpy's own state form (RandomState.get_state()[1:3]): key[624], the raw
// words of the current block, and pos, the index of the next word (624: the block is used up). Such a snapshot is 625 words.
#pragma once
#include <stdint.h>

namespace rb {

namespace {

constexpr int kMtN = 624, kMtM = 397;
constexpr int kMtSnapWords = kMtN + 1;  // key[624], pos
constexpr uint32_t kFull = 0xffffffffu;

// ---- MT19937, one warp per stream, state and two tempered blocks in shared memory ------------------------------------
struct MtSmem {
  uint32_t key[kMtN];
  uint32_t blk[2][kMtN];
};

__device__ __forceinline__ uint32_t mt_twist(uint32_t a, uint32_t b, uint32_t far) {
  const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
  return far ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908b0dfu);
}

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= (y >> 11);
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= (y >> 18);
  return y;
}

// exact inverse of mt_temper
__device__ __forceinline__ uint32_t mt_untemper(uint32_t y) {
  y ^= (y >> 18);
  y ^= (y << 15) & 0xefc60000u;  // self-inverse: the shifted mask has no bit inside the mask
  uint32_t x = y;
#pragma unroll
  for (int k = 0; k < 4; ++k) x = y ^ ((x << 7) & 0x9d2c5680u);  // 7 more correct low bits per round
  return x ^ (x >> 11) ^ (x >> 22);
}

// Advance the state by one block (624 words) and temper it into `out`. Warp-cooperative, three dependency phases.
__device__ void mt_next_block(uint32_t* key, uint32_t* out, int lane) {
  uint32_t v[8];
  // phase 1: i in [0, 227) reads old key[i], key[i+1], key[i+397]
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int i = c * 32 + lane;
    if (i < kMtN - kMtM) v[c] = mt_twist(key[i], key[i + 1], key[i + kMtM]);
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int i = c * 32 + lane;
    if (i < kMtN - kMtM) key[i] = v[c];
  }
  __syncwarp();
  // phase 2: i in [227, 454) reads new key[i-227], old key[i], key[i+1]
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int i = (kMtN - kMtM) + c * 32 + lane;
    if (i < 2 * (kMtN - kMtM)) v[c] = mt_twist(key[i], key[i + 1], key[i - (kMtN - kMtM)]);
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int i = (kMtN - kMtM) + c * 32 + lane;
    if (i < 2 * (kMtN - kMtM)) key[i] = v[c];
  }
  __syncwarp();
  // phase 3: i in [454, 623) reads new key[i-227], old key[i], key[i+1]
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const int i = 2 * (kMtN - kMtM) + c * 32 + lane;
    if (i < kMtN - 1) v[c] = mt_twist(key[i], key[i + 1], key[i - (kMtN - kMtM)]);
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const int i = 2 * (kMtN - kMtM) + c * 32 + lane;
    if (i < kMtN - 1) key[i] = v[c];
  }
  __syncwarp();
  if (lane == 0) key[kMtN - 1] = mt_twist(key[kMtN - 1], key[0], key[kMtM - 1]);
  __syncwarp();
#pragma unroll
  for (int c = 0; c < 20; ++c) {
    const int i = c * 32 + lane;
    if (i < kMtN) out[i] = mt_temper(key[i]);
  }
  __syncwarp();
}

// The stream as the warp sees it: the current and the next block are always tempered, so any window of up to 624 words
// starting at the read position can be addressed without synchronisation. `key` holds the raw words of the next block.
struct MtStream {
  MtSmem* sm;
  int cur;  // which blk[] holds the current block
  int pos;  // read position inside it, 0..623

  __device__ void seed(uint32_t s, int lane) {
    if (lane == 0) {
      for (int i = 0; i < kMtN; ++i) {
        sm->key[i] = s;
        s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i + 1u;
      }
    }
    __syncwarp();
    mt_next_block(sm->key, sm->blk[0], lane);
    mt_next_block(sm->key, sm->blk[1], lane);
    cur = 0;
    pos = 0;
  }
  // start from a snapshot in numpy's form: temper key into the current block (twisting first when pos == 624), then twist
  // once more for the next block. pos is clamped to 0..624, so that a malformed snapshot cannot address outside the blocks.
  __device__ void load(const uint32_t* __restrict__ snap, int lane) {
    for (int i = lane; i < kMtN; i += 32) sm->key[i] = snap[i];
    const int p = min(max((int)snap[kMtN], 0), kMtN);
    __syncwarp();
    if (p >= kMtN) {
      mt_next_block(sm->key, sm->blk[0], lane);
    } else {
      for (int i = lane; i < kMtN; i += 32) sm->blk[0][i] = mt_temper(sm->key[i]);
      __syncwarp();
    }
    mt_next_block(sm->key, sm->blk[1], lane);
    cur = 0;
    pos = p >= kMtN ? 0 : p;
  }
  // save the read position in numpy's form; pos is 0..623 (a used-up block is written as the next block at 0)
  __device__ void store(uint32_t* __restrict__ snap, int lane) const {
    for (int i = lane; i < kMtN; i += 32) snap[i] = mt_untemper(sm->blk[cur][i]);
    if (lane == 0) snap[kMtN] = (uint32_t)pos;
  }
  // word k (0 <= k < 624) after the read position
  __device__ __forceinline__ uint32_t word(int k) const {
    const int idx = pos + k;
    return idx < kMtN ? sm->blk[cur][idx] : sm->blk[cur ^ 1][idx - kMtN];
  }
  // consume n <= 624 words
  __device__ __forceinline__ void advance(int n, int lane) {
    pos += n;
    if (pos >= kMtN) {
      pos -= kMtN;
      __syncwarp();
      mt_next_block(sm->key, sm->blk[cur], lane);  // the exhausted block becomes the one after next
      cur ^= 1;
    }
  }
  __device__ void skip(int n, int lane) {
    while (n > 0) {
      const int s = n < kMtN ? n : kMtN;
      advance(s, lane);
      n -= s;
    }
  }
};

// numpy legacy rk_double from two stream words
__device__ __forceinline__ double mt_double(uint32_t wa, uint32_t wb) {
  const int32_t a = (int32_t)(wa >> 5), b = (int32_t)(wb >> 6);
  return __ddiv_rn(__dadd_rn(__dmul_rn((double)a, 67108864.0), (double)b), 9007199254740992.0);
}
// np.random.uniform(low, high): low + (high - low) * double, two roundings (no FMA contraction)
__device__ __forceinline__ double mt_uniform(double lo, double hi, double d) { return __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), d)); }

// per-filter design parameters: [f1, f2, c] x nBands, then G  -> 3*nBands + 1 doubles, drawn from twice as many words
__device__ __forceinline__ int filter_stride(int nBands) { return 3 * nBands + 1; }

// The stream words of numpy's legacy shuffle of arange(L): for i = L-1 .. 1: j = random_interval(i), which rejects masked
// words > i. A round looks at the next 32 stream words; word t is accepted iff (w_t & mask) <= i - (#accepted before t). The
// ballot fix-point settles lane t after at most t+1 iterations (lane 0 is exact at once), in practice after two. Accepted lanes
// are the consecutive steps i, i-1, ...; with kRecord their targets go to jseq[step], step = L-1-i. Without it the walk only
// consumes the words.
// Fast round: a word with v > i is rejected and one with v <= i - 31 accepted whatever A (A <= 31), so when no word lies in
// between, the first ballot is exact; when moreover at least 32 steps are left under the mask, all 32 words are consumed. For
// large masks that is almost every round, and it takes the fix-point's and the region's ballots off the round's critical path.
template <bool kRecord, typename JT>
__device__ __forceinline__ void shuffle_walk_warp(MtStream& s, int L, JT* __restrict__ jseq, int lane) {
  const uint32_t lt = (1u << lane) - 1u;
  int i = L - 1;
  while (i >= 1) {
    uint32_t mask = (uint32_t)i;
    mask |= mask >> 1;
    mask |= mask >> 2;
    mask |= mask >> 4;
    mask |= mask >> 8;
    mask |= mask >> 16;
    const int lo = (int)(mask >> 1) + 1;  // smallest i that uses this mask
    while (i >= lo) {
      const int v = (int)(s.word(lane) & mask);
      uint32_t acc = __ballot_sync(kFull, v <= i);
      const uint32_t unsure = __ballot_sync(kFull, v <= i && v > i - 31);
      if (unsure == 0 && i - lo + 1 >= 32) {
        if (kRecord && ((acc >> lane) & 1u)) jseq[(L - 1) - (i - __popc(acc & lt))] = (JT)v;
        i -= __popc(acc);
        s.advance(32, lane);
        continue;
      }
      int A;
      for (;;) {
        A = __popc(acc & lt);
        const uint32_t acc2 = __ballot_sync(kFull, v <= i - A);
        if (acc2 == acc) break;
        acc = acc2;
      }
      const int R = i - lo + 1;                                  // steps left under this mask
      const uint32_t in_region = __ballot_sync(kFull, A < R);    // a prefix of the lanes: the words this mask consumes
      if (kRecord) {
        const bool valid = ((acc >> lane) & 1u) && (A < R);
        if (valid) jseq[(L - 1) - (i - A)] = (JT)v;
      }
      i -= __popc(acc & in_region);
      s.advance(__popc(in_region), lane);
    }
  }
}

}  // namespace

}  // namespace rb
