// rb_items.cu -- whole Dataset_for items (asvspoof_2019_augall_3.py:103-146, RawBoost12 with online_aug) for a batch of items,
// either each seeded on its own (np.random.seed(seeds[g]) before item g, as a reproducible loader does per __getitem__) or
// sharing numpy's running stream (__getitem__ called for them one after another with no seed in between, as the reference's
// loader does).
//
// Item g consumes its stream in this order: RawBoost (algo 5) on every vocoded copy in vocoder order, then on the anchor --
// each of them N_f LnL parameter sets, ISD beta, permutation(L), rand(n) twice -- then np.random.choice(others, n_add,
// replace=False), which legacy numpy computes as permutation(N-1)[:n_add] mapped through `others` (v -> v + (v >= idx)),
// then the shared crop int(rand() * (L_anchor - trim)), drawn only when L_anchor >= trim.
//
// Two passes:
//   the walk             walk_item below, for one item on one warp: counts the item's words only (the shuffles with the ballot
//                        fix-point of shuffle_walk_warp), stores a snapshot of the stream (numpy's state form) at the start of
//                        every RawBoost utterance and of the choice, and draws the crop start. Two kernels run it:
//     items_walk_kernel         one warp per seeded item: seeds the stream, walks the item
//     items_stream_walk_kernel  one warp per running stream: loads the stream's state, walks its items in order, item k+1
//                               starting where item k ended, and stores the final state
//   then the per-utterance planner (rb_devplan.cu) runs unchanged over the G*(nvoc+1) utterances from their snapshots, and
//   shuffle_prefix applies the choice permutations.
//   items_rows_kernel    the batch's source rows in the corpus, their lengths, the view table of the assembly, the label vector
//   items_gather_kernel  one CTA per batch row: corpus row -> batch row (rb_items_run / rb_items_stream_run only)
//   items_gather_packed_kernel  the same from a packed corpus (the _packed run entries): float32 or PCM16 rows from 16-byte
//                        chunk boundaries, in device memory or in page-locked host memory
// The run entries then finish with rb_process(5) and rb_multiview_assemble_ex, exactly as ItemBatcher does; the padded and the
// packed entries share all of it and differ only in the gather they launch.
//
// Corpus layout: rows [R, ld], R = N * (1 + nvoc); row idx is bona fide utterance idx, row N + idx*nvoc + v is vocoder v's copy.
// A packed corpus has the same rows, each at its own length.
// Batch layout (ItemBatcher's): rows g*(nvoc+1) + v hold item g's vocoded copies (v < nvoc) and its anchor (v = nvoc); rows
// G*(nvoc+1) + g*n_add + k hold its additional bona fide utterances (not augmented).
#include <limits.h>
#include <string.h>

#include <algorithm>

#include "rb_common.cuh"
#include "rb_mt.cuh"

namespace rb {
namespace {

constexpr int kWalkWarps = 4;  // 30 KB of MT19937 state per CTA, as plan_body_kernel

__device__ __forceinline__ int clamp_index(int idx, int N) { return (idx >= 0 && idx < N) ? idx : 0; }

// Every draw of item g from the warp's stream `s`, which stands at the item's first word: the utterance snapshots, the choice
// snapshot, choice_len / choice_off and the crop start. Leaves `s` after the item's last word.
__device__ __forceinline__ void walk_item(const rb_args& a, MtStream& s, int g, int G, int nvoc, int n_add, int N, int trim,
                                          const int32_t* __restrict__ corpus_len, const int32_t* __restrict__ indices,
                                          uint32_t* __restrict__ snaps, uint32_t* __restrict__ csnaps, int32_t* __restrict__ start,
                                          int32_t* __restrict__ choice_len, int32_t* __restrict__ choice_off, int lane) {
  const int idx = clamp_index(indices[g], N);
  const int U = nvoc + 1;
  const int lnl_words = a.N_f * 2 * filter_stride(a.nBands);
  for (int v = 0; v < U; ++v) {
    const int L = corpus_len[v < nvoc ? N + idx * nvoc + v : idx];
    s.store(snaps + ((size_t)g * U + v) * kMtSnapWords, lane);
    s.skip(lnl_words, lane);
    const double beta = mt_uniform(0.0, a.P, mt_double(s.word(0), s.word(1)));  // as plan_head_kernel
    const int n = (int)__dmul_rn((double)L, __ddiv_rn(beta, 100.0));
    s.advance(2, lane);
    shuffle_walk_warp<false, uint32_t>(s, L, nullptr, lane);
    for (int k = 0; k < 4; ++k) s.skip(n, lane);  // f_r: rand(n) twice, two words per double
  }
  s.store(csnaps + (size_t)g * kMtSnapWords, lane);
  shuffle_walk_warp<false, uint32_t>(s, N - 1, nullptr, lane);
  const int La = corpus_len[idx];
  int st = 0;
  if (La >= trim) {
    st = (int)__dmul_rn(mt_double(s.word(0), s.word(1)), (double)(La - trim));
    s.advance(2, lane);
  }
  if (lane == 0) {
    start[g] = st;
    choice_len[g] = N - 1;
    choice_off[g] = g * n_add;
    if (g == G - 1) choice_off[G] = G * n_add;
  }
}

__global__ void __launch_bounds__(32 * kWalkWarps)
items_walk_kernel(rb_args a, int G, int nvoc, int n_add, int N, int trim, const int32_t* __restrict__ corpus_len,
                  const int32_t* __restrict__ indices, const uint32_t* __restrict__ seeds, uint32_t* __restrict__ snaps,
                  uint32_t* __restrict__ csnaps, int32_t* __restrict__ start, uint32_t* __restrict__ end_state,
                  int32_t* __restrict__ choice_len, int32_t* __restrict__ choice_off) {
  __shared__ MtSmem sm[kWalkWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x * kWalkWarps + warp;
  if (g >= G) return;
  MtStream s;
  s.sm = &sm[warp];
  s.seed(seeds[g], lane);
  walk_item(a, s, g, G, nvoc, n_add, N, trim, corpus_len, indices, snaps, csnaps, start, choice_len, choice_off, lane);
  if (end_state) s.store(end_state + (size_t)g * kMtSnapWords, lane);
}

// One warp per running stream, one stream per CTA so that few streams spread over as many SMs. Stream q walks the items
// [stream_off[q], stream_off[q+1]). The table is device data the host cannot check, so it is read defensively: every offset is
// clamped to [0, G], a decreasing step gives an empty stream, and the first stream starts at 0 and the last ends at G whatever
// the table says. Every item then belongs to at least one stream, so every output is written and stays in bounds; with a
// malformed table the items' values are unspecified (two streams that overlap both write the items they share).
// MtStream::load clamps the start states' pos.
__global__ void __launch_bounds__(32)
items_stream_walk_kernel(rb_args a, int S, const int32_t* __restrict__ stream_off, int G, int nvoc, int n_add, int N, int trim,
                         const int32_t* __restrict__ corpus_len, const int32_t* __restrict__ indices,
                         const uint32_t* __restrict__ start_state, uint32_t* __restrict__ snaps, uint32_t* __restrict__ csnaps,
                         int32_t* __restrict__ start, uint32_t* __restrict__ end_state, int32_t* __restrict__ choice_len,
                         int32_t* __restrict__ choice_off) {
  __shared__ MtSmem sm;
  const int q = blockIdx.x, lane = threadIdx.x;
  const int lo = q == 0 ? 0 : min(max(stream_off[q], 0), G);
  const int hi = q == S - 1 ? G : max(lo, min(stream_off[q + 1], G));
  MtStream s;
  s.sm = &sm;
  s.load(start_state + (size_t)q * kMtSnapWords, lane);
  for (int g = lo; g < hi; ++g)
    walk_item(a, s, g, G, nvoc, n_add, N, trim, corpus_len, indices, snaps, csnaps, start, choice_len, choice_off, lane);
  if (end_state) s.store(end_state + (size_t)q * kMtSnapWords, lane);
}

// row_len is clamped to [0, ld]: a corpus length table that names a row longer than the batch stride (a packed corpus's len is
// device data nothing checks against ld) gets that row processed as ld samples; valid lengths pass unchanged
__global__ void __launch_bounds__(256)
items_rows_kernel(int G, int nvoc, int n_add, int N, int ld, const int32_t* __restrict__ corpus_len, const int32_t* __restrict__ indices,
                  const int32_t* __restrict__ choice, int32_t* __restrict__ src_row, int32_t* __restrict__ row_len,
                  int32_t* __restrict__ view_row, float* __restrict__ view_label) {
  const int U = nvoc + 1, V = 2 + n_add + 2 * nvoc;
  const size_t nb = (size_t)G * U, rows = nb + (size_t)G * n_add;
  const size_t step = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (size_t r = t0; r < rows; r += step) {
    int src;
    if (r < nb) {
      const int g = (int)(r / U), v = (int)(r - (size_t)g * U);
      const int idx = clamp_index(indices[g], N);
      src = v < nvoc ? N + idx * nvoc + v : idx;
    } else {
      const size_t q = r - nb;
      const int idx = clamp_index(indices[q / n_add], N);
      const int c = choice[q];
      src = c + (c >= idx ? 1 : 0);  // position in others = list(range(N)) without idx
    }
    src_row[r] = src;
    row_len[r] = min(max(corpus_len[src], 0), ld);
  }
  // view order of Dataset_for (line 133): anchor, augmented anchor, additional bona fide, vocoded, augmented vocoded; a row
  // r >= 0 is read from the batch, -1-r from its RawBoost results
  for (size_t e = t0; e < (size_t)G * V; e += step) {
    const int g = (int)(e / V), k = (int)(e - (size_t)g * V);
    const int base = g * U;
    int r;
    if (k < 2) r = k == 0 ? base + nvoc : -1 - (base + nvoc);
    else if (k < 2 + n_add) r = (int)nb + g * n_add + (k - 2);
    else if (k < 2 + n_add + nvoc) r = base + (k - 2 - n_add);
    else r = -1 - (base + (k - 2 - n_add - nvoc));
    view_row[e] = r;
  }
  for (size_t k = t0; k < (size_t)V; k += step) view_label[k] = k < (size_t)(2 + n_add) ? 1.f : 0.f;  // asvspoof_2019_augall_3.py:143-146
}

__global__ void __launch_bounds__(256)
items_gather_kernel(const float* __restrict__ corpus, int ld, const int32_t* __restrict__ src_row, const int32_t* __restrict__ row_len,
                    float* __restrict__ x) {
  const size_t r = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(corpus + (size_t)src_row[r] * ld);
  float4* dst = reinterpret_cast<float4*>(x + r * ld);
  const int n4 = (row_len[r] + 3) >> 2;  // the row's padding up to ld is never read
  for (int k = threadIdx.x; k < n4; k += blockDim.x) dst[k] = __ldg(src + k);
}

// Packed corpus (rb_corpus) -> batch rows. Row r of the batch is read from 16-byte chunk start[src_row[r]] on, ceil(len * e / 16)
// chunks (e = 4 bytes per float32 sample, 2 per PCM16 sample); the samples past len in the row's last float4 are written as
// zeros, as a padded corpus holds them. Reading page-locked host memory over PCIe, the rate depends on how many 16-byte loads
// are in flight, so every thread issues kGatherU independent loads before its stores. The work is (row, segment of
// kGatherSegChunks chunks), grid-stride, so that long and short rows alike spread over the whole GPU; a segment past its row's
// end returns at once. Chunk reads are clamped to [0, chunks): a malformed start table reads wrong samples, never outside the
// corpus. row_len is already within [0, ld] (items_rows_kernel).
constexpr int kGatherThreads = 256, kGatherU = 8;
constexpr int kGatherStep = kGatherThreads * kGatherU;  // chunks per pass of a CTA
constexpr int kGatherSegChunks = 4 * kGatherStep;       // chunks per work item

__device__ __forceinline__ float pcm16_lo(uint32_t w) { return (float)(short)(w & 0xffffu) * (1.f / 32768.f); }  // as rb_dense.cu
__device__ __forceinline__ float pcm16_hi(uint32_t w) { return (float)(short)(w >> 16) * (1.f / 32768.f); }

template <bool PCM16>
__global__ void __launch_bounds__(kGatherThreads)
items_gather_packed_kernel(const uint4* __restrict__ samples, int64_t chunks, const int64_t* __restrict__ start,
                           const int32_t* __restrict__ src_row, const int32_t* __restrict__ row_len, int ld, size_t rows, int segs,
                           float* __restrict__ x) {
  constexpr int E = PCM16 ? 8 : 4;  // samples per chunk
  const size_t work = rows * (size_t)segs;
  for (size_t b = blockIdx.x; b < work; b += gridDim.x) {
    const size_t r = b / (size_t)segs;
    const int seg = (int)(b - r * (size_t)segs);
    const int n = row_len[r];
    const int nc = (n + E - 1) / E, n4 = (n + 3) >> 2;
    const int c_end = min(nc, (seg + 1) * kGatherSegChunks);
    if (seg * kGatherSegChunks >= c_end) continue;  // uniform over the CTA
    const int64_t base = min(max(start[src_row[r]], (int64_t)0), chunks);
    float4* dst = reinterpret_cast<float4*>(x + r * (size_t)ld);
    for (int c0 = seg * kGatherSegChunks; c0 < c_end; c0 += kGatherStep) {
      uint4 v[kGatherU];
#pragma unroll
      for (int j = 0; j < kGatherU; ++j) {
        const int c = c0 + j * kGatherThreads + threadIdx.x;
        v[j] = make_uint4(0u, 0u, 0u, 0u);
        if (c < c_end && chunks > 0) v[j] = __ldcs(samples + min(base + c, chunks - 1));
      }
#pragma unroll
      for (int j = 0; j < kGatherU; ++j) {
        const int c = c0 + j * kGatherThreads + threadIdx.x;
        if (c >= c_end) continue;
        float f[E];
        if constexpr (PCM16) {
          const uint32_t w[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
          for (int k = 0; k < 4; ++k) f[2 * k] = pcm16_lo(w[k]), f[2 * k + 1] = pcm16_hi(w[k]);
        } else {
          f[0] = __uint_as_float(v[j].x), f[1] = __uint_as_float(v[j].y), f[2] = __uint_as_float(v[j].z), f[3] = __uint_as_float(v[j].w);
        }
        if ((c + 1) * E > n) {  // the row's last chunk: zeros past len
#pragma unroll
          for (int k = 0; k < E; ++k)
            if (c * E + k >= n) f[k] = 0.f;
        }
        if constexpr (PCM16) {
          dst[2 * c] = make_float4(f[0], f[1], f[2], f[3]);
          if (2 * c + 1 < n4) dst[2 * c + 1] = make_float4(f[4], f[5], f[6], f[7]);
        } else {
          dst[c] = make_float4(f[0], f[1], f[2], f[3]);
        }
      }
    }
  }
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct ItemsLayout {
  size_t snaps, csnaps, clen, coff, cpos, shuffle, view_row, view_label, plan, plan_bytes, draw_bytes;
  size_t src_row, row_len, start, x, y, proc, proc_bytes, bytes;
};

ItemsLayout items_layout(const rb_args* args, int G, int nvoc, int n_add, int N, int ld) {
  ItemsLayout l{};
  size_t off = 0;
  auto take = [&](size_t n) {
    const size_t r = off;
    off += align_up(n, 256);
    return r;
  };
  const int U = nvoc + 1, V = 2 + n_add + 2 * nvoc;
  const size_t nb = (size_t)G * U, rows = nb + (size_t)G * n_add;
  l.snaps = take(nb * kMtSnapWords * 4);
  l.csnaps = take((size_t)G * kMtSnapWords * 4);
  l.clen = take((size_t)G * 4);
  l.coff = take((size_t)(G + 1) * 4);
  l.cpos = take((size_t)G * n_add * 4);
  l.shuffle = take(n_add > 0 ? shuffle_prefix_bytes(G, N - 1) : 0);
  l.view_row = take((size_t)G * V * 4);
  l.view_label = take((size_t)V * 4);
  l.plan_bytes = rb_devplan_bytes(args, 5, (int)nb, ld);
  l.plan = take(l.plan_bytes);
  l.draw_bytes = off;
  l.src_row = take(rows * 4);
  l.row_len = take(rows * 4);
  l.start = take((size_t)G * 4);
  l.x = take(rows * ld * 4);
  l.y = take(nb * ld * 4);
  l.proc_bytes = rb_workspace_bytes_for(5, (int)nb, ld);
  l.proc = take(l.proc_bytes);
  l.bytes = off;
  return l;
}

// shape checks shared by the three entries; RB_OK when the shape is drawable
int check_shape(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim) {
  if (!args || G < 0 || nvoc < 0 || n_add < 0 || N < 1 || ld <= 0 || trim < 1) return RB_ERR_INVALID_ARG;
  if (n_add > N - 1) return RB_ERR_INVALID_ARG;  // np.random.choice(..., replace=False) cannot take more than N-1
  if ((int64_t)N * (1 + nvoc) > INT_MAX || (int64_t)G * (nvoc + 1 + n_add) > INT_MAX) return RB_ERR_INVALID_ARG;
  if (G > 0 && (int64_t)G * (nvoc + 1) * args->N_f > INT_MAX) return RB_ERR_INVALID_ARG;
  if (ld % 4 != 0) return RB_ERR_ALIGNMENT;
  if (ld > (1 << 30) || N - 1 > (1 << 30)) return RB_ERR_UNSUPPORTED;
  if (G > 0 && rb_devplan_bytes(args, 5, G * (nvoc + 1), ld) == 0) return RB_ERR_UNSUPPORTED;
  return RB_OK;
}

int check_workspace(const void* ws, size_t have, size_t need) {
  if (!ws) return RB_ERR_WORKSPACE;
  if ((uintptr_t)ws & 255u) return RB_ERR_ALIGNMENT;
  return have < need ? RB_ERR_WORKSPACE : RB_OK;
}

// Where the items' streams start: item g seeded with seeds[g] (end_state per item), or S running streams (end_state per
// stream): the items of stream q are [stream_off[q], stream_off[q+1]), its state before the first of them start_state[q].
struct WalkSource {
  bool seeded;
  const uint32_t* seeds;
  int S;
  const int32_t* stream_off;
  const uint32_t* start_state;

  // checked before G == 0 returns: S >= 0, and at least one stream when there are items
  bool shape_ok(int G) const { return seeded || (S >= 0 && (S > 0 || G == 0)); }
  bool pointers_ok() const { return seeded ? seeds != nullptr : (stream_off && start_state); }
};

// every draw of the batch: snapshots, crop starts, choice, row tables, plan
int items_draw(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, const int32_t* corpus_len,
               const int32_t* indices, const WalkSource& src, int32_t* src_row, int32_t* row_len, int32_t* start,
               uint32_t* end_state, char* d, const ItemsLayout& l, rb_plan* plan, cudaStream_t st) {
  const int nb = G * (nvoc + 1);
  uint32_t *snaps = (uint32_t*)(d + l.snaps), *csnaps = (uint32_t*)(d + l.csnaps);
  int32_t *clen = (int32_t*)(d + l.clen), *coff = (int32_t*)(d + l.coff);
  if (src.seeded)
    items_walk_kernel<<<(G + kWalkWarps - 1) / kWalkWarps, 32 * kWalkWarps, 0, st>>>(
        *args, G, nvoc, n_add, N, trim, corpus_len, indices, src.seeds, snaps, csnaps, start, end_state, clen, coff);
  else
    items_stream_walk_kernel<<<src.S, 32, 0, st>>>(*args, src.S, src.stream_off, G, nvoc, n_add, N, trim, corpus_len, indices,
                                                   src.start_state, snaps, csnaps, start, end_state, clen, coff);
  RB_LAUNCH_CHECK();
  int rc;
  if (n_add > 0 && (rc = shuffle_prefix(G, N - 1, clen, csnaps, coff, (int32_t*)(d + l.cpos), d + l.shuffle, st)) != RB_OK)
    return rc;
  const size_t work = (size_t)G * (nvoc + 1 + n_add) + (size_t)G * (2 + n_add + 2 * nvoc);
  const int grid = (int)std::min<size_t>((work + 255) / 256, 148 * 8);
  items_rows_kernel<<<grid, 256, 0, st>>>(G, nvoc, n_add, N, ld, corpus_len, indices, (const int32_t*)(d + l.cpos), src_row, row_len,
                                         (int32_t*)(d + l.view_row), (float*)(d + l.view_label));
  RB_LAUNCH_CHECK();
  void* pm = d + l.plan;
  if ((rc = devplan_begin(args, 5, nb, ld, row_len, nullptr, pm, l.plan_bytes, plan, st, snaps)) != RB_OK) return rc;
  if ((rc = devplan_body(args, 5, nb, ld, row_len, nullptr, pm, 0, nb, st, snaps)) != RB_OK) return rc;
  if ((rc = devplan_apply(args, 5, nb, ld, row_len, pm, 0, nb, st)) != RB_OK) return rc;
  return devplan_end(args, 5, nb, ld, pm, st);
}

int draw_entry(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, const int32_t* corpus_len,
               const int32_t* indices, const WalkSource& src, int32_t* src_row, int32_t* row_len, int32_t* start,
               uint32_t* end_state, void* workspace, size_t workspace_bytes, rb_plan* plan, void* stream) {
  int rc = check_shape(args, G, nvoc, n_add, N, ld, trim);
  if (rc != RB_OK) return rc;
  if (!plan) return RB_ERR_INVALID_ARG;
  memset(plan, 0, sizeof(*plan));
  if (!src.shape_ok(G)) return RB_ERR_INVALID_ARG;
  if (G == 0) return RB_OK;
  if (!corpus_len || !indices || !src.pointers_ok() || !src_row || !row_len || !start) return RB_ERR_INVALID_ARG;
  const ItemsLayout l = items_layout(args, G, nvoc, n_add, N, ld);
  if ((rc = check_workspace(workspace, workspace_bytes, l.draw_bytes)) != RB_OK) return rc;
  return items_draw(args, G, nvoc, n_add, N, ld, trim, corpus_len, indices, src, src_row, row_len, start, end_state,
                    (char*)workspace, l, plan, (cudaStream_t)stream);
}

// Where the batch rows are gathered from: a padded float32 matrix [R, ld] with its lengths (rb_items_run / rb_items_stream_run)
// or a packed corpus (the _packed entries).
struct CorpusSource {
  bool is_packed;
  const float* padded;
  const int32_t* padded_len;
  const rb_corpus* packed;

  const int32_t* len() const { return is_packed ? packed->len : padded_len; }
  // RB_OK, or the error of the host-side checks that need no CUDA call
  int check(int N, int nvoc) const {
    if (!is_packed) {
      if (!padded || !padded_len) return RB_ERR_INVALID_ARG;
      return ((uintptr_t)padded & 15u) ? RB_ERR_ALIGNMENT : RB_OK;
    }
    if (!packed) return RB_ERR_INVALID_ARG;
    const rb_corpus& c = *packed;
    if (!c.samples || !c.start || !c.len || (c.kind != RB_CORPUS_F32 && c.kind != RB_CORPUS_PCM16)) return RB_ERR_INVALID_ARG;
    if ((int64_t)c.rows != (int64_t)N * (1 + nvoc) || c.chunks < 0) return RB_ERR_INVALID_ARG;
    return ((uintptr_t)c.samples & 15u) ? RB_ERR_ALIGNMENT : RB_OK;
  }
};

// The address at which the device reads a packed corpus's samples: the pointer itself for device memory of the current device,
// the mapped device pointer for page-locked host memory; nullptr for anything else (pageable memory, another device's memory,
// no allocation).
const void* corpus_device_ptr(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();  // an unknown pointer is an argument error, not a sticky one
    return nullptr;
  }
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  if (at.type == cudaMemoryTypeDevice) return at.device == dev ? p : nullptr;
  if (at.type == cudaMemoryTypeHost) return at.devicePointer;
  return nullptr;
}

int gather_packed(const rb_corpus& c, const void* samples, int ld, const int32_t* src_row, const int32_t* row_len, int rows,
                  float* x, cudaStream_t st) {
  const int e = c.kind == RB_CORPUS_PCM16 ? 8 : 4;  // samples per chunk
  const int segs = ((ld + e - 1) / e + kGatherSegChunks - 1) / kGatherSegChunks;
  const size_t work = (size_t)rows * segs;
  const int grid = (int)std::min<size_t>(work, 148 * 8 * 4);
  const uint4* s = (const uint4*)samples;
  if (c.kind == RB_CORPUS_PCM16)
    items_gather_packed_kernel<true><<<grid, kGatherThreads, 0, st>>>(s, c.chunks, c.start, src_row, row_len, ld, rows, segs, x);
  else
    items_gather_packed_kernel<false><<<grid, kGatherThreads, 0, st>>>(s, c.chunks, c.start, src_row, row_len, ld, rows, segs, x);
  RB_LAUNCH_CHECK();
  return RB_OK;
}

int run_entry(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, int repeat_pad, int layout,
              const CorpusSource& corpus, const int32_t* indices, const WalkSource& src, float* out, int32_t* out_len,
              float* labels, uint32_t* end_state, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_shape(args, G, nvoc, n_add, N, ld, trim);
  if (rc != RB_OK) return rc;
  const int V = 2 + n_add + 2 * nvoc;
  if ((layout != 0 && layout != 1) || (labels && V > 256)) return RB_ERR_INVALID_ARG;
  if (!src.shape_ok(G)) return RB_ERR_INVALID_ARG;
  if (G == 0) return RB_OK;
  if (!indices || !src.pointers_ok() || !out) return RB_ERR_INVALID_ARG;
  if ((rc = corpus.check(N, nvoc)) != RB_OK) return rc;
  const ItemsLayout l = items_layout(args, G, nvoc, n_add, N, ld);
  if ((rc = check_workspace(workspace, workspace_bytes, l.bytes)) != RB_OK) return rc;
  const void* samples = nullptr;
  if (corpus.is_packed && !(samples = corpus_device_ptr(corpus.packed->samples))) return RB_ERR_INVALID_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  char* d = (char*)workspace;
  int32_t *src_row = (int32_t*)(d + l.src_row), *row_len = (int32_t*)(d + l.row_len), *start = (int32_t*)(d + l.start);
  rb_plan plan;
  if ((rc = items_draw(args, G, nvoc, n_add, N, ld, trim, corpus.len(), indices, src, src_row, row_len, start, end_state, d, l,
                       &plan, st)) != RB_OK)
    return rc;
  const int rows = G * (nvoc + 1 + n_add), nb = G * (nvoc + 1);
  float *x = (float*)(d + l.x), *y = (float*)(d + l.y);
  if (corpus.is_packed) {
    if ((rc = gather_packed(*corpus.packed, samples, ld, src_row, row_len, rows, x, st)) != RB_OK) return rc;
  } else {
    items_gather_kernel<<<rows, 256, 0, st>>>(corpus.padded, ld, src_row, row_len, x);
    RB_LAUNCH_CHECK();
  }
  if ((rc = rb_process(5, x, row_len, nb, ld, &plan, y, d + l.proc, l.proc_bytes, stream)) != RB_OK) return rc;
  return rb_multiview_assemble_ex(x, y, (const int32_t*)(d + l.view_row), row_len, G, V, ld, start, trim, repeat_pad, layout, out,
                                  out_len, labels ? (const float*)(d + l.view_label) : nullptr, labels, stream);
}

}  // namespace
}  // namespace rb

using namespace rb;

extern "C" {

size_t rb_items_workspace_bytes(const rb_args* args, int G, int nvoc, int n_add, int N, int ld) {
  if (check_shape(args, G, nvoc, n_add, N, ld, 1) != RB_OK || G == 0) return 0;
  return items_layout(args, G, nvoc, n_add, N, ld).bytes;
}

int rb_items_draw(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, const int32_t* corpus_len,
                  const int32_t* indices, const uint32_t* seeds, int32_t* src_row, int32_t* row_len, int32_t* start,
                  uint32_t* end_state, void* workspace, size_t workspace_bytes, rb_plan* plan, void* stream) {
  return draw_entry(args, G, nvoc, n_add, N, ld, trim, corpus_len, indices, {true, seeds, 0, nullptr, nullptr}, src_row, row_len,
                    start, end_state, workspace, workspace_bytes, plan, stream);
}

int rb_items_run(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, int repeat_pad, int layout,
                 const float* corpus, const int32_t* corpus_len, const int32_t* indices, const uint32_t* seeds, float* out,
                 int32_t* out_len, float* labels, uint32_t* end_state, void* workspace, size_t workspace_bytes, void* stream) {
  return run_entry(args, G, nvoc, n_add, N, ld, trim, repeat_pad, layout, {false, corpus, corpus_len, nullptr}, indices,
                   {true, seeds, 0, nullptr, nullptr}, out, out_len, labels, end_state, workspace, workspace_bytes, stream);
}

int rb_items_run_packed(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, int repeat_pad, int layout,
                        const rb_corpus* corpus, const int32_t* indices, const uint32_t* seeds, float* out, int32_t* out_len,
                        float* labels, uint32_t* end_state, void* workspace, size_t workspace_bytes, void* stream) {
  return run_entry(args, G, nvoc, n_add, N, ld, trim, repeat_pad, layout, {true, nullptr, nullptr, corpus}, indices,
                   {true, seeds, 0, nullptr, nullptr}, out, out_len, labels, end_state, workspace, workspace_bytes, stream);
}

int rb_items_stream_draw(const rb_args* args, int S, const int32_t* stream_off, int G, int nvoc, int n_add, int N, int ld, int trim,
                         const int32_t* corpus_len, const int32_t* indices, const uint32_t* start_state, int32_t* src_row,
                         int32_t* row_len, int32_t* start, uint32_t* end_state, void* workspace, size_t workspace_bytes, rb_plan* plan,
                         void* stream) {
  return draw_entry(args, G, nvoc, n_add, N, ld, trim, corpus_len, indices, {false, nullptr, S, stream_off, start_state}, src_row,
                    row_len, start, end_state, workspace, workspace_bytes, plan, stream);
}

int rb_items_stream_run(const rb_args* args, int S, const int32_t* stream_off, int G, int nvoc, int n_add, int N, int ld, int trim,
                        int repeat_pad, int layout, const float* corpus, const int32_t* corpus_len, const int32_t* indices,
                        const uint32_t* start_state, float* out, int32_t* out_len, float* labels, uint32_t* end_state, void* workspace,
                        size_t workspace_bytes, void* stream) {
  return run_entry(args, G, nvoc, n_add, N, ld, trim, repeat_pad, layout, {false, corpus, corpus_len, nullptr}, indices,
                   {false, nullptr, S, stream_off, start_state}, out, out_len, labels, end_state, workspace, workspace_bytes, stream);
}

int rb_items_stream_run_packed(const rb_args* args, int S, const int32_t* stream_off, int G, int nvoc, int n_add, int N, int ld,
                               int trim, int repeat_pad, int layout, const rb_corpus* corpus, const int32_t* indices,
                               const uint32_t* start_state, float* out, int32_t* out_len, float* labels, uint32_t* end_state,
                               void* workspace, size_t workspace_bytes, void* stream) {
  return run_entry(args, G, nvoc, n_add, N, ld, trim, repeat_pad, layout, {true, nullptr, nullptr, corpus}, indices,
                   {false, nullptr, S, stream_off, start_state}, out, out_len, labels, end_state, workspace, workspace_bytes, stream);
}

}  // extern "C"
