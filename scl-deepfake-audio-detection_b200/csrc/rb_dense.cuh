// Launchers of the HBM-bound passes (rb_dense.cu). All asynchronous on `st`, no allocation, no sync.
#pragma once
#include "rb_common.cuh"

namespace rb {

// Effective support of each of nfilt filters (CSR taps / tap_off, as the plan holds them): support[i] = (lo, hi), the taps
// b[lo .. hi) that remain after dropping, from each end, the longest run whose |b| sum to at most 2^-31 sum|b| (float64 sums
// in tap order; plans.tap_support is the same rule in numpy). One warp per filter.
int launch_tap_support(const float* taps, const int32_t* tap_off, int nfilt, int2* support, cudaStream_t st);

// bit p of row u (stride mask_ld words) = 1 iff p is an impulse position of utterance u; every word of the row is written.
// support != NULL: the same launch also writes launch_tap_support's result for the B * n_f filters of taps / tap_off.
int launch_mask_build(const int32_t* isd_off, const int32_t* isd_idx, const int32_t* len, int B, uint32_t* mask,
                      int mask_ld, const float* taps, const int32_t* tap_off, int n_f, int2* support /*nullable*/,
                      cudaStream_t st);

// out[i] = in[i] / 32768 (16-bit PCM -> float32 as a wav reader does it); n % 8 == 0, both pointers 16-byte aligned
int launch_pcm16_to_f32(const int16_t* in, float* out, size_t n, cudaStream_t st);

// Utterances packed back to back: utterance r is packed[off[r] - off[0], off[r + 1] - off[0]) (off: device int64[B + 1]).
// len[r] = off[r + 1] - off[r]
int launch_lengths_from_offsets(const int64_t* off, int B, int32_t* len, cudaStream_t st);
// packed float32 (pcm16: int16, converted as sample / 32768) -> rows [B, ld] float32, zero from len[r] to ld; rows 16-byte aligned
int launch_unpack_rows(const void* packed, bool pcm16, const int64_t* off, int B, int ld, float* rows, cudaStream_t st);
// rows [B, ld] -> packed float32: [0, len[r]) of each row, nothing else written
int launch_pack_rows(const float* rows, const int64_t* off, int B, int ld, float* packed, cudaStream_t st);

// tiles per row of the streaming pass
int stream_tiles_for(int ld);

// out = normWav(v, always) where v = a (+ b when b != NULL), or -- with isd_off != NULL (b must be NULL) --
// out = normWav(a with the impulses applied, always). One streaming launch; see rb_dense.cu.
// state: B x 8 bytes of device scratch (zeroed here). out may equal a when b == NULL (in place: the copy is skipped).
int launch_norm_stream(const float* a, const float* b, const int32_t* len, int B, int ld, int always, const int32_t* isd_off,
                       const int32_t* isd_idx, const double* isd_fr, float g_sd, float* out, void* state, cudaStream_t st);

}  // namespace rb
