/*
 * rawboost_b200.h -- C ABI of the B200-native RawBoost waveform-augmentation path.
 *
 * The reference (josebeo2016/SCL-Deepfake-audio-detection) has no FFI of its own: its callers bind to
 * plain Python symbols in datautils/RawBoost.py (SURVEY.md 8b). This header is the boundary a
 * maintainer binds instead (ctypes stub in INTEGRATION.md); every entry point names the reference
 * function it replaces. Conventions:
 *
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every function returns an int: 0 = RB_OK, <0 = rb_status, >0 = a cudaError_t. Nothing throws.
 *   - `rb_*` device entry points take DEVICE pointers owned by the caller, an explicit stream
 *     (a cudaStream_t passed as void*; NULL = legacy default stream) and a caller-provided device
 *     workspace; they launch asynchronously, never allocate and never synchronise.
 *   - `rb_ctx_*` / `rb_process_host` take HOST pointers and own their device scratch, pinned staging
 *     and stream; they return after the results are in the host output buffer.
 *   - there is no CPU fallback anywhere: without a CUDA device every call fails loudly.
 *
 * Layout. A batch is B utterances stored as rows of a [B, ld] float32 matrix (row stride `ld` elements,
 * ld % 4 == 0, base pointer 16-byte aligned); utterance u uses the first len[u] <= ld samples of its row,
 * the rest is ignored on input and left untouched on output. Ragged per-utterance data is CSR: an int32
 * offset array with one more entry than there are owners, and a packed value array.
 *
 * Random parameters are NOT drawn here. The host draws them with the reference's own numpy calls, in the
 * reference's order (RawBoost.py:15,79,80,90), so both sides see identical filter taps and impulse
 * positions; this library only does the arithmetic.
 */
#ifndef RAWBOOST_B200_H_
#define RAWBOOST_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RB_ABI_VERSION 1

#if defined(__GNUC__)
#define RB_API __attribute__((visibility("default")))
#else
#define RB_API
#endif

typedef enum rb_status {
  RB_OK = 0,
  RB_ERR_INVALID_ARG = -1,   /* null pointer, negative size, unknown algo ...            */
  RB_ERR_ALIGNMENT = -2,     /* ld % 4 != 0 or a waveform pointer not 16-byte aligned     */
  RB_ERR_WORKSPACE = -3,     /* workspace smaller than rb_workspace_bytes()               */
  RB_ERR_NO_DEVICE = -4,     /* no CUDA device / wrong architecture (needs sm_100)        */
  RB_ERR_PLAN = -5,          /* a plan field required by the requested algo is missing    */
  RB_ERR_UNSUPPORTED = -6    /* arguments outside what the device-side planner handles    */
} rb_status;

/* Human-readable text for a return code of any function below (rb_status or cudaError_t). */
RB_API const char* rb_error_string(int code);
RB_API int rb_abi_version(void);

/*
 * Device-side plan for one batch: everything the reference draws from np.random, already on the device.
 * Fields an algo does not use may be NULL/0.
 *
 *  LnL  (RawBoost.py:59-69)  n_f filters per utterance; filter i of utterance u is applied to x**(i+1).
 *       lnl_taps      float32[lnl_tap_off[B*n_f]]   taps b (as genNotchCoeffs returns them, RawBoost.py:28-48)
 *       lnl_tap_off   int32  [B*n_f + 1]            filter (u,i) owns taps [off[u*n_f+i], off[u*n_f+i+1])
 *  ISD  (RawBoost.py:73-84)
 *       isd_off       int32  [B + 1]                impulses of utterance u: [off[u], off[u+1])
 *       isd_idx       int32  [isd_off[B]]           positions p (unique per utterance, < len[u])
 *       isd_fr        float64[isd_off[B]]           f_r = (2*rand-1)*(2*rand-1), kept in float64 so that ISD on
 *                                                   float32 input reproduces the reference bit for bit
 *       g_sd          gain
 *  SSI  (RawBoost.py:89-97)
 *       ssi_noise     float32[B, ld]                np.random.normal(0,1,len[u]) per row
 *       ssi_taps/off  as LnL with one filter per utterance (int32[B+1])
 *       ssi_snr_db    float32[B]
 */
typedef struct rb_plan {
  int32_t n_f;
  const float* lnl_taps;
  const int32_t* lnl_tap_off;
  const int32_t* isd_off;
  const int32_t* isd_idx;
  const double* isd_fr;
  float g_sd;
  const float* ssi_noise;
  const float* ssi_taps;
  const int32_t* ssi_tap_off;
  const float* ssi_snr_db;
} rb_plan;

/* Device workspace (bytes) that rb_* entry points need for a batch of B rows of stride ld: rb_workspace_bytes covers every
 * algo; rb_workspace_bytes_for is what one algo needs (algos 1, 2, 3 and 5 need no waveform-sized scratch at all, the
 * chained algos 4, 6, 7 one buffer, algo 8 two). */
RB_API size_t rb_workspace_bytes(int B, int ld);
RB_API size_t rb_workspace_bytes_for(int algo, int B, int ld);

/* ---- a-4  filterFIR(x, b)  (RawBoost.py:51-56), batched --------------------------------------------------
 * y[u][n] = sum_k b_u[k] * x[u][n + (K_u+1)/2 - k],  x == 0 outside [0, len[u]);  any K_u >= 1.
 * taps float32[tap_off[B]], tap_off int32[B+1]. No workspace. */
RB_API int rb_filter_fir(const float* x, const int32_t* len, int B, int ld, const float* taps,
                  const int32_t* tap_off, float* y, void* stream);

/* ---- a-2  normWav(x, always)  (RawBoost.py:20-25), batched ---------------------------------------------
 * y = x / max|x| if (always || max|x| > 1) else x. Bit-exact with numpy on float32 input (NaN propagates like np.amax).
 * y may equal x (in place: rows that need no scaling are not rewritten at all). */
RB_API int rb_normwav(const float* x, const int32_t* len, int B, int ld, int always, float* y, void* workspace,
               size_t workspace_bytes, void* stream);

/* ---- a-5  LnL_convolutive_noise  (RawBoost.py:59-69), arithmetic part ----------------------------------
 * y = normWav(s - mean(s), 0),  s = sum_i filterFIR(x**(i+1), b_i). Uses plan->n_f, lnl_taps, lnl_tap_off. */
RB_API int rb_lnl(const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
           size_t workspace_bytes, void* stream);

/* ---- a-6  ISD_additive_noise  (RawBoost.py:73-84), arithmetic part -------------------------------------
 * y = normWav(x with y[p] = x[p] + g_sd*x[p]*f_r at the impulse positions, 0); the impulses see the RAW x, whatever its
 * peak. Bit-exact on float32 input. Positions must be unique per utterance (they are a permutation prefix). */
RB_API int rb_isd(const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
           size_t workspace_bytes, void* stream);

/* ---- a-7  SSI_additive_noise  (RawBoost.py:89-97), arithmetic part -------------------------------------
 * y = x + filterFIR(noise, b) * ||x||_2 / (||filterFIR(noise, b)||_2 * 10^(snr/20)). */
RB_API int rb_ssi(const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
           size_t workspace_bytes, void* stream);

/* ---- a-8  process_Rawboost_feature(feature, sr, args, algo)  (asvspoof_2019_augall_3.py:377-439) -------
 * algo 1 LnL, 2 ISD, 3 SSI, 4 LnL>ISD>SSI, 5 LnL>ISD (fused), 6 LnL>SSI, 7 ISD>SSI, 8 normWav(LnL+ISD);
 * any other value copies x to y. x and y may alias only for the copy case. */
RB_API int rb_process(int algo, const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y,
               void* workspace, size_t workspace_bytes, void* stream);

/* ---- host-buffer entry points (what a non-torch caller binds; used for the end-to-end measurement) -----
 * A context owns five streams and eight device slots on `device`, grown on demand and reused. A batch is cut into
 * chunks (default: four utterances per SM, rb_ctx_set_chunk to change) that flow through a three-stage pipeline --
 * host->device copy | plan + kernels | device->host copy -- ordered by events only, so PCIe in both directions and
 * the SMs work at the same time; the call returns when y is complete. Page-locked x / y (and plan arrays) make
 * the copies asynchronous; pageable memory works but serialises them.
 * rb_process_host: every pointer (x, len, y and all plan fields) is a HOST pointer; the CSR plan is sliced per chunk.
 * rb_process_host_seeded: no plan at all -- np.random.seed(seeds[u]) precedes utterance u and the plans are drawn on
 * the device (rb_devplan_draw) while the previous chunk is being filtered. */
typedef struct rb_ctx rb_ctx;
RB_API int rb_ctx_create(rb_ctx** out, int device);
RB_API int rb_ctx_destroy(rb_ctx* ctx);
RB_API int rb_ctx_set_chunk(rb_ctx* ctx, int utterances /* 0 = default */);
RB_API int rb_process_host(rb_ctx* ctx, int algo, const float* x, const int32_t* len, int B, int ld,
                    const rb_plan* plan, float* y);
/* Tracing: with rb_ctx_trace(ctx, 1) every later call records, per pipeline chunk, six doubles -- first utterance, utterance
 * count, and the milliseconds after the start of the call at which its copy-in, plan, kernels and copy-out finished (device
 * time, CUDA events). rb_ctx_timeline copies up to `capacity` doubles of the last call and returns how many there are
 * (>= 0; this one function does not return an rb_status on success). */
RB_API int rb_ctx_trace(rb_ctx* ctx, int on);
RB_API int rb_ctx_timeline(const rb_ctx* ctx, double* out, int capacity);
/* bytes moved by the last rb_process_host call: host->device and device->host */
RB_API int rb_ctx_last_traffic(const rb_ctx* ctx, uint64_t* h2d_bytes, uint64_t* d2h_bytes);

/* ---- native host-side plan drawing (optional accelerator for the numpy path in plans.py) -------------------------
 * Bit-exact re-implementation of the numpy legacy MT19937 calls the reference makes (RawBoost.py:15,79,80,90: uniform,
 * permutation, rand, normal; seeding as np.random.seed(int)) plus the float64 filter design of genNotchCoeffs
 * (RawBoost.py:28-48). Integer results and the stream state are identical to numpy's; tap values agree to ~1e-15.
 * rb_args carries the reference's knobs (main.py:258-298) and the sample rate. */
typedef struct rb_args {
  int32_t N_f, nBands;
  double minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, minBiasLinNonLin, maxBiasLinNonLin;
  double P, g_sd, SNRmin, SNRmax, fs;
} rb_args;
/* numpy's RandomState.get_state() in C: ('MT19937', key[624], pos, has_gauss, cached_gaussian) */
typedef struct rb_rng_state {
  uint32_t key[624];
  int32_t pos;
  int32_t has_gauss;
  double cached_gaussian;
} rb_rng_state;
typedef struct rb_planner rb_planner;
/* threads <= 0: one per hardware thread. pinned != 0: plan buffers are page-locked (needs a CUDA device). */
RB_API int rb_planner_create(rb_planner** out, int threads, int pinned);
RB_API int rb_planner_destroy(rb_planner* planner);
/* Draw the plans process_Rawboost_feature(., ., args, algo) would draw for B utterances of len[u] samples.
 * seeds != NULL: np.random.seed(seeds[u]) precedes utterance u (independent, drawn in parallel by the thread pool).
 * seeds == NULL: the utterances consume ONE stream, *state, one after another, and *state is advanced.
 * *view receives HOST pointers (rb_plan layout, ssi_noise rows of stride ld) valid until the next draw on this planner;
 * pass it to rb_process_host. */
RB_API int rb_planner_draw(rb_planner* planner, const rb_args* args, int algo, int B, int ld, const int32_t* len,
                           const uint32_t* seeds, rb_rng_state* state, rb_plan* view);

/* ---- device-side plan drawing for independently seeded utterances -------------------------------------------------
 * Replays numpy's legacy MT19937 stream on the GPU (seeding, uniform, permutation, rand, normal -- the calls of
 * RawBoost.py:15,79,80,90) and designs the notch cascades of genNotchCoeffs (RawBoost.py:28-48) there, so a seeded batch
 * needs no host work and no plan upload: np.random.seed(seeds[u]) precedes utterance u, as in rb_planner_draw.
 * Tap counts, impulse counts / positions and the float64 impulse gains are bit-identical to numpy's; float32 taps and
 * SSI noise agree to 1 ulp (taps of ill-conditioned cascades -- many nearly all-stop stages -- only as far as numpy's own
 * rounding order determines them, DESIGN.md 4.4). len / seeds are DEVICE arrays; `storage` is device memory of rb_devplan_bytes() bytes,
 * 256-byte aligned; *plan (a HOST struct) receives device pointers into it, valid after the stream reaches this point.
 * Rows of any length (the permutation of rows beyond 65536 samples is walked in global memory).
 * Accepted domain (RB_ERR_UNSUPPORTED otherwise): N_f >= 1, nBands 1-100, P 0-100, fs > 0, stages of at most 255 taps
 * (1 <= minCoeff, maxCoeff <= 255, either order) and nBands * (ceil(max(minCoeff, maxCoeff)) + 1) <= 1024, a conservative
 * bound on the longest cascade (freqz's 1024-point path). */
RB_API size_t rb_devplan_bytes(const rb_args* args, int algo, int B, int ld);
RB_API int rb_devplan_draw(const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds,
                           void* storage, size_t storage_bytes, rb_plan* plan, void* stream);
/* host buffers in, host buffers out, plans drawn on the device (see the host-buffer section above) */
RB_API int rb_process_host_seeded(rb_ctx* ctx, int algo, const rb_args* args, const float* x, const int32_t* len,
                                  const uint32_t* seeds, int B, int ld, float* y);

/* ---- the step after the path, for the views of an item (SURVEY.md 8f-1 / 8f-2) -----------------------------------
 * batch_pad_for_multiview (core_scripts/data_io/wav_augmentation.py:209-282) + the view assembly of
 * Dataset_for.__getitem__ (asvspoof_2019_augall_3.py:133-142) + the [1,length,V] -> [V,length] reshape of main.py:57-60.
 * G groups (items) of V views each; view v of group g is row g*V+v of `views` ([G*V, ld], len[G*V], device). Every view
 * is cut / zero-extended / (repeat_pad) tiled to the length of the group's view 0, then one crop of `length` samples
 * starting at start[g] (device int32[G], drawn by the host: int(np.random.rand()*(len0-length)), 0 without random trim;
 * ignored when view 0 is shorter than `length`) is taken from all of them; a short view 0 is tiled up to `length` with
 * repeat_pad and left at its own length without. layout 0: out[G][length][V] (the Dataset's batch_data); layout 1:
 * out[G][V][length] (what the model consumes). out_len (nullable, device int32[G]) receives the samples written per view. */
RB_API int rb_multiview_assemble(const float* views, const int32_t* len, int G, int V, int ld, const int32_t* start, int length,
                                 int repeat_pad, int layout, float* out, int32_t* out_len, void* stream);
/* The same with the views read where they already are: view v of group g is row r = view_row[g*V+v] of `views` (r >= 0) or row
 * -1-r of `views_b` (r < 0) -- e.g. the original waveforms and their RawBoost results, two [R, ld] buffers with one length
 * array len[R] -- so assembling an item needs no regrouping copy. view_label (nullable, device float[V]) is broadcast to
 * labels (device float[G][V]): the label vector of Dataset_for.__getitem__ (asvspoof_2019_augall_3.py:143-146). */
RB_API int rb_multiview_assemble_ex(const float* views, const float* views_b, const int32_t* view_row, const int32_t* len, int G,
                                    int V, int ld, const int32_t* start, int length, int repeat_pad, int layout, float* out,
                                    int32_t* out_len, const float* view_label, float* labels, void* stream);

/* ---- reverb view, batched  (SURVEY.md 8f-4; audio_augmentor/reverb.py:39-42) -------------------------------------------
 * y_u = normWav(np.convolve(x_u, h_u), 1): the full convolution of each waveform with its room impulse response, peak-normalised.
 * x [B, ld] float32 and len[B] (device); impulse responses as CSR like rb_filter_fir: rir float32[rir_off[B]], rir_off int32[B+1]
 * (device), any K_u = rir_off[u+1] - rir_off[u]. y [B, ld_out] float32 (device), ld_out % 4 == 0, x != y. out_len int32[B]
 * (device) receives len[u] + K_u - 1, or 0 for an empty row (len[u] == 0). A row with K_u < 1, len[u] < 0, len[u] > ld,
 * len[u] + K_u - 1 > ld_out, or more taps than the workspace was sized for gets out_len[u] = -1 and is not written. Nothing is
 * ever written outside [0, out_len[u]) of a row. Peak normalisation as numpy: an all-zero result is NaN, and NaN propagates.
 * Uniformly partitioned FFT overlap-save (partitions of 8192 taps, 16384-point real FFTs; DESIGN.md 4.5): the cost per
 * output sample grows with the number of partitions, not with every tap. Float32 throughout; max-abs error against a float64
 * np.convolve is ~3e-7 after the normalisation.
 * rb_reverb_workspace_bytes(B, max_taps): device workspace (256-byte aligned) for B rows of at most max_taps taps each.
 * rb_reverb takes the partitions per row from workspace_bytes (one spectrum launch per row and partition), so pass the size
 * this function returned rather than that of a larger buffer. */
RB_API size_t rb_reverb_workspace_bytes(int B, int max_taps);
RB_API int rb_reverb(const float* x, const int32_t* len, int B, int ld, const float* rir, const int32_t* rir_off, float* y,
                     int ld_out, int32_t* out_len, void* workspace, size_t workspace_bytes, void* stream);

/* ---- whole items, each seeded on its own  (Dataset_for.__getitem__, asvspoof_2019_augall_3.py:103-146) ------------------
 * np.random.seed(seeds[g]) precedes item g, as in a loader that seeds every __getitem__; items are independent and are drawn in
 * parallel. Item g of index idx = indices[g] consumes its stream in the loader's order: RawBoost (algo 5) on each of the nvoc
 * vocoded copies in vocoder order, then on the anchor; np.random.choice(others, n_add, replace=False), i.e. permutation(N-1)[:n_add]
 * mapped through others = [0, N) without idx (consumed even when n_add == 0); then int(rand() * (L_anchor - trim)), drawn only
 * when L_anchor >= trim. The crop is batch_pad_for_multiview's with random_trim_nosil set.
 * Corpus (device): rows [R, ld] float32, R = N * (1 + nvoc), ld % 4 == 0, 16-byte aligned, lengths corpus_len[R] >= 1. Row idx is
 * bona fide utterance idx, row N + idx*nvoc + v is vocoder v's copy of it. indices (int32[G], each in [0, N)) and seeds
 * (uint32[G]) are device arrays. Batch rows, as multiview.ItemBatcher lays them out: rows g*(nvoc+1) + v are item g's vocoded
 * copies (v < nvoc) and its anchor (v = nvoc), the RawBoost inputs; rows G*(nvoc+1) + g*n_add + k its additional bona fide
 * utterances. Integer draws (tap counts, impulse positions, extra utterances, crop starts) and the float64 impulse gains equal
 * numpy's bit for bit; taps agree to 1 ulp.
 * rb_items_workspace_bytes: device workspace (256-byte aligned) of rb_items_run, which holds the gathered batch
 * [G*(nvoc+1+n_add), ld] and its RawBoost results [G*(nvoc+1), ld]; it is more than rb_items_draw needs. 0 for invalid shapes.
 * rb_items_draw: the plan of the G*(nvoc+1) RawBoost utterances (*plan, a HOST struct, receives device pointers into the
 * workspace), src_row / row_len (int32[G*(nvoc+1+n_add)]: each batch row's corpus row and its length), start (int32[G]: crop
 * starts, 0 where none is drawn) and, when end_state is not NULL, each item's stream state after its last draw (uint32[G][625]:
 * numpy's key[624] and pos, pos in 0..623).
 * rb_items_run: draw, gather, rb_process(5) and rb_multiview_assemble_ex in one call: out [G][trim][V] (layout 0) or
 * [G][V][trim] (layout 1), V = 2 + n_add + 2*nvoc in the Dataset's view order (anchor, augmented anchor, additional, vocoded,
 * augmented vocoded), out_len (nullable, int32[G]) and labels (nullable, float[G][V]: 1 for the anchor and its positives, 0 for
 * the vocoded views). repeat_pad as batch_pad_for_multiview. */
RB_API size_t rb_items_workspace_bytes(const rb_args* args, int G, int nvoc, int n_add, int N, int ld);
RB_API int rb_items_draw(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, const int32_t* corpus_len,
                         const int32_t* indices, const uint32_t* seeds, int32_t* src_row, int32_t* row_len, int32_t* start,
                         uint32_t* end_state, void* workspace, size_t workspace_bytes, rb_plan* plan, void* stream);
RB_API int rb_items_run(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, int repeat_pad, int layout,
                        const float* corpus, const int32_t* corpus_len, const int32_t* indices, const uint32_t* seeds, float* out,
                        int32_t* out_len, float* labels, uint32_t* end_state, void* workspace, size_t workspace_bytes, void* stream);

/* Items that share numpy's running stream (Dataset_for.__getitem__ called for them one after another, no per-item seed):
 * S independent streams; the items of stream s are [stream_off[s], stream_off[s+1]) of indices (device int32[S+1],
 * stream_off[0] = 0, non-decreasing, stream_off[S] = G). start_state (device uint32[S][625]) is numpy's key[624], pos (0..624),
 * as RandomState.get_state()[1:3]; end_state (nullable, device uint32[S][625]) receives each stream's state after its last
 * draw (pos 0..623). Every other argument, output, workspace and row layout as rb_items_draw / rb_items_run; the workspace is
 * rb_items_workspace_bytes(args, G, nvoc, n_add, N, ld). S < 0, or S == 0 with G > 0, is RB_ERR_INVALID_ARG; empty streams
 * are legal (S may exceed G; an empty stream's end state is its start state). G == 0 launches nothing and writes no end state.
 * One warp walks each stream's items in order, so a stream's walk takes time in proportion to its item count.
 * The table and the states are device data and are read defensively: offsets are clamped to [0, G], a decreasing step is an
 * empty stream, the first stream starts at item 0 and the last ends at item G, and pos is clamped to 0..624. A malformed table
 * never leads to an access out of bounds, but the items it does not describe (in no stream's range, or in two) and the end
 * states of the streams involved are unspecified. */
RB_API int rb_items_stream_draw(const rb_args* args, int S, const int32_t* stream_off, int G, int nvoc, int n_add, int N, int ld,
                                int trim, const int32_t* corpus_len, const int32_t* indices, const uint32_t* start_state,
                                int32_t* src_row, int32_t* row_len, int32_t* start, uint32_t* end_state,
                                void* workspace, size_t workspace_bytes, rb_plan* plan, void* stream);
RB_API int rb_items_stream_run(const rb_args* args, int S, const int32_t* stream_off, int G, int nvoc, int n_add, int N, int ld,
                               int trim, int repeat_pad, int layout, const float* corpus, const int32_t* corpus_len,
                               const int32_t* indices, const uint32_t* start_state, float* out, int32_t* out_len, float* labels,
                               uint32_t* end_state, void* workspace, size_t workspace_bytes, void* stream);

/* The same items from a packed corpus: rows stored back to back, each from a 16-byte chunk boundary, as float32 samples or as
 * 16-bit PCM, in device memory or read in place from page-locked host memory. A padded corpus stores every row at the length of
 * the longest; for a ragged corpus the packed form needs a fraction of that (ASVspoof 2019 LA train with three vocoders at the
 * lengths the loaders read: 8.71 GB padded, 2.94 GB packed float32, 1.47 GB packed PCM16; 0 device bytes in host memory).
 *   samples  16-byte aligned: device memory of the calling device, or page-locked host memory (cudaHostAlloc / cudaHostRegister,
 *            e.g. a torch pin_memory tensor), read in place by the gather kernel, 2 or 4 bytes per sample used
 *   kind     RB_CORPUS_F32 (float32) or RB_CORPUS_PCM16 (int16, read as sample / 32768: what librosa returns for 16-bit audio,
 *            exact in float32)
 *   rows     R = N * (1 + nvoc); row order exactly as rb_items_run's corpus
 *   chunks   size of `samples` in 16-byte chunks
 *   start    DEVICE int64[R]: row r begins at byte 16 * start[r] of samples
 *   len      DEVICE int32[R]: samples in row r, >= 1 (what rb_items_draw / rb_items_stream_draw take as corpus_len)
 * Every other argument, output and the workspace (rb_items_workspace_bytes) mean what they mean for rb_items_run /
 * rb_items_stream_run; ld is the row stride of the gathered batch only: a multiple of 4 and >= the longest len the items use.
 * When the corpus holds the float values of a padded corpus (k / 32768 for PCM16), the results equal the padded entries' bit for
 * bit. Checked on the host before anything is launched, after the checks of the padded entries (G == 0 returns RB_OK first):
 * RB_ERR_INVALID_ARG for a NULL corpus, samples, start or len, an unknown kind, rows != N * (1 + nvoc) or chunks < 0;
 * RB_ERR_ALIGNMENT for samples not 16-byte aligned; RB_ERR_INVALID_ARG for samples that are neither device memory of the current
 * device nor page-locked host memory (pageable memory, another device's memory, no allocation at all).
 * start and len are device data the host cannot check, so they are read defensively: chunk reads are clamped to [0, chunks)
 * and a row longer than ld is processed as ld samples. The items such a table describes get unspecified values; nothing is ever
 * read or written out of bounds. */
#define RB_CORPUS_F32 0   /* float32 samples                                */
#define RB_CORPUS_PCM16 1 /* int16 samples, read as sample / 32768 (exact)  */
typedef struct rb_corpus {
  const void* samples;
  int32_t kind;
  int32_t rows;
  int64_t chunks;
  const int64_t* start;
  const int32_t* len;
} rb_corpus;
RB_API int rb_items_run_packed(const rb_args* args, int G, int nvoc, int n_add, int N, int ld, int trim, int repeat_pad,
                               int layout, const rb_corpus* corpus, const int32_t* indices, const uint32_t* seeds, float* out,
                               int32_t* out_len, float* labels, uint32_t* end_state, void* workspace, size_t workspace_bytes,
                               void* stream);
RB_API int rb_items_stream_run_packed(const rb_args* args, int S, const int32_t* stream_off, int G, int nvoc, int n_add, int N,
                                      int ld, int trim, int repeat_pad, int layout, const rb_corpus* corpus,
                                      const int32_t* indices, const uint32_t* start_state, float* out, int32_t* out_len,
                                      float* labels, uint32_t* end_state, void* workspace, size_t workspace_bytes, void* stream);

/* Streaming form of rb_process_host_seeded: queues the whole call and returns at once; *ticket identifies it. Up to two calls
 * may be in flight (a third submit first waits for the oldest), so the copies of consecutive batches follow each other
 * without a gap and steady-state throughput is bound by PCIe alone. x, len, seeds and y must stay valid -- and y must not
 * be read -- until rb_ctx_wait(ctx, ticket) has returned (ticket 0 waits for everything submitted so far). */
RB_API int rb_submit_host_seeded(rb_ctx* ctx, int algo, const rb_args* args, const float* x, const int32_t* len,
                                 const uint32_t* seeds, int B, int ld, float* y, uint64_t* ticket);
RB_API int rb_ctx_wait(rb_ctx* ctx, uint64_t ticket);

/* The general streaming form: where the waveforms come from and where the results go are chosen per call.
 *   x_kind  RB_IO_HOST_F32    x = host float32 [B, ld]                       (what rb_submit_host_seeded takes)
 *           RB_IO_HOST_PCM16  x = host int16   [B, ld], ld % 8 == 0: 16-bit PCM as a wav file holds it; converted on the device
 *                             as sample / 32768 -- exactly what librosa / soundfile return for 16-bit audio -- so the
 *                             host->device traffic is halved
 *           RB_IO_DEVICE_F32  x = device float32 [B, ld]; len and seeds are then DEVICE arrays too and use_user_stream must be set
 *   y_kind  RB_IO_HOST_F32    y = host float32 [B, ld]
 *           RB_IO_DEVICE_F32  y = device float32 [B, ld]: the results stay on the device, where the consumer of the views
 *                             lives (main.py:57-60); nothing is copied back
 *   use_user_stream != 0: the call is ordered after the work already queued on user_stream (a cudaStream_t; NULL = the legacy
 *   default stream), and user_stream waits for the call's completion, so the caller needs no host synchronisation at all.
 * Chunking, the device planner and its overlap with the kernels are those of rb_submit_host_seeded; rb_ctx_wait(ticket) waits on
 * the host. Same ownership rule: every buffer stays valid and untouched until the call has completed. */
#define RB_IO_HOST_F32 0
#define RB_IO_HOST_PCM16 1
#define RB_IO_DEVICE_F32 2
RB_API int rb_submit_seeded_ex(rb_ctx* ctx, int algo, const rb_args* args, const void* x, int x_kind, const int32_t* len,
                               const uint32_t* seeds, int B, int ld, void* y, int y_kind, void* user_stream, int use_user_stream,
                               uint64_t* ticket);

/* Ragged host batches packed back to back: utterance u is x[off[u] .. off[u+1]), so the copies carry the real samples only
 * (a padded [B, ld] batch of un-cropped utterances moves ld / mean(len) times as many). Seeded semantics, chunking, the device
 * planner, use_user_stream and the two-calls-in-flight rule are those of rb_submit_seeded_ex; rb_ctx_wait(ctx, ticket) is the
 * blocking form.
 *   x_kind  RB_IO_HOST_F32 (float32) or RB_IO_HOST_PCM16 (int16, converted on the device as sample / 32768), packed, any alignment
 *   off     HOST int64[B + 1]: off[0] == 0, non-decreasing, every length off[u+1] - off[u] <= INT32_MAX. Checked at call time:
 *           RB_ERR_INVALID_ARG otherwise. A zero-length utterance is legal and occupies no bytes. int64, because a shard of long
 *           utterances exceeds 2^31 samples.
 *   y_kind  RB_IO_HOST_F32    y = host float32, packed at the same offsets as x; only y[off[0] .. off[B]) is written.
 *                             ld == 0: the rows the kernels see have stride round_up(max len, 4); ld > 0: that stride (ld % 4 == 0,
 *                             ld >= max len)
 *           RB_IO_DEVICE_F32  y = device float32 rows [B, ld] (16-byte aligned), what rb_multiview_assemble_ex and rb_process take:
 *                             ld is required, >= max len and a multiple of 4 (RB_ERR_INVALID_ARG / RB_ERR_ALIGNMENT otherwise)
 * The results equal rb_submit_seeded_ex's on the same utterances zero-padded to rows of the same ld, bit for bit.
 * Per chunk, the driver issues one copy of the chunk's packed span each way; kernels unpack it into zero-padded rows and (host
 * sink) pack the results. Traffic (rb_ctx_last_traffic), with e = 4 for float32 and 2 for PCM16 input:
 *   host->device  e * off[B] + 8 * (B + 1) (the offsets) + 4 * B (the seeds; not uploaded for an algo outside 1..8)
 *   device->host  4 * off[B] with a host sink, 0 with a device sink
 * x, off, seeds and y stay valid and untouched until the call has completed. Page-locked x, off and y keep the copies
 * asynchronous: a pageable off makes its upload wait for the copy stream. */
RB_API int rb_submit_seeded_packed(rb_ctx* ctx, int algo, const rb_args* args, const void* x, int x_kind, const int64_t* off,
                                   const uint32_t* seeds, int B, int ld, void* y, int y_kind, void* user_stream, int use_user_stream,
                                   uint64_t* ticket);

/* ---- measurement helpers (bench.py) ---------------------------------------------------------------------
 * rb_probe_fp32: runs a register-resident FFMA2 (packed=1) or FFMA (packed=0) chain on every SM and
 * returns the achieved FLOP count in *flops; the caller times it with events on `stream`.
 * rb_launch_count: number of kernels this library has launched in this process (all entry points). */
RB_API int rb_probe_fp32(int packed, int iters, float* sink /* device, >= 1 float */, double* flops, void* stream);
RB_API uint64_t rb_launch_count(void);
/* rb_profile_enable(1): bracket every FIR-bank kernel launch (the dominant kernel of algos 1,3,4,5,6,8) with CUDA
 * events on its launching stream. rb_profile_read: wait for them and return the accumulated device milliseconds and
 * launch count since the last reset. Off by default; costs two event records per launch when on. */
RB_API int rb_profile_enable(int on);
RB_API int rb_profile_read(double* fir_ms, uint64_t* fir_launches, int reset);
/* rb_set_tap_trim: process-wide, on (1) by default. The LnL and SSI filters (genNotchCoeffs cascades, whose end taps are ~1e-20
 * of the largest) then run over their effective support only: from each end, the longest run of taps whose |b| sum to at most
 * 2^-31 sum|b| is skipped (float64 sums in tap order over the float32 taps; plans.tap_support in Python). That changes an output
 * by at most 2^-30 sum_f ||b_f||_1 ||x^p||_inf before normWav -- 1/64 of what rounding the taps to float32 already allows -- and
 * removes about a quarter of the bank's multiply-adds at the default arguments. Banks of more than 16 filters per utterance,
 * and rb_filter_fir / rb_reverb (the caller's taps), always run every tap. rb_set_tap_trim(0): every tap, bit for bit the
 * results of a build without trimming. Takes effect for calls issued after it returns. */
RB_API int rb_set_tap_trim(int on);
/* The supports themselves, for counting the work that runs: support[i] = (lo, hi) of the n filters of a CSR tap array (device
 * taps float32[tap_off[n]], tap_off int32[n + 1], support int32[n][2]); the kernels run b[lo .. hi) of filter i. Asynchronous
 * on `stream`, no workspace. */
RB_API int rb_tap_support(const float* taps, const int32_t* tap_off, int n, int32_t* support, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAWBOOST_B200_H_ */
