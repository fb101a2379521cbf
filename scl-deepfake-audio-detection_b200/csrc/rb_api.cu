// rb_api.cu -- the extern "C" surface declared in include/rawboost_b200.h: argument checks, workspace carving and
// the composition of the kernels into the reference's operators and its 9-way dispatcher
// (/root/reference/datautils/asvspoof_2019_augall_3.py:377-439).
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <initializer_list>
#include <mutex>
#include <new>
#include <vector>

#include "rb_algo.h"
#include "rb_common.cuh"
#include "rb_dense.cuh"

namespace rb {

std::atomic<uint64_t> g_launches{0};

// ---- FIR-bank launch timing (see rb_common.cuh) -------------------------------------------------------
namespace {
std::atomic<int> g_profile_on{0};
std::mutex g_profile_mu;
std::vector<cudaEvent_t> g_profile_events;  // begin/end pairs not yet read
double g_profile_ms = 0.0;
uint64_t g_profile_launches = 0;
}  // namespace

void profile_begin(cudaStream_t st) {
  if (!g_profile_on.load(std::memory_order_relaxed)) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  std::lock_guard<std::mutex> lk(g_profile_mu);
  g_profile_events.push_back(e);
}

void profile_end(cudaStream_t st) {
  if (!g_profile_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_profile_mu);
  if (g_profile_events.size() % 2 == 0) return;  // begin failed
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) {
    cudaEventDestroy(g_profile_events.back());
    g_profile_events.pop_back();
    return;
  }
  cudaEventRecord(e, st);
  g_profile_events.push_back(e);
}

namespace {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int mask_ld_for(int ld) { return (int)align_up((size_t)ld / 32 + 2, 4); }

// Device workspace layout for one batch.
struct Workspace {
  float* stats_a;
  uint32_t* counters;  // per-utterance tile arrival counters of the fused FIR tail
  uint32_t* mask;
  int mask_ld;
  float* buf1;  // intermediate waveform of the chained algos 4, 6, 7, 8
  float* buf2;  // second branch of algo 8
  size_t bytes;
};

// Waveform-sized scratch buffers an algo needs: the single-operator algos (1, 2, 3) and the fused LnL -> ISD (5) write into
// the output buffer itself; the chains 4, 6, 7 hold one intermediate waveform; algo 8 two branches and their sum.
inline int scratch_waveforms(int algo) { return algo == 8 ? 2 : (algo == 4 || algo == 6 || algo == 7) ? 1 : 0; }

Workspace carve(void* base, int B, int ld, int nbuf) {
  Workspace w;
  const int ntiles = tiles_for(ld);
  size_t off = 0;
  char* p = (char*)base;
  auto take = [&](size_t n) {
    char* r = p ? p + off : nullptr;
    off += align_up(n, 256);
    return r;
  };
  w.stats_a = (float*)take((size_t)B * ntiles * kStatN * sizeof(float));
  w.counters = (uint32_t*)take((size_t)B * sizeof(uint32_t));
  w.mask_ld = mask_ld_for(ld);
  w.mask = (uint32_t*)take((size_t)B * w.mask_ld * sizeof(uint32_t));
  w.buf1 = nbuf >= 1 ? (float*)take((size_t)B * ld * sizeof(float)) : nullptr;
  w.buf2 = nbuf >= 2 ? (float*)take((size_t)B * ld * sizeof(float)) : nullptr;
  w.bytes = off;
  return w;
}

int check_batch(const void* x, const int32_t* len, int B, int ld, const void* y) {
  if (B < 0 || ld < 0) return RB_ERR_INVALID_ARG;
  if (B == 0 || ld == 0) return RB_OK;
  if (!x || !len || !y) return RB_ERR_INVALID_ARG;
  if (ld % 4 != 0 || ((uintptr_t)x & 15u) || ((uintptr_t)y & 15u)) return RB_ERR_ALIGNMENT;
  return RB_OK;
}

int check_ws(void* ws, size_t ws_bytes, int B, int ld, int algo, Workspace* out) {
  if (B == 0 || ld == 0) return RB_OK;
  if (!ws || ((uintptr_t)ws & 255u)) return ws ? RB_ERR_ALIGNMENT : RB_ERR_WORKSPACE;
  *out = carve(ws, B, ld, scratch_waveforms(algo));
  if (out->bytes > ws_bytes) return RB_ERR_WORKSPACE;
  return RB_OK;
}

#define RB_TRY(expr)          \
  do {                        \
    int rc__ = (expr);        \
    if (rc__ != RB_OK) return rc__; \
  } while (0)

// LnL (optionally followed by ISD): x -> out. One FIR-bank launch; its fused tail does mean removal, normWav, the impulse
// scatter and the second normWav per utterance.
int do_lnl(const float* x, const int32_t* len, int B, int ld, const rb_plan* pl, bool with_isd, float* out, const Workspace& w,
           cudaStream_t st) {
  if (!pl || pl->n_f < 1 || !pl->lnl_taps || !pl->lnl_tap_off) return RB_ERR_PLAN;
  if (with_isd && (!pl->isd_off || !pl->isd_idx || !pl->isd_fr)) return RB_ERR_PLAN;
  if (with_isd) RB_TRY(launch_mask_build(pl->isd_off, pl->isd_idx, len, B, w.mask, w.mask_ld, st));
  FirTail tail;
  tail.mode = TAIL_AFFINE;
  tail.counters = w.counters;
  tail.out = out;
  if (with_isd) {
    tail.isd_off = pl->isd_off;
    tail.isd_idx = pl->isd_idx;
    tail.isd_fr = pl->isd_fr;
    tail.g_sd = pl->g_sd;
  }
  // the raw sum goes into `out` itself and is finalised in place while still in L2: no intermediate buffer reaches HBM
  return launch_fir_bank(x, len, B, ld, pl->lnl_taps, pl->lnl_tap_off, pl->n_f, 1, 1, out, w.stats_a,
                         with_isd ? w.mask : nullptr, w.mask_ld, tail, st);
}

// ISD on an existing waveform: x -> out. ONE streaming launch (impulses, peak and the conditional rescale happen in its
// per-utterance finisher CTAs; no impulse mask is needed). The input is NOT normalised first: the reference applies the impulses to the raw x
// (RawBoost.py:76-84) and only then normWav(y, 0).
int do_isd(const float* x, const int32_t* len, int B, int ld, const rb_plan* pl, float* out, const Workspace& w, cudaStream_t st) {
  if (!pl || !pl->isd_off || !pl->isd_idx || !pl->isd_fr) return RB_ERR_PLAN;
  return launch_norm_stream(x, nullptr, len, B, ld, 0, pl->isd_off, pl->isd_idx, pl->isd_fr, pl->g_sd, out, w.stats_a, st);
}

// SSI: x -> out (out must not alias x: the tail of one utterance reads x while other tiles still compute statistics of it).
// One FIR-bank launch on the noise (the coloured noise is written into `out`); its fused tail takes both norms and mixes in place.
int do_ssi(const float* x, const int32_t* len, int B, int ld, const rb_plan* pl, float* out, const Workspace& w, cudaStream_t st) {
  if (!pl || !pl->ssi_noise || !pl->ssi_taps || !pl->ssi_tap_off || !pl->ssi_snr_db) return RB_ERR_PLAN;
  if ((uintptr_t)pl->ssi_noise & 15u) return RB_ERR_ALIGNMENT;
  FirTail tail;
  tail.mode = TAIL_SSI;
  tail.counters = w.counters;
  tail.out = out;
  tail.aux = x;
  tail.snr_db = pl->ssi_snr_db;
  // the coloured noise goes into `out` and is mixed in place while still in L2
  return launch_fir_bank(pl->ssi_noise, len, B, ld, pl->ssi_taps, pl->ssi_tap_off, 1, 1, 0, out, w.stats_a, nullptr, 0, tail, st);
}

// normWav: x -> out (out may equal x), or with `add`: normWav(x + add) -> out
int do_normwav(const float* x, const float* add, const int32_t* len, int B, int ld, int always, float* out, const Workspace& w,
               cudaStream_t st) {
  return launch_norm_stream(x, add, len, B, ld, always, nullptr, nullptr, nullptr, 0.f, out, w.stats_a, st);
}

}  // namespace
}  // namespace rb

using namespace rb;

extern "C" {

const char* rb_error_string(int code) {
  switch (code) {
    case RB_OK: return "ok";
    case RB_ERR_INVALID_ARG: return "rawboost_b200: invalid argument";
    case RB_ERR_ALIGNMENT: return "rawboost_b200: ld must be a multiple of 4 and waveform/workspace pointers 16/256-byte aligned";
    case RB_ERR_WORKSPACE: return "rawboost_b200: workspace missing or smaller than rb_workspace_bytes()";
    case RB_ERR_NO_DEVICE: return "rawboost_b200: no usable CUDA device (needs compute capability 10.0)";
    case RB_ERR_PLAN: return "rawboost_b200: a plan field required by this algo is NULL";
    case RB_ERR_UNSUPPORTED: return "rawboost_b200: arguments outside what the planner supports (cascades <= 1024 taps and stages <= 255 taps on the device; nBands / N_f >= 1, P >= 0)";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "rawboost_b200: unknown error";
}

int rb_abi_version(void) { return RB_ABI_VERSION; }

size_t rb_workspace_bytes(int B, int ld) {
  if (B <= 0 || ld <= 0) return 0;
  return carve(nullptr, B, ld, 2).bytes;
}

size_t rb_workspace_bytes_for(int algo, int B, int ld) {
  if (B <= 0 || ld <= 0) return 0;
  return carve(nullptr, B, ld, scratch_waveforms(algo)).bytes;
}

uint64_t rb_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int rb_profile_enable(int on) {
  g_profile_on.store(on ? 1 : 0, std::memory_order_relaxed);
  return RB_OK;
}

int rb_profile_read(double* fir_ms, uint64_t* fir_launches, int reset) {
  std::lock_guard<std::mutex> lk(g_profile_mu);
  for (size_t i = 0; i + 1 < g_profile_events.size(); i += 2) {
    float ms = 0.f;
    RB_CUDA(cudaEventSynchronize(g_profile_events[i + 1]));
    RB_CUDA(cudaEventElapsedTime(&ms, g_profile_events[i], g_profile_events[i + 1]));
    g_profile_ms += (double)ms;
    g_profile_launches += 1;
  }
  for (cudaEvent_t e : g_profile_events) cudaEventDestroy(e);
  g_profile_events.clear();
  if (fir_ms) *fir_ms = g_profile_ms;
  if (fir_launches) *fir_launches = g_profile_launches;
  if (reset) {
    g_profile_ms = 0.0;
    g_profile_launches = 0;
  }
  return RB_OK;
}

int rb_filter_fir(const float* x, const int32_t* len, int B, int ld, const float* taps, const int32_t* tap_off, float* y,
                  void* stream) {
  RB_TRY(check_batch(x, len, B, ld, y));
  if (B == 0 || ld == 0) return RB_OK;
  if (!taps || !tap_off || x == y) return RB_ERR_INVALID_ARG;  // not in-place safe: a tile reads its neighbours' samples
  return launch_fir_bank(x, len, B, ld, taps, tap_off, 1, 1, 0, y, nullptr, nullptr, 0, FirTail(), (cudaStream_t)stream);
}

int rb_normwav(const float* x, const int32_t* len, int B, int ld, int always, float* y, void* workspace, size_t workspace_bytes,
               void* stream) {
  RB_TRY(check_batch(x, len, B, ld, y));
  if (B == 0 || ld == 0) return RB_OK;
  Workspace w;
  RB_TRY(check_ws(workspace, workspace_bytes, B, ld, 0, &w));
  return do_normwav(x, nullptr, len, B, ld, always, y, w, (cudaStream_t)stream);
}

int rb_lnl(const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
           size_t workspace_bytes, void* stream) {
  return rb_process(1, x, len, B, ld, plan, y, workspace, workspace_bytes, stream);
}
int rb_isd(const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
           size_t workspace_bytes, void* stream) {
  return rb_process(2, x, len, B, ld, plan, y, workspace, workspace_bytes, stream);
}
int rb_ssi(const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
           size_t workspace_bytes, void* stream) {
  return rb_process(3, x, len, B, ld, plan, y, workspace, workspace_bytes, stream);
}

int rb_process(int algo, const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y, void* workspace,
               size_t workspace_bytes, void* stream) {
  RB_TRY(check_batch(x, len, B, ld, y));
  if (B == 0 || ld == 0) return RB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (algo < 1 || algo > 8) {  // identity (asvspoof_2019_augall_3.py:435-437)
    if (x != y) RB_CUDA(cudaMemcpyAsync(y, x, (size_t)B * ld * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return RB_OK;
  }
  if (x == y) return RB_ERR_INVALID_ARG;
  Workspace w;
  RB_TRY(check_ws(workspace, workspace_bytes, B, ld, algo, &w));
  switch (algo) {
    case 1: return do_lnl(x, len, B, ld, plan, false, y, w, st);
    case 2: return do_isd(x, len, B, ld, plan, y, w, st);
    case 3: return do_ssi(x, len, B, ld, plan, y, w, st);
    case 4:
      RB_TRY(do_lnl(x, len, B, ld, plan, true, w.buf1, w, st));
      return do_ssi(w.buf1, len, B, ld, plan, y, w, st);
    case 5: return do_lnl(x, len, B, ld, plan, true, y, w, st);
    case 6:
      RB_TRY(do_lnl(x, len, B, ld, plan, false, w.buf1, w, st));
      return do_ssi(w.buf1, len, B, ld, plan, y, w, st);
    case 7:
      RB_TRY(do_isd(x, len, B, ld, plan, w.buf1, w, st));
      return do_ssi(w.buf1, len, B, ld, plan, y, w, st);
    case 8:
      RB_TRY(do_lnl(x, len, B, ld, plan, false, w.buf1, w, st));
      RB_TRY(do_isd(x, len, B, ld, plan, w.buf2, w, st));
      return do_normwav(w.buf1, w.buf2, len, B, ld, 0, y, w, st);  // the sum of the branches is formed inside the streaming pass
  }
  return RB_ERR_INVALID_ARG;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// host-buffer context: a chunked three-stage pipeline (H2D | plan + kernels | D2H)
// ---------------------------------------------------------------------------------------------------
namespace {
constexpr int kSlots = 8;

struct Slot {
  char* dev = nullptr;
  size_t bytes = 0;
  cudaEvent_t ev_in = nullptr, ev_done = nullptr, ev_out = nullptr;
};
}  // namespace

// Resources one call owns while it is in flight; two sets, so that a second call can be submitted while the first drains.
struct CallRes {
  char* meta = nullptr;  // device copy of len[] and seeds[]
  size_t meta_bytes = 0;
  char* planmem = nullptr;  // device-drawn plans of the whole batch (rb_process_host_seeded)
  size_t planmem_bytes = 0;
  std::vector<cudaEvent_t> ev_planned;  // one per chunk
  std::vector<cudaEvent_t> ev_body;     // one per planner piece
  cudaEvent_t ev_meta = nullptr, ev_done = nullptr, ev_user = nullptr;
  bool inflight = false;
  uint64_t ticket = 0;
};

struct rb_ctx {
  int device;
  int sm_count;
  int chunk;  // utterances per pipeline chunk (0: four per SM)
  cudaStream_t s_in, s_plan, s_apply, s_cmp, s_out;
  Slot slot[kSlots];
  uint64_t seq = 0;    // chunks issued so far (slot = seq % kSlots)
  uint64_t calls = 0;  // calls issued so far (resources = calls % 2)
  CallRes res[2];
  uint64_t h2d, d2h;
  int trace = 0;                 // rb_ctx_trace: record a per-chunk timeline of the next calls
  std::vector<double> timeline;  // per chunk: first utterance, utterances, ms at which copy-in / plan / kernels / copy-out ended
};

namespace {

// Grow a device buffer to hold `need` bytes (allocating need + slack) once the device has drained: queued work may still use it.
int grow(char*& p, size_t& bytes, size_t need, size_t slack) {
  if (need <= bytes) return RB_OK;
  RB_CUDA(cudaDeviceSynchronize());
  if (p) RB_CUDA(cudaFree(p));
  p = nullptr;
  bytes = 0;
  RB_CUDA(cudaMalloc((void**)&p, need + slack));
  bytes = need + slack;
  return RB_OK;
}

int add_events(std::vector<cudaEvent_t>& v, int n) {
  while ((int)v.size() < n) {
    cudaEvent_t e;
    RB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    v.push_back(e);
  }
  return RB_OK;
}

struct Take {
  size_t off = 0;
  size_t operator()(size_t n) {
    const size_t r = off;
    off += align_up(n, 256);
    return r;
  }
};

// Where a call's waveforms come from and where its results go.
struct IoSpec {
  const void* x = nullptr;
  int x_kind = RB_IO_HOST_F32;   // RB_IO_HOST_F32 | RB_IO_HOST_PCM16 | RB_IO_DEVICE_F32 (then len / seeds are device arrays too)
  void* y = nullptr;
  int y_kind = RB_IO_HOST_F32;   // RB_IO_HOST_F32 | RB_IO_DEVICE_F32
  cudaStream_t user = nullptr;   // device-side ordering: the call starts after the work queued on it and (has_user) it waits for the call
  bool has_user = false;
  const int64_t* off = nullptr;  // packed host I/O: utterance u is x[off[u], off[u + 1]) (host int64[B + 1]); a host y is packed alike
};

// Events of a traced synchronous call (rb_ctx_trace): [0] its start, [1..4] per chunk: copy-in, plan, kernels, copy-out done.
struct Trace {
  bool on;
  std::vector<cudaEvent_t> ev[5];
  void mark(int stage, cudaStream_t st) {
    if (!on) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) == cudaSuccess) {
      cudaEventRecord(e, st);
      ev[stage].push_back(e);
    }
  }
  // rb_ctx_timeline's rows, once the device has drained (none if an event could not be created)
  void rows(const std::vector<int>& first, std::vector<double>& out) const {
    const size_t nchunks = first.size() - 1;
    bool complete = ev[0].size() == 1;
    for (int k = 1; k < 5; ++k) complete = complete && ev[k].size() == nchunks;
    if (!complete) return;
    for (size_t ci = 0; ci < nchunks; ++ci) {
      out.push_back((double)first[ci]);
      out.push_back((double)(first[ci + 1] - first[ci]));
      for (int k = 1; k < 5; ++k) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[0][0], ev[k][ci]);
        out.push_back((double)ms);
      }
    }
  }
  ~Trace() {
    for (auto& v : ev)
      for (cudaEvent_t e : v) cudaEventDestroy(e);
  }
};

// ---- host CSR plan (rb_process_host): each chunk's slices are uploaded beside its waveforms ---------------------------------
struct HostPlanSlots {  // slot offsets of the slices
  size_t lnl_off, lnl_taps, isd_off, isd_idx, isd_fr, ssi_noise, ssi_off, ssi_taps, ssi_snr;
};

// Slot space for the slices of chunks of at most `chunk` utterances, the tap and impulse arrays sized for the largest payload.
HostPlanSlots host_plan_slots(Take& take, const rb_plan* plan, int algo, const std::vector<int>& first, int chunk, int ld) {
  const bool lnl = algo_uses_lnl(algo), isd = algo_uses_isd(algo), ssi = algo_uses_ssi(algo);
  const int n_f = plan->n_f;
  size_t max_lt = 0, max_isd = 0, max_st = 0;
  for (size_t ci = 0; ci + 1 < first.size(); ++ci) {
    const int u0 = first[ci], u1 = first[ci + 1];
    if (lnl) max_lt = std::max(max_lt, (size_t)(plan->lnl_tap_off[(size_t)u1 * n_f] - plan->lnl_tap_off[(size_t)u0 * n_f]));
    if (isd) max_isd = std::max(max_isd, (size_t)(plan->isd_off[u1] - plan->isd_off[u0]));
    if (ssi) max_st = std::max(max_st, (size_t)(plan->ssi_tap_off[u1] - plan->ssi_tap_off[u0]));
  }
  HostPlanSlots o;
  o.lnl_off = take(lnl ? ((size_t)chunk * n_f + 1) * 4 : 0);
  o.lnl_taps = take(max_lt * 4);
  o.isd_off = take(isd ? (size_t)(chunk + 1) * 4 : 0);
  o.isd_idx = take(max_isd * 4);
  o.isd_fr = take(max_isd * 8);
  o.ssi_noise = take(ssi ? (size_t)chunk * ld * sizeof(float) : 0);
  o.ssi_off = take(ssi ? (size_t)(chunk + 1) * 4 : 0);
  o.ssi_taps = take(max_st * 4);
  o.ssi_snr = take(ssi ? (size_t)chunk * 4 : 0);
  return o;
}

// Copy the slices of utterances [u0, u0 + bc) into slot memory d on stream st and return the chunk's plan in *dp. CSR slices
// keep their absolute offsets; the value pointers are rebased so that ptr[off] lands in the slice.
int upload_plan_slice(const rb_plan* plan, int algo, const HostPlanSlots& o, char* d, int u0, int bc, int ld, cudaStream_t st,
                      uint64_t& h2d, rb_plan* dp) {
  const int n_f = plan->n_f;
  memset(dp, 0, sizeof(*dp));
  dp->n_f = n_f;
  dp->g_sd = plan->g_sd;
  auto up = [&](size_t off, const void* src, size_t n) -> int {
    if (n == 0) return RB_OK;
    h2d += n;
    return (int)cudaMemcpyAsync(d + off, src, n, cudaMemcpyHostToDevice, st);
  };
  if (algo_uses_lnl(algo)) {
    const int32_t* off = plan->lnl_tap_off + (size_t)u0 * n_f;
    const size_t base = (size_t)off[0], cnt = (size_t)off[(size_t)bc * n_f] - base;
    RB_TRY(up(o.lnl_off, off, ((size_t)bc * n_f + 1) * 4));
    RB_TRY(up(o.lnl_taps, plan->lnl_taps + base, cnt * 4));
    dp->lnl_tap_off = (const int32_t*)(d + o.lnl_off);
    dp->lnl_taps = (const float*)(d + o.lnl_taps) - base;
  }
  if (algo_uses_isd(algo)) {
    const int32_t* off = plan->isd_off + u0;
    const size_t base = (size_t)off[0], cnt = (size_t)off[bc] - base;
    RB_TRY(up(o.isd_off, off, (size_t)(bc + 1) * 4));
    RB_TRY(up(o.isd_idx, plan->isd_idx + base, cnt * 4));
    RB_TRY(up(o.isd_fr, plan->isd_fr + base, cnt * 8));
    dp->isd_off = (const int32_t*)(d + o.isd_off);
    dp->isd_idx = (const int32_t*)(d + o.isd_idx) - base;
    dp->isd_fr = (const double*)(d + o.isd_fr) - base;
  }
  if (algo_uses_ssi(algo)) {
    const int32_t* off = plan->ssi_tap_off + u0;
    const size_t base = (size_t)off[0], cnt = (size_t)off[bc] - base;
    RB_TRY(up(o.ssi_noise, plan->ssi_noise + (size_t)u0 * ld, (size_t)bc * ld * sizeof(float)));
    RB_TRY(up(o.ssi_off, off, (size_t)(bc + 1) * 4));
    RB_TRY(up(o.ssi_taps, plan->ssi_taps + base, cnt * 4));
    RB_TRY(up(o.ssi_snr, plan->ssi_snr_db + u0, (size_t)bc * 4));
    dp->ssi_noise = (const float*)(d + o.ssi_noise);
    dp->ssi_tap_off = (const int32_t*)(d + o.ssi_off);
    dp->ssi_taps = (const float*)(d + o.ssi_taps) - base;
    dp->ssi_snr_db = (const float*)(d + o.ssi_snr);
  }
  return RB_OK;
}

// ---- device plan (the seeded entries): drawn for the whole batch, read in place -----------------------------------------
// The slice of utterances [u0, ...): CSR offsets are absolute, so only the owner arrays move.
rb_plan device_plan_slice(const rb_plan& whole, int u0, int ld) {
  rb_plan dp = whole;
  if (dp.lnl_tap_off) dp.lnl_tap_off += (size_t)u0 * dp.n_f;
  if (dp.isd_off) dp.isd_off += u0;
  if (dp.ssi_tap_off) {
    dp.ssi_noise += (size_t)u0 * ld;
    dp.ssi_tap_off += u0;
    dp.ssi_snr_db += u0;
  }
  return dp;
}

// Queue the device planner of a whole call; R.ev_planned[ci] fires once chunk ci's plan is complete. The plans need only
// lengths and seeds. Its kernels are latency-bound (one warp per utterance: the stream replay of one utterance takes ~2 ms
// however few utterances a launch holds), so they are issued in pieces -- chunk 0, chunk 1, then about 4096 utterances at a
// time (one full wave of the replay kernel) -- so that the first results leave early (a host-buffer call is bound by the
// copy-out stream, which starts with the first filtered chunk) while large batches pay the replay latency once per wave, not
// once per chunk. Stream replay runs on s_plan, swap application on s_apply, both at low priority beside the kernels.
// Measured (scripts/gpu_overlap_probe.py): while the FIR-bank kernel still has CTAs to dispatch, the hardware does not place
// another kernel's CTAs in the registers / shared memory its resident CTAs leave free, so the planner really runs in the
// gaps: during copies, at the tail of each FIR launch, and before the first chunk.
int queue_devplan(rb_ctx* c, CallRes& R, const rb_args* args, int algo, int B, int ld, const int32_t* d_len, const uint32_t* d_seeds,
                  const std::vector<int>& first, int chunk, bool x_dev, Trace& trace, rb_plan* whole) {
  const bool ssi = algo_uses_ssi(algo);
  const int nchunks = (int)first.size() - 1;
  std::vector<int> piece_end;  // one past the last chunk of each piece
  if (!ssi && nchunks >= 3) {  // SSI tap offsets need the stream positions of every utterance: one piece
    const int per_wave = std::max(1, 4096 / chunk);
    if (!x_dev) {
      piece_end.push_back(1);
      piece_end.push_back(2);
    }
    while ((piece_end.empty() ? 0 : piece_end.back()) < nchunks)
      piece_end.push_back(std::min(nchunks, (piece_end.empty() ? 0 : piece_end.back()) + per_wave));
  } else {
    piece_end.push_back(nchunks);
  }
  RB_TRY(add_events(R.ev_planned, nchunks));
  RB_TRY(add_events(R.ev_body, (int)piece_end.size()));
  RB_TRY(devplan_begin(args, algo, B, ld, d_len, d_seeds, R.planmem, R.planmem_bytes, whole, c->s_plan));
  for (int pc = 0; pc < (int)piece_end.size(); ++pc) {
    const int cb = pc ? piece_end[pc - 1] : 0;
    const int u0 = first[cb], u1 = first[piece_end[pc]];
    RB_TRY(devplan_body(args, algo, B, ld, d_len, d_seeds, R.planmem, u0, u1 - u0, c->s_plan));
    if (ssi) RB_TRY(devplan_end(args, algo, B, ld, R.planmem, c->s_plan));
    RB_CUDA(cudaEventRecord(R.ev_body[pc], c->s_plan));
    RB_CUDA(cudaStreamWaitEvent(c->s_apply, R.ev_body[pc], 0));
    for (int ci = cb; ci < piece_end[pc]; ++ci) {
      RB_TRY(devplan_apply(args, algo, B, ld, d_len, R.planmem, first[ci], first[ci + 1] - first[ci], c->s_apply));
      RB_CUDA(cudaEventRecord(R.ev_planned[ci], c->s_apply));
      trace.mark(2, c->s_apply);
    }
  }
  return RB_OK;
}

// Common driver. plan != NULL: host CSR plan, sliced and uploaded per chunk. plan == NULL: seeds/args given, drawn on the device.
int run_pipeline(rb_ctx* c, int algo, const IoSpec& io, const int32_t* len, int B, int ld, const rb_plan* plan, const rb_args* args,
                 const uint32_t* seeds, bool async, uint64_t* ticket) {
  const bool x_dev = io.x_kind == RB_IO_DEVICE_F32, x_pcm = io.x_kind == RB_IO_HOST_PCM16, y_dev = io.y_kind == RB_IO_DEVICE_F32;
  const bool packed = io.off != nullptr;
  const size_t elem = x_pcm ? 2 : 4;
  const float* x = (const float*)io.x;
  float* y = (float*)io.y;
  RB_CUDA(cudaSetDevice(c->device));
  CallRes& R = c->res[c->calls & 1];
  if (R.inflight) {  // at most two calls in flight: the one that used this resource set must be complete
    RB_CUDA(cudaEventSynchronize(R.ev_done));
    R.inflight = false;
  }
  const bool active = algo >= 1 && algo <= 8;
  const bool devplan = active && plan == nullptr;
  const int chunk = std::max(1, std::min(B, c->chunk > 0 ? c->chunk : 4 * c->sm_count));
  // Equal chunks. Shorter chunks at the start and / or the end (to get the first results out earlier, to shorten the last
  // copy-out) were measured and do not help: with both PCIe directions busy the call is bound by the two ~22 ms copy streams
  // and their mutual offset of one chunk's filtering.
  std::vector<int> first;  // first utterance of each chunk, plus B
  for (int u = 0; u < B; u += chunk) first.push_back(u);
  first.push_back(B);
  const int nchunks = (int)first.size() - 1;

  // everything queued below is ordered by events only; the host blocks once, at the end
  // per-call metadata: lengths (+ seeds) for the whole batch, and the offsets of packed I/O
  const size_t meta4 = align_up((size_t)B * 4, 256);
  RB_TRY(grow(R.meta, R.meta_bytes, meta4 * 2 + (packed ? (size_t)(B + 1) * 8 : 0), 0));
  const int32_t* d_len = (int32_t*)R.meta;
  const uint32_t* d_seeds = (uint32_t*)(R.meta + meta4);
  const int64_t* d_off = (const int64_t*)(R.meta + meta4 * 2);
  uint64_t h2d = 0, d2h = 0;
  if (io.has_user || x_dev) {  // everything of this call comes after what the caller queued on its stream
    RB_CUDA(cudaEventRecord(R.ev_user, io.user));
    RB_CUDA(cudaStreamWaitEvent(c->s_in, R.ev_user, 0));
  }
  if (x_dev) {  // lengths and seeds are already on the device
    d_len = len;
    d_seeds = seeds;
  } else {
    if (packed) {  // the offsets go up from the caller's buffer; the lengths are their differences
      RB_CUDA(cudaMemcpyAsync((void*)d_off, io.off, (size_t)(B + 1) * 8, cudaMemcpyHostToDevice, c->s_in));
      h2d += (size_t)(B + 1) * 8;
      RB_TRY(launch_lengths_from_offsets(d_off, B, (int32_t*)d_len, c->s_in));
    } else {
      RB_CUDA(cudaMemcpyAsync((void*)d_len, len, (size_t)B * 4, cudaMemcpyHostToDevice, c->s_in));
      h2d += (size_t)B * 4;
    }
    if (devplan) {
      RB_CUDA(cudaMemcpyAsync((void*)d_seeds, seeds, (size_t)B * 4, cudaMemcpyHostToDevice, c->s_in));
      h2d += (size_t)B * 4;
    }
  }
  RB_CUDA(cudaEventRecord(R.ev_meta, c->s_in));
  RB_CUDA(cudaStreamWaitEvent(c->s_plan, R.ev_meta, 0));
  RB_CUDA(cudaStreamWaitEvent(c->s_cmp, R.ev_meta, 0));

  // slot layout for the largest chunk
  const size_t wave = (size_t)chunk * ld * sizeof(float);
  const size_t ws_bytes = active ? rb_workspace_bytes_for(algo, chunk, ld) : 0;
  const size_t dp_bytes = devplan ? rb_devplan_bytes(args, algo, B, ld) : 0;
  if (devplan && dp_bytes == 0) return RB_ERR_UNSUPPORTED;
  RB_TRY(grow(R.planmem, R.planmem_bytes, dp_bytes, dp_bytes / 8));
  Take take;
  const size_t o_x = take(x_dev ? 0 : wave), o_x16 = take(x_pcm && !packed ? wave / 2 : 0), o_y = take(y_dev ? 0 : wave);
  // Packed input is staged in the output rows, which are free until the kernels write them, and packed results in the input
  // rows, which are free once the kernels are done. A device sink has no output rows: its input gets a staging area sized by
  // the largest chunk span.
  size_t max_span = 0;
  if (packed)
    for (int ci = 0; ci < nchunks; ++ci) max_span = std::max(max_span, (size_t)(io.off[first[ci + 1]] - io.off[first[ci]]));
  const size_t o_pin = packed && y_dev ? take(elem * max_span) : o_y, o_pout = o_x;
  const size_t o_ws = take(ws_bytes);
  HostPlanSlots hp{};
  if (active && !devplan) hp = host_plan_slots(take, plan, algo, first, chunk, ld);
  for (int k = 0; k < std::min(kSlots, nchunks); ++k) {
    Slot& sl = c->slot[(c->seq + k) % kSlots];
    RB_TRY(grow(sl.dev, sl.bytes, take.off, take.off / 8));
  }

  Trace trace{c->trace && !async};
  trace.mark(0, c->s_in);
  rb_plan whole{};
  if (devplan) RB_TRY(queue_devplan(c, R, args, algo, B, ld, d_len, d_seeds, first, chunk, x_dev, trace, &whole));
  for (int ci = 0; ci < nchunks; ++ci) {
    Slot& sl = c->slot[(c->seq + ci) % kSlots];
    char* d = sl.dev;
    const int u0 = first[ci], bc = first[ci + 1] - u0;
    const size_t cw = (size_t)bc * ld * sizeof(float);
    const int64_t p0 = packed ? io.off[u0] : 0, pn = packed ? io.off[u0 + bc] - p0 : 0;  // the chunk's packed span
    // ---- stage 1: host -> device: the waveforms and, of a host plan, the chunk's slices -------------------------------
    if (c->seq + ci >= kSlots) RB_CUDA(cudaStreamWaitEvent(c->s_in, sl.ev_out, 0));  // the slot's previous chunk has left the device
    if (packed) {  // one copy of the contiguous span, whatever the number of utterances
      if (pn) RB_CUDA(cudaMemcpyAsync(d + o_pin, (const char*)io.x + elem * p0, elem * pn, cudaMemcpyHostToDevice, c->s_in));
      h2d += elem * pn;
    } else if (x_pcm) {
      RB_CUDA(cudaMemcpyAsync(d + o_x16, (const int16_t*)io.x + (size_t)u0 * ld, cw / 2, cudaMemcpyHostToDevice, c->s_in));
      h2d += cw / 2;
    } else if (!x_dev) {
      RB_CUDA(cudaMemcpyAsync(d + o_x, x + (size_t)u0 * ld, cw, cudaMemcpyHostToDevice, c->s_in));
      h2d += cw;
    }
    rb_plan dp{};
    if (devplan) dp = device_plan_slice(whole, u0, ld);
    else if (active) RB_TRY(upload_plan_slice(plan, algo, hp, d, u0, bc, ld, c->s_in, h2d, &dp));
    RB_CUDA(cudaEventRecord(sl.ev_in, c->s_in));
    trace.mark(1, c->s_in);
    // ---- stage 2: kernels, once the chunk's plan (drawn beside the previous chunks' kernels) and waveforms are there ------
    if (devplan) RB_CUDA(cudaStreamWaitEvent(c->s_cmp, R.ev_planned[ci], 0));
    else trace.mark(2, c->s_in);
    RB_CUDA(cudaStreamWaitEvent(c->s_cmp, sl.ev_in, 0));
    if (packed) {
      RB_TRY(launch_unpack_rows(d + o_pin, x_pcm, d_off + u0, bc, ld, (float*)(d + o_x), c->s_cmp));
    } else if (x_pcm) {
      RB_TRY(launch_pcm16_to_f32((const int16_t*)(d + o_x16), (float*)(d + o_x), (size_t)bc * ld, c->s_cmp));
    }
    const float* xin = x_dev ? x + (size_t)u0 * ld : (const float*)(d + o_x);
    float* yout = y_dev ? y + (size_t)u0 * ld : (float*)(d + o_y);
    RB_TRY(rb_process(algo, xin, d_len + u0, bc, ld, active ? &dp : nullptr, yout, d + o_ws, ws_bytes, c->s_cmp));
    if (packed && !y_dev) RB_TRY(launch_pack_rows(yout, d_off + u0, bc, ld, (float*)(d + o_pout), c->s_cmp));
    RB_CUDA(cudaEventRecord(sl.ev_done, c->s_cmp));
    trace.mark(3, c->s_cmp);
    // ---- stage 3: device -> host (or nothing: the results stay where the kernels wrote them) ---------------------------
    if (y_dev) {
      RB_CUDA(cudaEventRecord(sl.ev_out, c->s_cmp));
    } else {
      RB_CUDA(cudaStreamWaitEvent(c->s_out, sl.ev_done, 0));
      if (packed) {
        if (pn) RB_CUDA(cudaMemcpyAsync(y + p0, d + o_pout, 4 * pn, cudaMemcpyDeviceToHost, c->s_out));
        d2h += 4 * pn;
      } else {
        RB_CUDA(cudaMemcpyAsync(y + (size_t)u0 * ld, d + o_y, cw, cudaMemcpyDeviceToHost, c->s_out));
        d2h += cw;
      }
      RB_CUDA(cudaEventRecord(sl.ev_out, c->s_out));
    }
    trace.mark(4, y_dev ? c->s_cmp : c->s_out);
  }
  c->seq += (uint64_t)nchunks;
  RB_CUDA(cudaEventRecord(R.ev_done, y_dev ? c->s_cmp : c->s_out));
  if (io.has_user) RB_CUDA(cudaStreamWaitEvent(io.user, R.ev_done, 0));  // the caller's stream continues after the results exist
  R.inflight = true;
  R.ticket = ++c->calls;
  if (ticket) *ticket = R.ticket;
  c->h2d = h2d;
  c->d2h = d2h;
  if (async) return RB_OK;  // the caller collects the results with rb_ctx_wait
  RB_CUDA(cudaEventSynchronize(R.ev_done));
  R.inflight = false;
  if (c->trace) {
    c->timeline.clear();
    RB_CUDA(cudaDeviceSynchronize());
    trace.rows(first, c->timeline);
  }
  return RB_OK;
}

int check_host_batch(const rb_ctx* c, const void* x, const int32_t* len, int B, int ld, const void* y) {
  if (!c) return RB_ERR_INVALID_ARG;
  if (B < 0 || ld < 0) return RB_ERR_INVALID_ARG;
  if (B == 0 || ld == 0) return RB_OK;
  if (!x || !len || !y) return RB_ERR_INVALID_ARG;
  if (ld % 4 != 0) return RB_ERR_ALIGNMENT;
  return RB_OK;
}

// The seeded entries: argument checks, then the pipeline with the plans drawn on the device.
int run_seeded(rb_ctx* c, int algo, const rb_args* args, const void* x, int x_kind, const int32_t* len, const uint32_t* seeds, int B,
               int ld, void* y, int y_kind, void* user_stream, int use_user_stream, bool async, uint64_t* ticket) {
  if (ticket) *ticket = 0;
  if (x_kind != RB_IO_HOST_F32 && x_kind != RB_IO_HOST_PCM16 && x_kind != RB_IO_DEVICE_F32) return RB_ERR_INVALID_ARG;
  if (y_kind != RB_IO_HOST_F32 && y_kind != RB_IO_DEVICE_F32) return RB_ERR_INVALID_ARG;
  RB_TRY(check_host_batch(c, x, len, B, ld, y));
  if (B == 0 || ld == 0) return RB_OK;
  if (algo >= 1 && algo <= 8 && (!args || !seeds)) return RB_ERR_INVALID_ARG;
  if (x_kind == RB_IO_DEVICE_F32 && !use_user_stream) return RB_ERR_INVALID_ARG;  // device input needs the stream that produced it
  if ((x_kind == RB_IO_DEVICE_F32 && ((uintptr_t)x & 15u)) || (y_kind == RB_IO_DEVICE_F32 && ((uintptr_t)y & 15u))) return RB_ERR_ALIGNMENT;
  if (x_kind == RB_IO_DEVICE_F32 && x == y && algo >= 1 && algo <= 8) return RB_ERR_INVALID_ARG;
  if (x_kind == RB_IO_HOST_PCM16 && ld % 8 != 0) return RB_ERR_ALIGNMENT;
  const IoSpec io{x, x_kind, y, y_kind, (cudaStream_t)user_stream, use_user_stream != 0};
  return run_pipeline(c, algo, io, len, B, ld, nullptr, args, seeds, async, ticket);
}

}  // namespace

extern "C" {

int rb_ctx_create(rb_ctx** out, int device) {
  if (!out) return RB_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return RB_ERR_NO_DEVICE;
  cudaDeviceProp prop;
  RB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return RB_ERR_NO_DEVICE;
  RB_CUDA(cudaSetDevice(device));
  rb_ctx* c = new (std::nothrow) rb_ctx();
  if (!c) return RB_ERR_INVALID_ARG;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->chunk = 0;
  c->h2d = c->d2h = 0;
  c->s_in = c->s_plan = c->s_apply = c->s_cmp = c->s_out = nullptr;
  // Stream priorities: copies first, then the FIR kernel's stream, the planner's streams last. The planner only needs to stay
  // ahead of the filtering (it is ~2.5x faster per chunk), so it runs in the gaps -- while the filtering waits for the next
  // chunk's waveforms, and in whatever an SM has left beside the FIR-bank CTAs -- instead of displacing them: measured 27.3 ms
  // per 4096 utterances against 29.6 ms with the planner's streams on top.
  int prio_lo = 0, prio_hi = 0;
  cudaError_t e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  for (cudaStream_t* s : {&c->s_in, &c->s_out, &c->s_cmp})
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, prio_hi);
  for (cudaStream_t* s : {&c->s_plan, &c->s_apply})
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, prio_lo);
  for (CallRes& R : c->res)
    for (cudaEvent_t* ev : {&R.ev_meta, &R.ev_done, &R.ev_user})
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
  for (Slot& sl : c->slot)
    for (cudaEvent_t* ev : {&sl.ev_in, &sl.ev_done, &sl.ev_out})
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    rb_ctx_destroy(c);
    return (int)e;
  }
  *out = c;
  return RB_OK;
}

int rb_ctx_destroy(rb_ctx* c) {
  if (!c) return RB_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (Slot& sl : c->slot) {
    if (sl.dev) cudaFree(sl.dev);
    for (cudaEvent_t ev : {sl.ev_in, sl.ev_done, sl.ev_out})
      if (ev) cudaEventDestroy(ev);
  }
  for (CallRes& R : c->res) {
    if (R.meta) cudaFree(R.meta);
    if (R.planmem) cudaFree(R.planmem);
    for (cudaEvent_t e : R.ev_planned) cudaEventDestroy(e);
    for (cudaEvent_t e : R.ev_body) cudaEventDestroy(e);
    for (cudaEvent_t e : {R.ev_meta, R.ev_done, R.ev_user})
      if (e) cudaEventDestroy(e);
  }
  for (cudaStream_t s : {c->s_in, c->s_plan, c->s_apply, c->s_cmp, c->s_out})
    if (s) cudaStreamDestroy(s);
  delete c;
  return RB_OK;
}

int rb_ctx_set_chunk(rb_ctx* c, int utterances) {
  if (!c || utterances < 0) return RB_ERR_INVALID_ARG;
  c->chunk = utterances;
  return RB_OK;
}

int rb_ctx_trace(rb_ctx* c, int on) {
  if (!c) return RB_ERR_INVALID_ARG;
  c->trace = on ? 1 : 0;
  return RB_OK;
}

int rb_ctx_timeline(const rb_ctx* c, double* out, int capacity) {
  if (!c || capacity < 0 || (capacity > 0 && !out)) return RB_ERR_INVALID_ARG;
  const int n = (int)std::min<size_t>(c->timeline.size(), (size_t)capacity);
  for (int i = 0; i < n; ++i) out[i] = c->timeline[i];
  return (int)c->timeline.size();
}

int rb_ctx_last_traffic(const rb_ctx* c, uint64_t* h2d, uint64_t* d2h) {
  if (!c) return RB_ERR_INVALID_ARG;
  if (h2d) *h2d = c->h2d;
  if (d2h) *d2h = c->d2h;
  return RB_OK;
}

int rb_process_host(rb_ctx* c, int algo, const float* x, const int32_t* len, int B, int ld, const rb_plan* plan, float* y) {
  RB_TRY(check_host_batch(c, x, len, B, ld, y));
  if (B == 0 || ld == 0) return RB_OK;
  if (algo >= 1 && algo <= 8) {
    if (!plan) return RB_ERR_PLAN;
    if (algo_uses_lnl(algo) && (plan->n_f < 1 || !plan->lnl_taps || !plan->lnl_tap_off)) return RB_ERR_PLAN;
    if (algo_uses_isd(algo) && (!plan->isd_off || !plan->isd_idx || !plan->isd_fr)) return RB_ERR_PLAN;
    if (algo_uses_ssi(algo) && (!plan->ssi_noise || !plan->ssi_taps || !plan->ssi_tap_off || !plan->ssi_snr_db)) return RB_ERR_PLAN;
  }
  IoSpec io;
  io.x = x;
  io.y = y;
  return run_pipeline(c, algo, io, len, B, ld, plan, nullptr, nullptr, false, nullptr);
}

int rb_process_host_seeded(rb_ctx* c, int algo, const rb_args* args, const float* x, const int32_t* len, const uint32_t* seeds, int B,
                           int ld, float* y) {
  return run_seeded(c, algo, args, x, RB_IO_HOST_F32, len, seeds, B, ld, y, RB_IO_HOST_F32, nullptr, 0, false, nullptr);
}

int rb_submit_host_seeded(rb_ctx* c, int algo, const rb_args* args, const float* x, const int32_t* len, const uint32_t* seeds, int B,
                          int ld, float* y, uint64_t* ticket) {
  return rb_submit_seeded_ex(c, algo, args, x, RB_IO_HOST_F32, len, seeds, B, ld, y, RB_IO_HOST_F32, nullptr, 0, ticket);
}

int rb_submit_seeded_ex(rb_ctx* c, int algo, const rb_args* args, const void* x, int x_kind, const int32_t* len, const uint32_t* seeds,
                        int B, int ld, void* y, int y_kind, void* user_stream, int use_user_stream, uint64_t* ticket) {
  return run_seeded(c, algo, args, x, x_kind, len, seeds, B, ld, y, y_kind, user_stream, use_user_stream, true, ticket);
}

// The offsets are checked here, on the host, before anything is queued.
int rb_submit_seeded_packed(rb_ctx* c, int algo, const rb_args* args, const void* x, int x_kind, const int64_t* off,
                            const uint32_t* seeds, int B, int ld, void* y, int y_kind, void* user_stream, int use_user_stream,
                            uint64_t* ticket) {
  if (ticket) *ticket = 0;
  if (!c || B < 0 || ld < 0) return RB_ERR_INVALID_ARG;
  if (x_kind != RB_IO_HOST_F32 && x_kind != RB_IO_HOST_PCM16) return RB_ERR_INVALID_ARG;
  if (y_kind != RB_IO_HOST_F32 && y_kind != RB_IO_DEVICE_F32) return RB_ERR_INVALID_ARG;
  if (B == 0) return RB_OK;
  if (!x || !off || !y) return RB_ERR_INVALID_ARG;
  if (algo >= 1 && algo <= 8 && (!args || !seeds)) return RB_ERR_INVALID_ARG;
  if (off[0] != 0) return RB_ERR_INVALID_ARG;
  int64_t max_len = 0;
  for (int u = 0; u < B; ++u) {
    const int64_t n = off[u + 1] - off[u];
    if (n < 0 || n > INT32_MAX) return RB_ERR_INVALID_ARG;
    max_len = std::max(max_len, n);
  }
  if (y_kind == RB_IO_HOST_F32 && ld == 0) {  // the call's own stride
    if (max_len > INT32_MAX - 3) return RB_ERR_INVALID_ARG;
    ld = (int)align_up((size_t)max_len, 4);
  }
  if (ld < max_len) return RB_ERR_INVALID_ARG;
  if (ld % 4 != 0 || (y_kind == RB_IO_DEVICE_F32 && ((uintptr_t)y & 15u))) return RB_ERR_ALIGNMENT;
  if (ld == 0) return RB_OK;  // every utterance is empty
  IoSpec io{x, x_kind, y, y_kind, (cudaStream_t)user_stream, use_user_stream != 0};
  io.off = off;
  return run_pipeline(c, algo, io, nullptr, B, ld, nullptr, args, seeds, true, ticket);
}

int rb_ctx_wait(rb_ctx* c, uint64_t ticket) {
  if (!c) return RB_ERR_INVALID_ARG;
  RB_CUDA(cudaSetDevice(c->device));
  for (CallRes& R : c->res) {
    if (R.inflight && (ticket == 0 || R.ticket <= ticket)) {  // 0: everything submitted so far
      RB_CUDA(cudaEventSynchronize(R.ev_done));
      R.inflight = false;
    }
  }
  return RB_OK;
}

}  // extern "C"
