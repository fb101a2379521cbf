// rb_planner.cpp -- native host-side plan drawing (host code only, compiled by g++; no kernels).
//
// The reference draws every random parameter of RawBoost from numpy's process-global legacy MT19937 stream
// (/root/reference/datautils/RawBoost.py:15,79,80,90). The Python path in plans.py issues those numpy calls itself and
// is the contract; this file is the fast equivalent for batched use: a bit-exact re-implementation of the pieces of
// numpy's legacy generator the path consumes --
//   seeding          np.random.seed(int)            -> mt19937_seed (Knuth LCG fill)
//   uniform          low + (high-low) * double53    -> two 32-bit words per double, (a>>5, b>>6)
//   permutation(n)   arange + legacy shuffle        -> Fisher-Yates from the end, masked rejection on 32-bit words
//   rand(n)          double53
//   normal(0,1,n)    legacy polar Box-Muller with the cached second value
// -- plus the float64 filter design of genNotchCoeffs (RawBoost.py:28-48: Hamming-windowed two-band firwin stages,
// cascade convolution, peak normalisation on the 512-point freqz grid). Integer results (tap counts, impulse count and
// positions) and the stream state are bit-identical to numpy's; tap values agree to ~1e-15 relative (libm vs numpy's SIMD
// sin/cos, radix-2 FFT vs pocketfft), far inside the float32 they are shipped as. tests/test_host_logic.py checks both.
//
// Utterances are drawn by a pool of host threads straight into page-locked CSR buffers laid out as struct rb_plan.
#include <math.h>
#include <string.h>
#include <atomic>
#include <thread>
#include <vector>

#include <cuda_runtime.h>  // cudaMallocHost for the page-locked plan buffers only
#include "rawboost_b200.h"
#include "rb_algo.h"

namespace {

constexpr int kMT = 624;

// One MT19937 block: advance the 624-word state in place and temper it into `out`. Compiled for AVX-512 / AVX2 / SSE2
// and dispatched at load time (the build machine is not the machine it runs on).
__attribute__((target_clones("avx512f", "avx2", "default")))
void mt_block(uint32_t* __restrict__ key, uint32_t* __restrict__ out, int advance) {
  constexpr uint32_t kUpper = 0x80000000u, kLower = 0x7fffffffu, kMatrix = 0x9908b0dfu;
  constexpr int N = kMT, M = 397;
  if (advance) {
    int i;
    for (i = 0; i < N - M; ++i) {
      const uint32_t y = (key[i] & kUpper) | (key[i + 1] & kLower);
      key[i] = key[i + M] ^ (y >> 1) ^ ((0u - (y & 1u)) & kMatrix);
    }
    for (; i < N - 1; ++i) {
      const uint32_t y = (key[i] & kUpper) | (key[i + 1] & kLower);
      key[i] = key[i - (N - M)] ^ (y >> 1) ^ ((0u - (y & 1u)) & kMatrix);
    }
    const uint32_t y = (key[N - 1] & kUpper) | (key[0] & kLower);
    key[N - 1] = key[M - 1] ^ (y >> 1) ^ ((0u - (y & 1u)) & kMatrix);
  }
  for (int i = 0; i < N; ++i) {
    uint32_t y = key[i];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    out[i] = y;
  }
}

struct Mt {
  uint32_t key[kMT];   // raw state, numpy layout
  uint32_t out[kMT];   // tempered outputs of the current block (filled by regen, consumed by u32)
  int pos;
  int has_gauss;
  double gauss;

  void seed(uint32_t s) {
    for (int i = 0; i < kMT; ++i) {
      key[i] = s;
      s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i + 1u;
    }
    pos = kMT;
    has_gauss = 0;
    gauss = 0.0;
  }
  // Adopt a numpy state whose block is partly consumed: temper the current block so u32() can continue at `pos`.
  void adopt(const uint32_t* k, int p, int hg, double g) {
    memcpy(key, k, sizeof(key));
    pos = p;
    has_gauss = hg;
    gauss = g;
    temper_block();
  }
  void temper_block() { mt_block(key, out, 0); }
  void regen() {
    mt_block(key, out, 1);
    pos = 0;
  }
  inline uint32_t u32() {
    if (__builtin_expect(pos == kMT, 0)) regen();
    return out[pos++];
  }
  inline double dbl() {
    const int32_t a = (int32_t)(u32() >> 5), b = (int32_t)(u32() >> 6);
    return (a * 67108864.0 + b) / 9007199254740992.0;
  }
  inline double uniform(double lo, double hi) { return lo + (hi - lo) * dbl(); }
  inline uint32_t interval(uint32_t max) {  // numpy random_interval, max <= 0xffffffff
    if (max == 0) return 0;
    uint32_t mask = max;
    mask |= mask >> 1;
    mask |= mask >> 2;
    mask |= mask >> 4;
    mask |= mask >> 8;
    mask |= mask >> 16;
    uint32_t v;
    while ((v = (u32() & mask)) > max) {
    }
    return v;
  }
  double gauss_legacy() {
    if (has_gauss) {
      const double t = gauss;
      has_gauss = 0;
      gauss = 0.0;
      return t;
    }
    double f, x1, x2, r2;
    do {
      x1 = 2.0 * dbl() - 1.0;
      x2 = 2.0 * dbl() - 1.0;
      r2 = x1 * x1 + x2 * x2;
    } while (r2 >= 1.0 || r2 == 0.0);
    f = sqrt(-2.0 * log(r2) / r2);
    gauss = f * x1;
    has_gauss = 1;
    return f * x2;
  }
};

// ---- filter design ------------------------------------------------------------------------------------------------
// |H| peak on scipy.signal.freqz's default grid (512 points on [0, pi)): the first half of a 1024-point DFT of the taps.
// Radix-2 decimation in time on split real / imaginary arrays (plain double arithmetic: std::complex products without
// -ffast-math go through __muldc3 and cost several times more). Direct evaluation for cascades longer than 1024 taps.
struct Twiddles {
  double c[512], s[512];
  Twiddles() {
    for (int k = 0; k < 512; ++k) {
      c[k] = cos(-2.0 * M_PI * k / 1024.0);
      s[k] = sin(-2.0 * M_PI * k / 1024.0);
    }
  }
};

double peak_response(const std::vector<double>& b) {
  const int K = (int)b.size();
  double best = 0.0;
  if (K <= 1024) {
    static const Twiddles tw;  // thread-safe one-time initialisation
    constexpr int n = 1024;
    double re[n], im[n];
    for (int i = 0, j = 0; i < n; ++i) {  // bit-reversed load of the real input
      re[j] = i < K ? b[i] : 0.0;
      im[j] = 0.0;
      int bit = n >> 1;
      for (; j & bit; bit >>= 1) j ^= bit;
      j ^= bit;
    }
    for (int len = 2; len <= n; len <<= 1) {
      const int half = len >> 1, step = n / len;
      for (int i = 0; i < n; i += len)
        for (int k = 0; k < half; ++k) {
          const double wr = tw.c[k * step], wi = tw.s[k * step];
          const double xr = re[i + k + half], xi = im[i + k + half];
          const double tr = xr * wr - xi * wi, ti = xr * wi + xi * wr;
          const double ur = re[i + k], ui = im[i + k];
          re[i + k] = ur + tr;
          im[i + k] = ui + ti;
          re[i + k + half] = ur - tr;
          im[i + k + half] = ui - ti;
        }
    }
    // max |H|: hypot is the expensive part, so squared magnitudes pick the candidates first. A bin whose squared magnitude is
    // more than 1e-12 (relative) below the largest cannot hold the maximum of hypot (whose error is ~1e-16), so the result
    // is the same value the full scan returns.
    double m2[512], m2max = 0.0;
    bool finite = true;
    for (int i = 0; i < 512; ++i) {
      m2[i] = re[i] * re[i] + im[i] * im[i];
      finite &= (m2[i] <= 1.0e300);  // false for inf / NaN too
      m2max = fmax(m2max, m2[i]);
    }
    if (finite && m2max >= 1.0e-280) {
      const double cut = m2max * (1.0 - 1.0e-12);
      for (int i = 0; i < 512; ++i)
        if (m2[i] >= cut) best = fmax(best, hypot(re[i], im[i]));
    } else {  // squares over- or underflow: plain scan
      for (int i = 0; i < 512; ++i) best = fmax(best, hypot(re[i], im[i]));
    }
  } else {
    for (int i = 0; i < 512; ++i) {
      const double w = M_PI * i / 512.0;
      double sr = 0.0, si = 0.0;
      for (int k = 0; k < K; ++k) {
        sr += b[k] * cos(w * k);
        si -= b[k] * sin(w * k);
      }
      best = fmax(best, hypot(sr, si));
    }
  }
  return best;
}

inline double sinc_pi(double x) {  // numpy.sinc
  if (x == 0.0) return 1.0;
  const double y = M_PI * x;
  return sin(y) / y;
}

// Values that depend on the stage length only, computed once per length and thread: the Hamming window
// 0.54 - 0.46 cos(2 pi i / (n - 1)) and, for odd n, numpy.sinc at the integer offsets m = i - (n - 1) / 2.
struct FirwinCache {
  static constexpr int kMaxN = 256;
  std::vector<double> win[kMaxN + 1];
  double sinc_int[kMaxN + 1];  // sinc_pi(m), m = 0 .. kMaxN
  FirwinCache() {
    for (int m = 0; m <= kMaxN; ++m) sinc_int[m] = sinc_pi(1.0 * m);
  }
  const std::vector<double>& window(int n) {
    std::vector<double>& w = win[n];
    if (w.empty()) {
      w.resize(n);
      for (int i = 0; i < n; ++i) w[i] = (n == 1) ? 1.0 : 0.54 - 0.46 * cos(2.0 * M_PI * i / (n - 1));
    }
    return w;
  }
};

// scipy.signal.firwin(n, [f1, f2], window='hamming', fs=fs) with the default pass_zero=True: a band-stop, DC gain 1.
// Every value is produced by the same operations in the same order as the plain loop over i; the sinc terms are even in
// m (glibc's sin is odd, the products and the quotient only change sign), so for odd n the upper half is copied from the lower.
void firwin_bandstop(int n, double f1, double f2, double fs, std::vector<double>& h) {
  const double nyq = fs / 2.0, c1 = f1 / nyq, c2 = f2 / nyq, alpha = 0.5 * (n - 1);
  h.resize(n);
  double dc = 0.0;
  if ((n & 1) && n <= FirwinCache::kMaxN) {
    thread_local FirwinCache cache;
    const std::vector<double>& win = cache.window(n);
    const int half = (n - 1) / 2;  // = alpha
    for (int i = 0; i <= half; ++i) {
      const double m = i - alpha;  // integer, <= 0
      double v = c1 * sinc_pi(c1 * m);
      v -= 0.0 * 1.0;              // 0.0 * sinc_pi(0.0 * m): sinc_pi(+-0) = 1
      v += 1.0 * cache.sinc_int[half - i];
      v -= c2 * sinc_pi(c2 * m);
      h[i] = v;
      h[n - 1 - i] = v;
    }
    for (int i = 0; i < n; ++i) {
      h[i] = h[i] * win[i];
      dc += h[i];  // scale_frequency = 0 -> cos term is 1
    }
  } else {
    for (int i = 0; i < n; ++i) {
      const double m = i - alpha;
      // bands [0, c1] and [c2, 1]
      double v = c1 * sinc_pi(c1 * m);  // same association as scipy's loop over the bands
      v -= 0.0 * sinc_pi(0.0 * m);
      v += 1.0 * sinc_pi(1.0 * m);
      v -= c2 * sinc_pi(c2 * m);
      const double win = (n == 1) ? 1.0 : 0.54 - 0.46 * cos(2.0 * M_PI * i / (n - 1));
      h[i] = v * win;
      dc += h[i];  // scale_frequency = 0 -> cos term is 1
    }
  }
  for (int i = 0; i < n; ++i) h[i] /= dc;
}

struct Args {  // mirrors rb_args
  int32_t N_f, nBands;
  double minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, minBiasLinNonLin, maxBiasLinNonLin, P, g_sd, SNRmin, SNRmax, fs;
};

// genNotchCoeffs (RawBoost.py:28-48): 3*nBands + 1 uniforms.
void gen_notch(Mt& rng, const Args& a, double minG, double maxG, std::vector<double>& taps, std::vector<double>& stage,
               std::vector<double>& tmp) {
  taps.assign(1, 1.0);
  for (int band = 0; band < a.nBands; ++band) {
    const double fc = rng.uniform(a.minF, a.maxF);
    const double bw = rng.uniform(a.minBW, a.maxBW);
    int c = (int)rng.uniform(a.minCoeff, a.maxCoeff);  // int() truncation
    if (c % 2 == 0) c += 1;
    double f1 = fc - bw / 2, f2 = fc + bw / 2;
    if (f1 <= 0) f1 = 1.0 / 1000;
    if (f2 >= a.fs / 2) f2 = a.fs / 2 - 1.0 / 1000;
    firwin_bandstop(c, f1, f2, a.fs, stage);
    tmp.assign(taps.size() + stage.size() - 1, 0.0);
    for (size_t i = 0; i < stage.size(); ++i)
      for (size_t j = 0; j < taps.size(); ++j) tmp[i + j] += stage[i] * taps[j];
    taps.swap(tmp);
  }
  const double G = rng.uniform(minG, maxG);
  const double scale = pow(10.0, G / 20.0) / peak_response(taps);
  for (double& t : taps) t *= scale;
}

struct UttDraw {
  std::vector<float> lnl_taps;
  std::vector<int32_t> lnl_k;
  std::vector<int32_t> isd_idx;
  std::vector<double> isd_fr;
  std::vector<float> ssi_taps;
  float snr = 0.f;
};

struct Scratch {
  std::vector<double> taps, stage, tmp;
  std::vector<uint32_t> perm;
  std::vector<uint16_t> perm16;
  std::vector<uint32_t> targets;
  std::vector<uint16_t> targets16;
};

// numpy's legacy shuffle of arange(n): for i = n-1 .. 1: j = random_interval(i); swap(x[i], x[j]), in two passes.
// Pass 1 settles the swap targets: the mask only changes when i crosses a power of two, and inside such a region the
// rejection loop is branch-free (every masked word is stored, the cursor only advances when it is accepted), so the ~28 % of
// rejected words cost no mispredicted branches. Pass 2 applies the swaps with the targets known ahead, which lets it
// prefetch the (cache-missing, 129 KB at 64600 samples) target slots a few steps in advance.
template <typename T>
void shuffle_legacy(Mt& rng, T* x, int n, std::vector<T>& js) {  // targets are < n, so they fit the element type
  if (n < 2) return;
  js.resize((size_t)n + 1);
  T* jp = js.data();
  int k = 0;  // steps settled so far; step k has i = n-1-k
  int i = n - 1;
  while (i >= 1) {
    uint32_t mask = (uint32_t)i;
    mask |= mask >> 1;
    mask |= mask >> 2;
    mask |= mask >> 4;
    mask |= mask >> 8;
    mask |= mask >> 16;
    const int lo = (int)(mask >> 1) + 1;  // smallest i with this mask
    while (i >= lo) {
      const uint32_t v = rng.u32() & mask;
      jp[k] = (T)v;
      const int ok = v <= (uint32_t)i;
      k += ok;
      i -= ok;
    }
  }
  constexpr int kAhead = 12;
  const int steps = n - 1;
  for (int s = 0; s < steps; ++s) {
    if (s + kAhead < steps) __builtin_prefetch(&x[jp[s + kAhead]], 1);
    const int ii = n - 1 - s;
    const uint32_t j = jp[s];
    const T t = x[j];
    x[j] = x[ii];
    x[ii] = t;
  }
}

// All draws of process_Rawboost_feature for one utterance, in the dispatcher's order: LnL, ISD, SSI.
void draw_utt(Mt& rng, const Args& a, int algo, int length, UttDraw& out, float* noise_row, Scratch& sc) {
  const bool lnl = rb::algo_uses_lnl(algo), isd = rb::algo_uses_isd(algo), ssi = rb::algo_uses_ssi(algo);
  out.lnl_taps.clear();
  out.lnl_k.clear();
  out.isd_idx.clear();
  out.isd_fr.clear();
  out.ssi_taps.clear();
  if (lnl) {
    double minG = a.minG, maxG = a.maxG;
    for (int f = 0; f < a.N_f; ++f) {
      if (f == 1) {
        minG -= a.minBiasLinNonLin;
        maxG -= a.maxBiasLinNonLin;
      }
      gen_notch(rng, a, minG, maxG, sc.taps, sc.stage, sc.tmp);
      out.lnl_k.push_back((int32_t)sc.taps.size());
      for (double t : sc.taps) out.lnl_taps.push_back((float)t);
    }
  }
  if (isd) {
    const double beta = rng.uniform(0.0, a.P);
    // numpy slices the permutation with [:n], which clips at the array's length (reachable with P > 100)
    const int n = std::min(std::max((int)(length * (beta / 100)), 0), length);
    out.isd_idx.resize(n);
    out.isd_fr.resize(n);
    if (length <= 65536) {  // 16-bit permutation array: half the cache footprint of the Fisher-Yates walk
      sc.perm16.resize(length);
      uint16_t* pm = sc.perm16.data();
      for (int i = 0; i < length; ++i) pm[i] = (uint16_t)i;
      shuffle_legacy(rng, pm, length, sc.targets16);
      for (int i = 0; i < n; ++i) out.isd_idx[i] = (int32_t)pm[i];
    } else {
      sc.perm.resize(length);
      uint32_t* pm = sc.perm.data();
      for (int i = 0; i < length; ++i) pm[i] = (uint32_t)i;
      shuffle_legacy(rng, pm, length, sc.targets);
      for (int i = 0; i < n; ++i) out.isd_idx[i] = (int32_t)pm[i];
    }
    for (int i = 0; i < n; ++i) out.isd_fr[i] = 2 * rng.dbl() - 1;
    for (int i = 0; i < n; ++i) out.isd_fr[i] *= 2 * rng.dbl() - 1;
  }
  if (ssi) {
    for (int i = 0; i < length; ++i) noise_row[i] = (float)(0.0 + 1.0 * rng.gauss_legacy());
    gen_notch(rng, a, a.minG, a.maxG, sc.taps, sc.stage, sc.tmp);
    for (double t : sc.taps) out.ssi_taps.push_back((float)t);
    out.snr = (float)rng.uniform(a.SNRmin, a.SNRmax);
  }
}

template <typename T>
struct PinnedBuf {
  T* p = nullptr;
  size_t cap = 0;
  bool pinned = false;
  int ensure(size_t n, bool want_pinned) {
    if (n <= cap) return 0;
    release();
    const size_t bytes = (n + n / 8 + 64) * sizeof(T);
    if (want_pinned && cudaMallocHost((void**)&p, bytes) == cudaSuccess) {
      pinned = true;
    } else {
      (void)cudaGetLastError();
      p = (T*)malloc(bytes);
      pinned = false;
      if (!p) return -1;
    }
    cap = bytes / sizeof(T);
    return 0;
  }
  void release() {
    if (!p) return;
    if (pinned) cudaFreeHost(p);
    else free(p);
    p = nullptr;
    cap = 0;
  }
};

}  // namespace

struct rb_planner {
  int threads;
  bool pinned;
  std::vector<UttDraw> draws;
  PinnedBuf<float> lnl_taps, ssi_taps, ssi_noise, ssi_snr;
  PinnedBuf<int32_t> lnl_off, isd_off, isd_idx, ssi_off;
  PinnedBuf<double> isd_fr;
};

extern "C" {

int rb_planner_create(rb_planner** out, int threads, int pinned) {
  if (!out) return RB_ERR_INVALID_ARG;
  rb_planner* p = new (std::nothrow) rb_planner();
  if (!p) return RB_ERR_INVALID_ARG;
  p->threads = threads > 0 ? threads : (int)std::max(1u, std::thread::hardware_concurrency());
  p->pinned = pinned != 0;
  *out = p;
  return RB_OK;
}

int rb_planner_destroy(rb_planner* p) {
  if (!p) return RB_OK;
  p->lnl_taps.release();
  p->ssi_taps.release();
  p->ssi_noise.release();
  p->ssi_snr.release();
  p->lnl_off.release();
  p->isd_off.release();
  p->isd_idx.release();
  p->ssi_off.release();
  p->isd_fr.release();
  delete p;
  return RB_OK;
}

// Draw the plans of B utterances. seeds != NULL: np.random.seed(seeds[u]) before utterance u (utterances independent,
// drawn in parallel). seeds == NULL: the utterances consume ONE stream, `state` (numpy get_state layout), sequentially,
// and `state` is advanced -- what a loader calling the reference once per view does. `view` receives host pointers into
// the planner's buffers, valid until the next draw on this planner.
int rb_planner_draw(rb_planner* p, const rb_args* args, int algo, int B, int ld, const int32_t* len, const uint32_t* seeds,
                    rb_rng_state* state, rb_plan* view) {
  if (!p || !args || !view || B < 0 || ld < 0 || (B > 0 && !len)) return RB_ERR_INVALID_ARG;
  if (!seeds && !state) return RB_ERR_INVALID_ARG;
  {  // what the reference's own calls would reject or what has no numpy equivalent here: refuse instead of throwing
    if (rb::algo_uses_lnl(algo) || rb::algo_uses_ssi(algo)) {
      const double cmin = std::min(args->minCoeff, args->maxCoeff), cmax = std::max(args->minCoeff, args->maxCoeff);
      if (args->nBands < 1 || args->nBands > 1000 || !(cmin >= 1.0) || !(cmax <= 1e6) || !(args->fs > 0.0)) return RB_ERR_UNSUPPORTED;
      if (rb::algo_uses_lnl(algo) && (args->N_f < 1 || args->N_f > 1000)) return RB_ERR_UNSUPPORTED;
    }
    if (rb::algo_uses_isd(algo) && !(args->P >= 0.0)) return RB_ERR_UNSUPPORTED;  // a negative count would mean numpy's "all but the last |n|"
  }
  try {
  Args a;
  a.N_f = args->N_f;
  a.nBands = args->nBands;
  a.minF = args->minF;
  a.maxF = args->maxF;
  a.minBW = args->minBW;
  a.maxBW = args->maxBW;
  a.minCoeff = args->minCoeff;
  a.maxCoeff = args->maxCoeff;
  a.minG = args->minG;
  a.maxG = args->maxG;
  a.minBiasLinNonLin = args->minBiasLinNonLin;
  a.maxBiasLinNonLin = args->maxBiasLinNonLin;
  a.P = args->P;
  a.g_sd = args->g_sd;
  a.SNRmin = args->SNRmin;
  a.SNRmax = args->SNRmax;
  a.fs = args->fs;
  const bool lnl = rb::algo_uses_lnl(algo), isd = rb::algo_uses_isd(algo), ssi = rb::algo_uses_ssi(algo);
  memset(view, 0, sizeof(*view));
  view->n_f = lnl ? a.N_f : 0;
  view->g_sd = (float)a.g_sd;
  if (B == 0) return RB_OK;
  for (int u = 0; u < B; ++u)
    if (len[u] < 0 || len[u] > ld) return RB_ERR_INVALID_ARG;
  p->draws.resize(B);
  if (ssi) {
    if (p->ssi_noise.ensure((size_t)B * ld, p->pinned)) return RB_ERR_INVALID_ARG;
    memset(p->ssi_noise.p, 0, (size_t)B * ld * sizeof(float));
  }
  if (seeds) {
    std::atomic<int> next{0};
    std::atomic<int> failed{0};
    auto work = [&]() {
      try {
        Mt rng;
        Scratch sc;
        for (;;) {
          const int u = next.fetch_add(1);
          if (u >= B) break;
          rng.seed(seeds[u]);
          draw_utt(rng, a, algo, len[u], p->draws[u], ssi ? p->ssi_noise.p + (size_t)u * ld : nullptr, sc);
        }
      } catch (...) {  // an exception escaping a std::thread would terminate the process
        failed.store(1);
        next.store(B);
      }
    };
    const int nt = std::max(1, std::min(p->threads, B));
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    if (failed.load()) return RB_ERR_INVALID_ARG;
  } else {
    Mt rng;
    rng.adopt(state->key, state->pos, state->has_gauss, state->cached_gaussian);
    Scratch sc;
    for (int u = 0; u < B; ++u) draw_utt(rng, a, algo, len[u], p->draws[u], ssi ? p->ssi_noise.p + (size_t)u * ld : nullptr, sc);
    memcpy(state->key, rng.key, sizeof(rng.key));
    state->pos = rng.pos;
    state->has_gauss = rng.has_gauss;
    state->cached_gaussian = rng.gauss;
  }
  // ---- pack into CSR ------------------------------------------------------------------------------------------------
  if (lnl) {
    size_t total = 0;
    for (int u = 0; u < B; ++u) total += p->draws[u].lnl_taps.size();
    if (p->lnl_taps.ensure(total, p->pinned) || p->lnl_off.ensure((size_t)B * a.N_f + 1, p->pinned)) return RB_ERR_INVALID_ARG;
    size_t off = 0;
    p->lnl_off.p[0] = 0;
    for (int u = 0; u < B; ++u) {
      const UttDraw& d = p->draws[u];
      memcpy(p->lnl_taps.p + off, d.lnl_taps.data(), d.lnl_taps.size() * sizeof(float));
      size_t o = off;
      for (int f = 0; f < a.N_f; ++f) {
        o += d.lnl_k[f];
        p->lnl_off.p[(size_t)u * a.N_f + f + 1] = (int32_t)o;
      }
      off = o;
    }
    view->lnl_taps = p->lnl_taps.p;
    view->lnl_tap_off = p->lnl_off.p;
  }
  if (isd) {
    size_t total = 0;
    for (int u = 0; u < B; ++u) total += p->draws[u].isd_idx.size();
    if (p->isd_idx.ensure(total, p->pinned) || p->isd_fr.ensure(total, p->pinned) || p->isd_off.ensure((size_t)B + 1, p->pinned))
      return RB_ERR_INVALID_ARG;
    size_t off = 0;
    p->isd_off.p[0] = 0;
    for (int u = 0; u < B; ++u) {
      const UttDraw& d = p->draws[u];
      memcpy(p->isd_idx.p + off, d.isd_idx.data(), d.isd_idx.size() * sizeof(int32_t));
      memcpy(p->isd_fr.p + off, d.isd_fr.data(), d.isd_fr.size() * sizeof(double));
      off += d.isd_idx.size();
      p->isd_off.p[u + 1] = (int32_t)off;
    }
    view->isd_off = p->isd_off.p;
    view->isd_idx = p->isd_idx.p;
    view->isd_fr = p->isd_fr.p;
  }
  if (ssi) {
    size_t total = 0;
    for (int u = 0; u < B; ++u) total += p->draws[u].ssi_taps.size();
    if (p->ssi_taps.ensure(total, p->pinned) || p->ssi_off.ensure((size_t)B + 1, p->pinned) || p->ssi_snr.ensure((size_t)B, p->pinned))
      return RB_ERR_INVALID_ARG;
    size_t off = 0;
    p->ssi_off.p[0] = 0;
    for (int u = 0; u < B; ++u) {
      const UttDraw& d = p->draws[u];
      memcpy(p->ssi_taps.p + off, d.ssi_taps.data(), d.ssi_taps.size() * sizeof(float));
      off += d.ssi_taps.size();
      p->ssi_off.p[u + 1] = (int32_t)off;
      p->ssi_snr.p[u] = d.snr;
    }
    view->ssi_noise = p->ssi_noise.p;
    view->ssi_taps = p->ssi_taps.p;
    view->ssi_tap_off = p->ssi_off.p;
    view->ssi_snr_db = p->ssi_snr.p;
  }
  return RB_OK;
  } catch (...) {  // std::bad_alloc / std::length_error from the scratch vectors: no C++ exception crosses the C ABI
    return RB_ERR_INVALID_ARG;
  }
}

}  // extern "C"
