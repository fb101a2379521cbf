// rb_reverb.cu -- the reverb view (SURVEY.md 8f-4) as a uniformly partitioned FFT overlap-save convolution:
//   y_u = normWav(np.convolve(x_u, h_u), 1)        (/root/reference/datautils/audio_augmentor/reverb.py:39-42)
//
// Sizes: real transforms of kN = 16384 points, computed as complex FFTs of kM = 8192 points in shared memory (68 KB of padded
// float2 per CTA) plus the real split (two real samples per complex point). The impulse response is cut into partitions of
// kP = 8192 taps, so any length works with the one transform size; a CTA produces one output block of kP samples with one
// forward FFT per partition and one inverse FFT.
//
//   reverb_twiddle_kernel        W_M^m and W_N^k, computed in double and rounded once, into the workspace
//   reverb_rir_spectrum_kernel   one CTA per (row, partition p): H_p = RFFT(h[p kP, p kP + kP) zero-padded to kN) / kM
//   reverb_ols_kernel            one CTA per (row, output block): sum_p RFFT(input window of the block, p) . H_p, one inverse
//                                real FFT, whose last kP points are the block (overlap-save)
// followed by the existing normWav stream (launch_norm_stream, always = 1) in place over out_len. DESIGN.md 4.5 has the
// accuracy and the measured comparison with the direct-form FIR path.
//
// The FFT is a radix-8 / radix-2 Stockham pass sequence (E. Bainville's formulation): each pass reads R points of stride
// kM / R, twiddles, runs an R-point DFT in registers and writes them back at stride Ns; with all loads in registers before
// the stores, one buffer serves both sides of a pass. Results come out in natural order.
#include <algorithm>

#include "rb_common.cuh"
#include "rb_dense.cuh"

namespace rb {
namespace {

constexpr int kM = 8192;          // complex FFT points
constexpr int kN = 2 * kM;        // real points per transform (packed two per complex point)
constexpr int kP = kN / 2;        // taps per partition = samples per output block
constexpr int kRT = 1024;         // threads per CTA
constexpr int kPer = kM / kRT;    // points per thread in the element-wise steps (8)
static_assert(kM % kRT == 0 && (kM & (kM - 1)) == 0, "power-of-two transform");
// Shared-memory index of point i: one float2 of padding after every 16. Without it, the stores of the radix-8 pass at Ns = 2
// land 16 float2 apart (a 16-way bank conflict) and those of the radix-2 pass 2 apart.
__device__ __forceinline__ int sp(int i) { return i + (i >> 4); }
constexpr size_t kSmem = (size_t)(kM + kM / 16) * sizeof(float2);

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// a * W_M^idx; the eighth-turn twiddles of the register DFTs are exact constants (0.70710677f is sqrt(1/2) rounded to float),
// so unrolled code multiplies by immediates instead of loading them
__device__ __forceinline__ float2 twiddle_mul(float2 a, int idx, const float2* __restrict__ tw) {
  constexpr float c = 0.70710677f;
  if (idx == kM / 4) return make_float2(a.y, -a.x);                                 // -i
  if (idx == kM / 8) return make_float2(c * (a.x + a.y), c * (a.y - a.x));          // (1 - i) / sqrt 2
  if (idx == 3 * kM / 8) return make_float2(c * (a.y - a.x), -c * (a.x + a.y));     // (-1 - i) / sqrt 2
  return cmul(a, __ldg(tw + idx));
}

// R-point DFT in registers (radix-2 decimation in frequency, then the bit-reversal permutation). tw is the kM-point table.
template <int R>
__device__ __forceinline__ void dft_regs(float2 (&v)[R], const float2* __restrict__ tw) {
#pragma unroll
  for (int h = R / 2; h >= 1; h >>= 1) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      if (i & h) continue;
      const int m = i & (h - 1);
      const float2 a = v[i], b = v[i + h];
      v[i] = cadd(a, b);
      v[i + h] = m ? twiddle_mul(csub(a, b), m * (kM / (2 * h)), tw) : csub(a, b);
    }
  }
  float2 t[R];
#pragma unroll
  for (int i = 0; i < R; ++i) t[i] = v[i];
#pragma unroll
  for (int k = 0; k < R; ++k) {
    int r = 0;
#pragma unroll
    for (int b = 1, c = R / 2; b < R; b <<= 1, c >>= 1)
      if (k & b) r |= c;
    v[k] = t[r];
  }
}

// One Stockham pass of radix R over the kM points in s; Ns = product of the radices of the earlier passes.
template <int R>
__device__ __forceinline__ void fft_pass(float2* s, int Ns, const float2* __restrict__ tw) {
  constexpr int kItems = kM / (R * kRT);
  const int tid = threadIdx.x;
  float2 v[kItems][R];
#pragma unroll
  for (int it = 0; it < kItems; ++it) {
    const int j = tid + it * kRT;
    const int k = j & (Ns - 1);
#pragma unroll
    for (int r = 0; r < R; ++r) v[it][r] = s[sp(j + r * (kM / R))];
    if (Ns > 1) {
      const int step = k * (kM / (Ns * R));  // exp(-2 pi i k r / (Ns R)) = W_M^(k r M / (Ns R))
#pragma unroll
      for (int r = 1; r < R; ++r) v[it][r] = cmul(v[it][r], __ldg(tw + r * step));
    }
    dft_regs<R>(v[it], tw);
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < kItems; ++it) {
    const int j = tid + it * kRT;
    const int k = j & (Ns - 1);
    const int o = (j - k) * R + k;
#pragma unroll
    for (int r = 0; r < R; ++r) s[sp(o + r * Ns)] = v[it][r];
  }
  __syncthreads();
}

// Radix-2 butterfly of the first pass (Ns = 1), for callers that fold it into the fill of s: with z the natural-order input,
// points 2m and 2m + 1 of the pass output are z[m] + z[m + kM/2] and z[m] - z[m + kM/2].
__device__ __forceinline__ void store_radix2(float2* s, int m, float2 a, float2 b) {
  s[sp(2 * m)] = cadd(a, b);
  s[sp(2 * m + 1)] = csub(a, b);
}

// The remaining passes of the forward kM-point FFT of s, after the radix-2 pass (natural order out). Callers synchronise
// before it.
__device__ __forceinline__ void fft_after_radix2_but_last(float2* s, const float2* __restrict__ tw) {
  static_assert(kM == 2 * 8 * 8 * 8 * 8, "pass sequence");
  fft_pass<8>(s, 2, tw);
  fft_pass<8>(s, 16, tw);
  fft_pass<8>(s, 128, tw);
}
__device__ __forceinline__ void fft_after_radix2(float2* s, const float2* __restrict__ tw) {
  fft_after_radix2_but_last(s, tw);
  fft_pass<8>(s, kM / 8, tw);
}

// The last radix-8 pass (Ns = kM / 8) without its store: thread t ends up holding points t + r kM/8 of the transform in v[r].
__device__ __forceinline__ void fft_last_pass_regs(const float2* s, const float2* __restrict__ tw, float2 (&v)[8]) {
  static_assert(kM / 8 == kRT, "one radix-8 item per thread");
  const int j = threadIdx.x;  // k = j, step = k * kM / (Ns * 8) = j
#pragma unroll
  for (int r = 0; r < 8; ++r) v[r] = s[sp(j + r * (kM / 8))];
#pragma unroll
  for (int r = 1; r < 8; ++r) v[r] = cmul(v[r], __ldg(tw + r * j));
  dft_regs<8>(v, tw);
}

// Output length of row u, or -1 for a row that is not computed (see rawboost_b200.h); npart = partitions the workspace holds.
__device__ __forceinline__ int row_out_len(const int32_t* len, const int32_t* off, int u, int ld, int ld_out, int npart) {
  const int K = off[u + 1] - off[u], L = len[u];
  if (K < 1 || L < 0 || L > ld) return -1;
  if (L == 0) return 0;
  const long long n = (long long)L + K - 1;
  if (n > ld_out || (long long)K > (long long)npart * kP) return -1;
  return (int)n;
}

// tw[m] = W_M^m (the complex passes), tw[kM + k] = W_N^k (the real split); computed in double, rounded once
__global__ void __launch_bounds__(256)
reverb_twiddle_kernel(float2* __restrict__ tw) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= 2 * kM) return;
  double sn, cs;
  sincospi(m < kM ? 2.0 * m / kM : 2.0 * (m - kM) / kN, &sn, &cs);
  tw[m] = make_float2((float)cs, (float)-sn);
}

// Real split. A real sequence v of kN points packed as z[m] = v[2m] + i v[2m+1] has Z = FFT_M(z); its real transform is
// X[k] = E[k] + W_N^k O[k] with E = (Z[k] + conj Z[M-k]) / 2, O = (Z[k] - conj Z[M-k]) / 2i, and X[M-k] = conj(E[k] - W_N^k O[k]).
// For k = 0 (Z[M] = Z[0]) this gives the two real bins X[0] and X[M].
__device__ __forceinline__ void split_forward(float2 zk, float2 zm, float2 w, float2& xk, float2& xm) {
  const float2 e = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
  const float2 o = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
  const float2 wo = cmul(w, o);
  xk = make_float2(e.x + wo.x, e.y + wo.y);
  xm = make_float2(e.x - wo.x, wo.y - e.y);
}
// The inverse: from Y[k], Y[M-k] of a real kN-point sequence, Z'[k] and Z'[M-k] of its packed form (z' = IFFT_M(Z')), with
// E = (Y[k] + conj Y[M-k]) / 2, O = conj(W_N^k) (Y[k] - conj Y[M-k]) / 2, Z'[k] = E + i O, Z'[M-k] = conj E + i conj O.
__device__ __forceinline__ void split_inverse(float2 yk, float2 ym, float2 w, float2& zk, float2& zm) {
  const float2 e = make_float2(0.5f * (yk.x + ym.x), 0.5f * (yk.y - ym.y));
  const float2 o = cmul(make_float2(0.5f * (yk.x - ym.x), 0.5f * (yk.y + ym.y)), make_float2(w.x, -w.y));
  zk = make_float2(e.x - o.y, e.y + o.x);
  zm = make_float2(e.x + o.y, o.x - e.y);
}

struct ReverbArgs {
  const float* x;          // [B][ld] (rows of this launch)
  const int32_t* len;      // [B]
  const float* rir;        // CSR values (absolute offsets)
  const int32_t* off;      // [B + 1]
  float* y;                // [B][ld_out]
  int32_t* out_len;        // [B]
  const float2* tw;        // [2 kM]: W_M^m, then W_N^k
  float2* spec;            // [B][npart][kM]: bins 1 .. M-1 of H_p, bin 0 holds (H_p[0], H_p[M]) (both real)
  int ld, ld_out, npart;
};

// The split steps pair bin k with bin M - k: thread t owns k = t + q kRT for q < kSplit, k <= M/2 (k = M/2 only in thread 0).
constexpr int kSplit = kM / 2 / kRT + 1;

// grid (npart, rows): H_p = RFFT_N(h[p kP, p kP + kP) zero-padded) / kM (the inverse transform's factor); partition 0 also
// writes out_len[u].
__global__ void __launch_bounds__(kRT)
reverb_rir_spectrum_kernel(const ReverbArgs a) {
  extern __shared__ float2 s[];
  const int p = blockIdx.x, u = blockIdx.y, tid = threadIdx.x;
  const int n = row_out_len(a.len, a.off, u, a.ld, a.ld_out, a.npart);
  if (p == 0 && tid == 0) a.out_len[u] = n;
  const int K = a.off[u + 1] - a.off[u];
  if (n <= 0 || (long long)p * kP >= K) return;
  const float* h = a.rir + a.off[u] + (size_t)p * kP;
  const int kp = min(kP, K - p * kP);
  auto tap = [&](int i) { return i < kp ? __ldg(h + i) : 0.f; };
#pragma unroll
  for (int q = 0; q < kPer / 2; ++q) {
    const int m = tid + q * kRT;
    store_radix2(s, m, make_float2(tap(2 * m), tap(2 * m + 1)), make_float2(tap(2 * m + kM), tap(2 * m + kM + 1)));
  }
  __syncthreads();
  fft_after_radix2(s, a.tw);
  float2* dst = a.spec + ((size_t)u * a.npart + p) * kM;
  constexpr float kScale = 1.f / kM;  // exact: a power of two
#pragma unroll
  for (int q = 0; q < kSplit; ++q) {
    const int k = tid + q * kRT, km = (kM - k) & (kM - 1);
    if (k > kM / 2) break;
    float2 xk, xm;
    split_forward(s[sp(k)], s[sp(km)], __ldg(a.tw + kM + k), xk, xm);
    if (k == 0) {
      dst[0] = make_float2(xk.x * kScale, xm.x * kScale);
    } else {
      dst[k] = make_float2(xk.x * kScale, xk.y * kScale);
      dst[km] = make_float2(xm.x * kScale, xm.y * kScale);
    }
  }
}

// grid (blocks, rows): outputs [c kP, c kP + kP) of row u. For partition p the circular convolution of length kN runs over
// the input window x[c kP - p kP - kP + i], i < kN, whose last kP points are exact (overlap-save).
__global__ void __launch_bounds__(kRT)
reverb_ols_kernel(const ReverbArgs a) {
  extern __shared__ float2 s[];
  const int c = blockIdx.x, u = blockIdx.y, tid = threadIdx.x;
  const int n = row_out_len(a.len, a.off, u, a.ld, a.ld_out, a.npart);
  const long long o0 = (long long)c * kP;  // first output of the block
  if (n <= 0 || o0 >= n) return;
  const int L = a.len[u], K = a.off[u + 1] - a.off[u];
  const int nparts = (K + kP - 1) / kP;
  const float* xr = a.x + (size_t)u * a.ld;
  const float2* H = a.spec + (size_t)u * a.npart * kM;
  float2 acck[kSplit], accm[kSplit];  // Y[k] and Y[M-k] of the thread's bins
#pragma unroll
  for (int q = 0; q < kSplit; ++q) acck[q] = accm[q] = make_float2(0.f, 0.f);
  for (int p = 0; p < nparts; ++p) {
    const long long w0 = o0 - (long long)(p + 1) * kP;  // window start (even)
    if (w0 + 2 * kP <= 0 || w0 >= L) continue;          // the window lies outside the signal
    // packed point m of the window is (x[w0 + 2m], x[w0 + 2m + 1]); 8-byte aligned: rows are 16-byte aligned, w0 is even
    auto pair = [&](long long i0) {
      if (i0 >= 0 && i0 + 1 < L) return __ldg(reinterpret_cast<const float2*>(xr + i0));
      return make_float2((i0 >= 0 && i0 < L) ? __ldg(xr + i0) : 0.f, (i0 + 1 >= 0 && i0 + 1 < L) ? __ldg(xr + i0 + 1) : 0.f);
    };
#pragma unroll
    for (int q = 0; q < kPer / 2; ++q) {
      const int m = tid + q * kRT;
      store_radix2(s, m, pair(w0 + 2 * m), pair(w0 + 2 * m + kM));
    }
    __syncthreads();
    fft_after_radix2(s, a.tw);
    const float2* hp = H + (size_t)p * kM;
#pragma unroll
    for (int q = 0; q < kSplit; ++q) {
      const int k = tid + q * kRT, km = (kM - k) & (kM - 1);
      if (k > kM / 2) break;
      float2 xk, xm, hk, hm;
      split_forward(s[sp(k)], s[sp(km)], __ldg(a.tw + kM + k), xk, xm);
      if (k == 0) {
        const float2 h0 = __ldg(hp);
        hk = make_float2(h0.x, 0.f);
        hm = make_float2(h0.y, 0.f);
      } else {
        hk = __ldg(hp + k);
        hm = __ldg(hp + km);
      }
      acck[q].x = fmaf(xk.x, hk.x, fmaf(-xk.y, hk.y, acck[q].x));
      acck[q].y = fmaf(xk.x, hk.y, fmaf(xk.y, hk.x, acck[q].y));
      accm[q].x = fmaf(xm.x, hm.x, fmaf(-xm.y, hm.y, accm[q].x));
      accm[q].y = fmaf(xm.x, hm.y, fmaf(xm.y, hm.x, accm[q].y));
    }
    __syncthreads();  // s is refilled next
  }
  // inverse: packed spectrum, then IFFT as conj(FFT(conj(.))); the 1 / kM is already in H. Bins k and M-k are distinct
  // across threads (k = 0 and k = M/2 write one bin twice, with the same value).
#pragma unroll
  for (int q = 0; q < kSplit; ++q) {
    const int k = tid + q * kRT, km = (kM - k) & (kM - 1);
    if (k > kM / 2) break;
    float2 zk, zm;
    split_inverse(acck[q], accm[q], __ldg(a.tw + kM + k), zk, zm);
    s[sp(k)] = make_float2(zk.x, -zk.y);
    s[sp(km)] = make_float2(zm.x, -zm.y);
  }
  __syncthreads();
  fft_pass<2>(s, 1, a.tw);
  fft_after_radix2_but_last(s, a.tw);
  float2 v[8];
  fft_last_pass_regs(s, a.tw, v);
  // outputs 2i, 2i + 1 of the block are packed point kM/2 + i of the circular result (point kP + 2i of the real one); the thread
  // holds points tid + r kM/8, of which r >= 4 are in that half. Stored straight from registers, coalesced across the warp.
  float* yr = a.y + (size_t)u * a.ld_out;
#pragma unroll
  for (int r = 4; r < 8; ++r) {
    const long long e = o0 + 2 * (tid + (r - 4) * (kM / 8));
    if (e + 1 < n) *reinterpret_cast<float2*>(yr + e) = make_float2(v[r].x, -v[r].y);
    else if (e < n) yr[e] = v[r].x;
  }
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline size_t tw_bytes() { return align_up((size_t)2 * kM * sizeof(float2), 256); }
inline size_t state_bytes(int B) { return align_up((size_t)B * sizeof(uint2), 256); }
inline size_t spec_bytes(int B, int npart) { return (size_t)B * npart * kM * sizeof(float2); }

}  // namespace
}  // namespace rb

using namespace rb;

extern "C" size_t rb_reverb_workspace_bytes(int B, int max_taps) {
  if (B <= 0) return 0;
  const int npart = std::max(1, (int)(((long long)std::max(max_taps, 1) + kP - 1) / kP));
  return tw_bytes() + state_bytes(B) + spec_bytes(B, npart);
}

extern "C" int rb_reverb(const float* x, const int32_t* len, int B, int ld, const float* rir, const int32_t* rir_off, float* y,
                         int ld_out, int32_t* out_len, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 0 || ld < 0 || ld_out < 0) return RB_ERR_INVALID_ARG;
  if (B == 0) return RB_OK;
  if (!x || !len || !rir || !rir_off || !y || !out_len) return RB_ERR_INVALID_ARG;
  if (ld % 4 != 0 || ld_out % 4 != 0 || ((uintptr_t)x & 15u) || ((uintptr_t)y & 15u)) return RB_ERR_ALIGNMENT;
  if (x == y) return RB_ERR_INVALID_ARG;
  if (!workspace || ((uintptr_t)workspace & 255u)) return workspace ? RB_ERR_ALIGNMENT : RB_ERR_WORKSPACE;
  const size_t fixed = tw_bytes() + state_bytes(B);
  if (workspace_bytes < fixed + spec_bytes(B, 1)) return RB_ERR_WORKSPACE;
  // partitions per row the workspace holds (one spectrum CTA each); a valid row never has more taps than ld_out
  const long long fit = (long long)((workspace_bytes - fixed) / spec_bytes(B, 1));
  const int npart = (int)std::min<long long>(fit, std::max<long long>(1, ((long long)ld_out + kP - 1) / kP));
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  ReverbArgs a;
  a.tw = (const float2*)ws;
  void* state = ws + tw_bytes();
  a.spec = (float2*)(ws + fixed);
  a.ld = ld;
  a.ld_out = ld_out;
  a.npart = npart;
  // per call: the attribute belongs to the kernel in the current device's context
  RB_CUDA(cudaFuncSetAttribute(reverb_rir_spectrum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
  RB_CUDA(cudaFuncSetAttribute(reverb_ols_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
  reverb_twiddle_kernel<<<2 * kM / 256, 256, 0, st>>>((float2*)a.tw);
  RB_LAUNCH_CHECK();
  const int blocks = (int)(((long long)ld_out + kP - 1) / kP);
  for (int b0 = 0; b0 < B; b0 += 65535) {  // grid.y limit
    const int nb = std::min(65535, B - b0);
    ReverbArgs r = a;
    r.x = x + (size_t)b0 * ld;
    r.len = len + b0;
    r.rir = rir;
    r.off = rir_off + b0;
    r.y = y + (size_t)b0 * ld_out;
    r.out_len = out_len + b0;
    r.spec = a.spec + (size_t)b0 * npart * kM;
    reverb_rir_spectrum_kernel<<<dim3(npart, nb), kRT, kSmem, st>>>(r);
    RB_LAUNCH_CHECK();
    if (blocks > 0) {
      reverb_ols_kernel<<<dim3(blocks, nb), kRT, kSmem, st>>>(r);
      RB_LAUNCH_CHECK();
    }
  }
  // rows with out_len <= 0 are skipped by the normWav stream (no tile starts below the length)
  return launch_norm_stream(y, nullptr, out_len, B, ld_out, 1, nullptr, nullptr, nullptr, 0.f, y, state, st);
}
