// Per-utterance finalisers of the fused tails of the FIR-bank kernel (rb_fir_bank.cu; isd_value is shared with rb_dense.cu):
// reduce the per-tile statistics of one utterance and derive the scalars of the dense apply pass.
// One CTA of kThreads threads per call; every global read goes to L2 (__ldcg) because in the fused tail the data was
// written by other SMs a moment ago.
//
// Reference arithmetic (file:line under /root/reference/datautils/RawBoost.py): normWav 20-25, LnL tail 67-68, ISD 76-84,
// SSI tail 93-96.
#pragma once
#include "rb_common.cuh"

namespace rb {

// The impulsive-noise value at one position, with the reference's exact operation order and precisions
// (RawBoost.py:81-82 on float32 input): t = fl32(g_sd*x), r = fl64(t*f_r), y = fl32(fl64(x + r)).
__device__ __forceinline__ float isd_value(float v, float g_sd, double fr) {
  const float t = __fmul_rn(g_sd, v);
  const double r = __dmul_rn((double)t, fr);
  return (float)__dadd_rn((double)v, r);
}

// out = ((in - sub) / div1) / div2 with IEEE operations in the reference's order
__device__ __forceinline__ float affine_value(float e, const UttParams& p) {
  return __fdiv_rn(__fdiv_rn(__fsub_rn(e, p.sub), p.div1), p.div2);
}

// Impulses gathered per thread and round: all their index loads go out together, then all their sample loads, so an
// utterance's impulses cost a few L2 round trips instead of two dependent ones per impulse and thread.
constexpr int kIsdInFlight = 8;

// LnL / normWav / ISD scalars of one utterance: st = its [ntiles][kStatN] tile statistics (only the first `ntiles` are read),
// n = its length, row = the waveform the statistics were taken from. isd_beg < isd_end: impulses applied after the first
// normalisation; the new value isd_value((row[p] - sub) / div1) of impulse i < isd_beg + cap is left in vals[i - isd_beg]
// (shared memory, visible to the whole CTA on return) for the scatter. Returns the same value in every thread of the CTA.
__device__ __forceinline__ UttParams finalize_block(const float* __restrict__ st, int ntiles, int n, int center, int always,
                                                    const float* __restrict__ row, const int32_t* __restrict__ isd_idx,
                                                    const double* __restrict__ isd_fr, int isd_beg, int isd_end, bool with_isd,
                                                    float g_sd, float* __restrict__ vals, int cap) {
  __shared__ double red_sum[4];
  __shared__ float red_f[4][4];
  __shared__ float bc[4];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double sum = 0.0;
  float mn = INFINITY, mx = -INFINITY, mnu = INFINITY, mxu = -INFINITY;
  for (int t = tid; t < ntiles; t += kThreads) {
    sum += (double)__ldcg(st + t * kStatN + S_SUM);
    mn = fminf(mn, __ldcg(st + t * kStatN + S_MIN));
    mx = fmaxf(mx, __ldcg(st + t * kStatN + S_MAX));
    mnu = fminf(mnu, __ldcg(st + t * kStatN + S_MINU));
    mxu = fmaxf(mxu, __ldcg(st + t * kStatN + S_MAXU));
  }
  sum = warp_sum(sum);
  mn = warp_min(mn);
  mx = warp_max(mx);
  mnu = warp_min(mnu);
  mxu = warp_max(mxu);
  __syncthreads();  // the shared scratch may still be in use by a previous call
  if (lane == 0) {
    red_sum[warp] = sum;
    red_f[warp][0] = mn;
    red_f[warp][1] = mx;
    red_f[warp][2] = mnu;
    red_f[warp][3] = mxu;
  }
  __syncthreads();
  if (tid == 0) {
    const double s = (red_sum[0] + red_sum[1]) + (red_sum[2] + red_sum[3]);
    const float fmn = fminf(fminf(red_f[0][0], red_f[1][0]), fminf(red_f[2][0], red_f[3][0]));
    const float fmx = fmaxf(fmaxf(red_f[0][1], red_f[1][1]), fmaxf(red_f[2][1], red_f[3][1]));
    const float fmnu = fminf(fminf(red_f[0][2], red_f[1][2]), fminf(red_f[2][2], red_f[3][2]));
    const float fmxu = fmaxf(fmaxf(red_f[0][3], red_f[1][3]), fmaxf(red_f[2][3], red_f[3][3]));
    const float sub = (center && n > 0) ? (float)(s / (double)n) : 0.f;
    const float m1 = (n > 0) ? fmaxf(fabsf(fmx - sub), fabsf(fmn - sub)) : 0.f;
    const float div1 = (n > 0 && (always || m1 > 1.f)) ? m1 : 1.f;
    // peak of the untouched samples after the first normalisation (fp32 division is monotone, so the peak of
    // the quotients is the quotient of the peak)
    float mu = 0.f;
    if (fmnu <= fmxu) mu = fmaxf(fabsf(fmxu - sub), fabsf(fmnu - sub)) / div1;
    bc[0] = sub;
    bc[1] = div1;
    bc[2] = mu;
  }
  __syncthreads();
  const float sub = bc[0], div1 = bc[1];
  if (with_isd) {
    float mt = 0.f;  // fmaxf is order-free, so the grouping of the impulses does not change the peak
    for (int i0 = isd_beg + tid; i0 < isd_end; i0 += kIsdInFlight * kThreads) {
      int p[kIsdInFlight];
      double fr[kIsdInFlight];
      float e[kIsdInFlight];
#pragma unroll
      for (int k = 0; k < kIsdInFlight; ++k) {
        const int i = i0 + k * kThreads;
        p[k] = i < isd_end ? isd_idx[i] : -1;
      }
#pragma unroll
      for (int k = 0; k < kIsdInFlight; ++k) {
        const bool in = p[k] >= 0 && p[k] < n;
        e[k] = in ? __ldcg(row + p[k]) : 0.f;
        fr[k] = in ? isd_fr[i0 + k * kThreads] : 0.0;
      }
#pragma unroll
      for (int k = 0; k < kIsdInFlight; ++k) {
        if (p[k] >= 0 && p[k] < n) {
          const float v = isd_value((e[k] - sub) / div1, g_sd, fr[k]);
          mt = fmaxf(mt, fabsf(v));
          const int j = i0 + k * kThreads - isd_beg;
          if (j < cap) vals[j] = v;
        }
      }
    }
    mt = warp_max(mt);
    __syncthreads();
    if (lane == 0) red_f[warp][0] = mt;
    __syncthreads();
    if (tid == 0) {
      const float m2 = fmaxf(bc[2], fmaxf(fmaxf(red_f[0][0], red_f[1][0]), fmaxf(red_f[2][0], red_f[3][0])));
      bc[3] = (m2 > 1.f) ? m2 : 1.f;
    }
    __syncthreads();
  }
  UttParams p;
  p.sub = sub;
  p.div1 = div1;
  p.div2 = with_isd ? bc[3] : 1.f;
  p.scale = 0.f;
  return p;
}

// SSI gain ||x||_2 / (||coloured noise||_2 * 10^(snr/20))  (RawBoost.py:95). stats_x[S_SUMSQ-like slot sx_slot] holds the
// per-tile sum of squares of x, stats_n[S_SUMSQ] that of the coloured noise. Evaluated by the first warp; the value is
// returned in every thread of the CTA.
__device__ __forceinline__ float ssi_scale_block(const float* __restrict__ stats_x, int sx_slot, const float* __restrict__ stats_n,
                                                 int ntiles, float snr_db) {
  __shared__ float bcs;
  const int tid = threadIdx.x;
  if (tid < 32) {
    double sx = 0.0, sn = 0.0;
    for (int t = tid; t < ntiles; t += 32) {
      sx += (double)__ldcg(stats_x + t * kStatN + sx_slot);
      sn += (double)__ldcg(stats_n + t * kStatN + S_SUMSQ);
    }
    sx = warp_sum(sx);
    sn = warp_sum(sn);
    if (tid == 0) bcs = (float)(sqrt(sx) / (sqrt(sn) * pow(10.0, 0.05 * (double)snr_db)));
  }
  __syncthreads();
  return bcs;
}

}  // namespace rb
