// Phase vocoder over full STFT spectra (the time-stretch and pitch-shift attacks; aw_phase_vocoder).
//
// The classical algorithm of librosa.phase_vocoder, in float64, on spectra laid out frame-major,
// [clip][frame][AW_NBINS_FULL] complex64 (aw_stft_full's output).  For output frame t, with
// s = t * rate (what np.arange(0, T, rate) produces), i = floor(s), alpha = s - i, and D extended by
// two zero frames:
//   out_t = mag * (cos acc_t, sin acc_t),   mag = (1 - alpha) |D_i| + alpha |D_{i+1}|,   acc_0 = angle(D_0)
//   dphi  = angle(D_{i+1}) - angle(D_i) - phi_k,   phi_k = (pi / 2) k  (= hop 2 pi k / n_fft)
//   dphi -= 2 pi rint(dphi / 2 pi);   acc_{t+1} = acc_t + (phi_k + dphi)
// |.| and angle are hypot / atan2 in float64 of the float32 components; out_t is rounded to complex64.
//
// One thread per (clip, bin) walks the output frames in ascending order, so the float64 recurrence runs
// in exactly the restatement's order (every operation is an explicitly rounded intrinsic: no FMA
// contraction) and each warp's reads of D_i / D_{i+1} and writes of out_t are 256-byte rows.  The |D| and
// angle of a frame are computed once and carried while i stays or advances by one.  No atomics: a clip's
// result does not depend on the batch it is computed in.
#pragma once
#include "common.cuh"
#include "fft.cuh"

namespace aw {

__device__ __forceinline__ void pv_polar(const float2* __restrict__ d, int i, int T, double& mag, double& ang) {
  if (i >= T) {                       // the two zero frames appended to D
    mag = 0.0;
    ang = 0.0;
    return;
  }
  const float2 v = d[(long long)i * AW_NBINS_FULL];
  mag = hypot((double)v.x, (double)v.y);
  ang = atan2((double)v.y, (double)v.x);
}

__global__ void __launch_bounds__(128) k_phase_vocoder(const float2* __restrict__ spec, int n_clips, int T,
                                                       double rate, int T_out, float2* __restrict__ out) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)n_clips * AW_NBINS_FULL) return;
  const int clip = (int)(g / AW_NBINS_FULL);
  const int k = (int)(g - (long long)clip * AW_NBINS_FULL);
  const float2* d = spec + (long long)clip * T * AW_NBINS_FULL + k;
  float2* o = out + (long long)clip * T_out * AW_NBINS_FULL + k;

  const double phi = __dmul_rn(M_PI * 0.5, (double)k);
  const double two_pi = 2.0 * M_PI;
  double m0, a0, m1, a1;
  pv_polar(d, 0, T, m0, a0);
  pv_polar(d, 1, T, m1, a1);
  int i_cur = 0;
  double acc = a0;
  for (int t = 0; t < T_out; ++t) {
    const double s = __dmul_rn((double)t, rate);
    const int i = (int)s;
    const double alpha = __dsub_rn(s, (double)i);
    if (i != i_cur) {
      if (i == i_cur + 1) {
        m0 = m1;
        a0 = a1;
      } else {
        pv_polar(d, i, T, m0, a0);
      }
      pv_polar(d, i + 1, T, m1, a1);
      i_cur = i;
    }
    const double mag = __dadd_rn(__dmul_rn(__dsub_rn(1.0, alpha), m0), __dmul_rn(alpha, m1));
    double sn, cs;
    sincos(acc, &sn, &cs);
    o[(long long)t * AW_NBINS_FULL] = make_float2((float)__dmul_rn(mag, cs), (float)__dmul_rn(mag, sn));
    double dphi = __dsub_rn(__dsub_rn(a1, a0), phi);
    dphi = __dsub_rn(dphi, __dmul_rn(two_pi, rint(__ddiv_rn(dphi, two_pi))));
    acc = __dadd_rn(acc, __dadd_rn(phi, dphi));
  }
}

}  // namespace aw
