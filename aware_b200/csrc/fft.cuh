// Shared-memory-staged radix FFT kernels for the band-limited STFT / iSTFT
// (SURVEY K2,K3,K4,K13; reference utils/audio/stft.py:28,48,55,62): the one-off passes
// around the optimisation loop -- detector STFT, initial STFT + state, out-of-band waveform,
// final synthesis.  The loop's own transforms and their adjoints are fused in spec.cuh.
//
// One warp transforms TWO real frames at once as one 1024-point complex FFT
// (z = a + i b), decomposed 32 x 32: a radix-32 pass held entirely in registers,
// a twiddle multiply, a 32x32 transpose through a padded per-warp shared tile, and
// a second in-register radix-32 pass.  No __syncthreads inside the transform.
// Only the embedding band (bins bin0 .. bin0+nbins-1) is read or written: the
// out-of-band bins never exist on the device (detection/multibit_detector.py:34-37,
// embedding/multibit_embedder.py:104), and by linearity the out-of-band part of
// the reference's iSTFT is a per-clip constant waveform (y_oob).
//
// The kernels are templated on the 32-bin groups [K2LO, K2HI] that contain the band
// (44.1 kHz: bins 12..92 -> groups 0..2; 16 kHz: bins 32..256 -> groups 1..8), so all
// per-bin-group control flow is resolved at compile time.
#pragma once
#include "common.cuh"

namespace aw {

// cos/sin(2 pi j / 32), j = 0..15
__constant__ float c_cos32[16] = {
    1.0f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254524f,
    0.70710678118654757f, 0.55557023301960229f, 0.38268343236508984f, 0.19509032201612833f,
    0.0f, -0.19509032201612819f, -0.38268343236508973f, -0.55557023301960196f,
    -0.70710678118654746f, -0.83146961230254535f, -0.92387953251128674f, -0.98078528040323043f};
__constant__ float c_sin32[16] = {
    0.0f, 0.19509032201612825f, 0.38268343236508978f, 0.55557023301960218f,
    0.70710678118654746f, 0.83146961230254524f, 0.92387953251128674f, 0.98078528040323043f,
    1.0f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254546f,
    0.70710678118654757f, 0.55557023301960218f, 0.38268343236508989f, 0.19509032201612861f};

// One radix-2 decimation-in-frequency stage over 32 register-resident points.
// SIGN = -1: forward (e^{-i}), +1: inverse (e^{+i}).
template <int SIGN, int HALF>
__device__ __forceinline__ void fft32_stage(float (&re)[32], float (&im)[32]) {
#pragma unroll
  for (int g = 0; g < 32; g += 2 * HALF) {
#pragma unroll
    for (int j = 0; j < HALF; ++j) {
      const int i0 = g + j, i1 = g + j + HALF;
      const float ar = re[i0], ai = im[i0], br = re[i1], bi = im[i1];
      re[i0] = ar + br;
      im[i0] = ai + bi;
      const float dr = ar - br, di = ai - bi;
      const int tw = j * (16 / HALF);
      if (tw == 0) {
        re[i1] = dr;
        im[i1] = di;
      } else if (tw == 8) {            // W = SIGN * i
        re[i1] = -SIGN * di;
        im[i1] = SIGN * dr;
      } else {
        const float c = c_cos32[tw], s = SIGN * c_sin32[tw];
        re[i1] = dr * c - di * s;
        im[i1] = dr * s + di * c;
      }
    }
  }
}

__host__ __device__ constexpr int brev5(int p) {
  return ((p & 1) << 4) | ((p & 2) << 2) | (p & 4) | ((p & 8) >> 2) | ((p & 16) >> 4);
}

// In-register 32-point DFT, natural order in, BIT-REVERSED order out:
// register p holds X[brev5(p)].  Consumers index with brev5() at compile time, which
// costs nothing, whereas an explicit un-permutation costs ~70 register moves.
template <int SIGN>
__device__ __forceinline__ void fft32_br(float (&re)[32], float (&im)[32]) {
  fft32_stage<SIGN, 16>(re, im);
  fft32_stage<SIGN, 8>(re, im);
  fft32_stage<SIGN, 4>(re, im);
  fft32_stage<SIGN, 2>(re, im);
  fft32_stage<SIGN, 1>(re, im);
}

#define AW_TR_STRIDE 33
#define AW_TR_FLOATS (2 * 32 * AW_TR_STRIDE)   // per-warp transpose tile (float2 [32][33])

// 1024-point complex FFT across one warp.
//   in : lane l, register j  holds x[32 j + l]
//   out: lane k1, register p holds X[k1 + 32 * brev5(p)]
// s_tr: this warp's float2[32*33]; s_tw[k1*32 + l] = (cos, sin)(2 pi l k1 / 1024), a layout
// in which both the twiddle reads and the transpose accesses are bank-conflict free.
template <int SIGN>
__device__ __forceinline__ void warp_fft1024(float (&re)[32], float (&im)[32], float2* s_tr,
                                             const float2* s_tw, int lane) {
  fft32_br<SIGN>(re, im);
#pragma unroll
  for (int p = 0; p < 32; ++p) {
    const int k1 = brev5(p);
    const float2 w = s_tw[k1 * 32 + lane];
    const float c = w.x, s = SIGN * w.y;
    s_tr[k1 * AW_TR_STRIDE + lane] = make_float2(re[p] * c - im[p] * s, re[p] * s + im[p] * c);
  }
  __syncwarp();
#pragma unroll
  for (int n2 = 0; n2 < 32; ++n2) {
    const float2 t = s_tr[lane * AW_TR_STRIDE + n2];
    re[n2] = t.x;
    im[n2] = t.y;
  }
  __syncwarp();
  fft32_br<SIGN>(re, im);
}

// 1 / sum_t w^2[m - 256 t] over the frames that cover padded sample m (torch.istft's window
// envelope, accumulated in ascending t).  `env256[256 + j]` holds the reciprocal of the
// interior value (4 covering frames); edges are evaluated directly.  Multiplying by the
// correctly rounded reciprocal differs from torch's division by <= 1 ulp.
__device__ __forceinline__ float ola_inv_envelope(int m, int T, const float* s_win,
                                                  const float* __restrict__ env256) {
  const int hop = m >> 8;
  if (hop >= 3 && hop <= T - 1) return env256[256 + (m & 255)];
  int tlo = m >= AW_NFFT ? ((m - (AW_NFFT - 1) + (AW_HOP - 1)) >> 8) : 0;
  int thi = hop;
  if (thi > T - 1) thi = T - 1;
  float e = 0.f;
  for (int t = tlo; t <= thi; ++t) {
    const float w = s_win[m - (t << 8)];
    e = __fmaf_rn(w, w, e);
  }
  return __fdiv_rn(1.0f, e);
}

// per-iteration NAdam scalars (torch/optim/nadam.py _single_tensor_nadam)
struct NadamStep {
  float a_g;      // -lr (1 - mu_t) / (1 - prod mu)
  float a_m;      // -lr mu_{t+1} / (1 - prod mu * mu_{t+1})
  float inv_bc2;  // 1 / (1 - beta2^t)   (ATen divides by a CPU scalar as x * (1/s))
  float pad;
};

// ---------------------------------------------------------------------------
// analysis: frames -> band spectrum
// ---------------------------------------------------------------------------
enum { ANA_MAG = 0, ANA_INIT = 1, ANA_CPLX = 2 };   // CPLX: complex band spectrum only (spectc.cuh's S_oob)
// FULL: all 513 bins of the input as it is (no peak scaling), complex, for aw_stft_full; bin0 = 0,
// nbins = AW_NBINS_FULL, instantiated over k2 = 0..16 (lane 0 of k2 = 16 is the Nyquist bin, its own mirror)
enum { ANA_FULL = 3 };
#define AW_NBINS_FULL 513

struct AnaArgs {
  const float* sig;            // per clip signal x
  long long sig_stride;
  int len;                     // signal length N
  int T, bin0, nbins;
  const unsigned long long* peak;   // [clip] packed peak of x
  const float* window;         // [1024] device
  const float2* twiddle;       // [1024] device, layout [k1][lane]
  const float* env256;         // [512] interior window envelope and its reciprocal
  // outputs
  float* mag;                  // [clip][T][nbins]  (MAG; INIT -> c0)
  float2* ph;                  // [clip][T][nbins]  (INIT -> u)
  // embed state initialised by INIT
  float* c; float* m; float* v; float* cbest;
  float tol_ratio;             // 10^(-tolerance_db/20) as float32
};

#define AW_ANA_FRAMES 16
#define AW_ANA_SIG (AW_ANA_FRAMES * AW_HOP + 768)
#define AW_ANA_SMEM ((AW_ANA_SIG + 1024 + 2048 + 4 * AW_TR_FLOATS) * 4)

template <int MODE, int K2LO, int K2HI>
__global__ void __launch_bounds__(128, 3) k_analysis(AnaArgs a) {
  extern __shared__ float smem[];
  float* s_sig = smem;
  float* s_win = s_sig + AW_ANA_SIG;
  float2* s_tw = reinterpret_cast<float2*>(s_win + 1024);
  float2* s_tr = s_tw + 1024;

  const int clip = blockIdx.y;
  const int t0 = blockIdx.x * AW_ANA_FRAMES;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = a.len, T = a.T;

  for (int i = tid; i < 1024; i += 128) {
    s_win[i] = a.window[i];
    s_tw[i] = a.twiddle[i];
  }
  __syncthreads();   // tables

  // ---- stage the (scaled / padded) signal segment -------------------------
  const float* sig = a.sig + (long long)clip * a.sig_stride;
  const int m_end = AW_HOP * (T - 1) + AW_NFFT;   // padded length
  if (MODE == ANA_FULL) {
    for (int j = tid; j < AW_ANA_SIG; j += 128) {
      const int m = AW_HOP * t0 + j;
      s_sig[j] = m < m_end ? sig[reflect_idx(m - AW_HALF, L)] : 0.f;
    }
  } else {
    const unsigned long long pk = a.peak[clip];
    const float p1 = peak_value(pk);
    const float d1 = p1 + 1e-8f;
    // x / d1 as one multiply by the correctly rounded reciprocal (<= 1 ulp from the division)
    const float inv = __fdiv_rn(1.0f, d1);
    for (int j = tid; j < AW_ANA_SIG; j += 128) {
      const int m = AW_HOP * t0 + j;
      float val = 0.f;
      if (m < m_end) val = sig[reflect_idx(m - AW_HALF, L)] * inv;
      s_sig[j] = val;
    }
  }
  __syncthreads();

  float2* my_tr = s_tr + warp * (32 * AW_TR_STRIDE);

  for (int p = warp; p < AW_ANA_FRAMES / 2; p += 4) {
    const int ta = t0 + 2 * p, tb = ta + 1;
    if (ta >= T) break;                     // warp-uniform
    float re[32], im[32];
    const float* fa = s_sig + AW_HOP * (2 * p) + lane;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float w = s_win[32 * j + lane];
      re[j] = fa[32 * j] * w;
      im[j] = fa[32 * j + AW_HOP] * w;      // frame tb (zeros past the end: staged as 0)
    }
    warp_fft1024<-1>(re, im, my_tr, s_tw, lane);

    const bool has_b = tb < T;
    const int src = (32 - lane) & 31;
#pragma unroll
    for (int k2 = K2LO; k2 <= K2HI; ++k2) {
      // Z[k], k = lane + 32 k2, is register brev5(k2); its mirror Z[1024-k] is register
      // brev5(31-k2) of lane 32-lane (lane > 0) or register brev5(32-k2) of lane 0.
      float mr = __shfl_sync(0xffffffffu, re[brev5(31 - k2)], src);
      float mi = __shfl_sync(0xffffffffu, im[brev5(31 - k2)], src);
      // (lane 0 of k2 = 0 is the DC bin, its own mirror: only the full spectrum contains it)
      if ((k2 >= 1 || MODE == ANA_FULL) && lane == 0) {
        mr = re[brev5((32 - k2) & 31)];
        mi = im[brev5((32 - k2) & 31)];
      }
      const int b = lane + 32 * k2 - a.bin0;
      if (b < 0 || b >= a.nbins) continue;
      const float zr = re[brev5(k2)], zi = im[brev5(k2)];
      // frame a: (Z[k] + conj Z[N-k]) / 2 ; frame b: (Z[k] - conj Z[N-k]) / (2i)
      const float fr[2] = {0.5f * (zr + mr), 0.5f * (zi + mi)};
      const float fi[2] = {0.5f * (zi - mi), 0.5f * (mr - zr)};
#pragma unroll
      for (int f = 0; f < 2; ++f) {
        if (f == 1 && !has_b) break;
        const long long o = ((long long)clip * T + (ta + f)) * a.nbins + b;
        const float sr = fr[f], si = fi[f];
        if (MODE == ANA_CPLX || MODE == ANA_FULL) {
          a.ph[o] = make_float2(sr, si);
        } else {
          const float mag = sqrtf(sr * sr + si * si);
          a.mag[o] = mag;
          if (MODE == ANA_INIT) {
            const float inv = mag > 0.f ? 1.0f / mag : 0.f;
            a.ph[o] = make_float2(sr * inv, si * inv);
          }
          if (MODE == ANA_INIT) {
            a.c[o] = mag;
            a.cbest[o] = mag;
            a.m[o] = 0.f;
            a.v[o] = 0.f;
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// synthesis: band spectrum -> windowed overlap-add
// ---------------------------------------------------------------------------
enum { SYN_OOB = 0, SYN_WAVE = 1 };   // the loop passes live in spec.cuh
// FULL: torch.istft(spec, length=L) of a full complex spectrum (`ph`: [clip][T][AW_NBINS_FULL], no `amp`,
// no y_oob, no peak) into y with row stride x_stride (aw_istft_full)
enum { SYN_FULL = 2 };

struct SynArgs {
  const float* amp;            // [clip][T][nbins] real factor (c / cbest / dA~)
  const float2* ph;            // [clip][T][nbins] unit phasor (u / q)
  int T, L, bin0, nbins;
  float scale;                 // 1/N (irfft)
  const float* window;
  const float2* twiddle;       // layout [k1][lane]
  const float* env256;
  // SYN_OOB: y_oob = x/(peak_x+1e-8) - ola/env  (SYN_FULL: x_stride is the row stride of y, x is unused)
  const float* x; long long x_stride; const unsigned long long* peak_x;
  float* y_oob;                // [clip][L]   (OOB: out; WAVE: in)
  float* z_oob;                // [clip][L]   (OOB: optional out) y_oob * envelope, for spec.cuh
  // SYN_WAVE: y = ola/env + y_oob, peak_y
  float* y;                    // [clip][L]   (WAVE: out)
  unsigned long long* peak_y;  // [clip]      (WAVE: atomicMax out)
  int pk_lo, pk_hi;            // WAVE: samples competing for the peak (frame-sharded mode); pk_hi = 0: all
};

#define AW_SYN_FRAMES 32
#define AW_SYN_HOPS 29
#define AW_SYN_OLA (AW_SYN_FRAMES * AW_HOP + 768)
#define AW_SYN_SMEM ((AW_SYN_OLA + 1024 + 2048 + 4 * AW_TR_FLOATS) * 4)

// Build the hermitian pair for frames (ta, tb) of one warp, inverse-FFT it and return the
// two windowed real frames in (re[p], im[p]) for sample n = lane + 32 * brev5(p).
template <int K2LO, int K2HI>
__device__ __forceinline__ void syn_pair(const SynArgs& a, int clip, int ta, int tb, bool va, bool vb,
                                         float (&re)[32], float (&im)[32], float2* my_tr,
                                         const float2* s_tw, const float* s_win, int lane) {
#pragma unroll
  for (int j = 0; j < 32; ++j) { re[j] = 0.f; im[j] = 0.f; }
  const long long oa = ((long long)clip * a.T + (va ? ta : 0)) * a.nbins;
  const long long ob = ((long long)clip * a.T + (vb ? tb : 0)) * a.nbins;
  const float sa = va ? a.scale : 0.f, sb = vb ? a.scale : 0.f;
  const int lm = (32 - lane) & 31;
#pragma unroll
  for (int k2 = K2LO; k2 <= K2HI; ++k2) {
    // direct entry Z[k], k = lane + 32 k2:  Xa + i Xb
    {
      const int b = lane + 32 * k2 - a.bin0;
      const bool ok = b >= 0 && b < a.nbins;
      const int bc = ok ? b : 0;
      const float s0 = ok ? sa * a.amp[oa + bc] : 0.f, s1 = ok ? sb * a.amp[ob + bc] : 0.f;
      const float2 p0 = a.ph[oa + bc], p1 = a.ph[ob + bc];
      const float ar = s0 * p0.x, ai = s0 * p0.y, br = s1 * p1.x, bi = s1 * p1.y;
      re[k2] = ar - bi;
      im[k2] = ai + br;
    }
    // mirrored entry Z[1024-k'] = conj(Xa[k']) + i conj(Xb[k']), k' = ((32-lane)&31) + 32 k2,
    // which lives in this lane at register 31-k2 (lane > 0) or 32-k2 (lane 0)
    {
      const int kp = lm + 32 * k2;
      const int b = kp - a.bin0;
      const bool ok = b >= 0 && b < a.nbins && kp > 0;
      const int bc = ok ? b : 0;
      const float s0 = ok ? sa * a.amp[oa + bc] : 0.f, s1 = ok ? sb * a.amp[ob + bc] : 0.f;
      const float2 p0 = a.ph[oa + bc], p1 = a.ph[ob + bc];
      const float ar = s0 * p0.x, ai = s0 * p0.y, br = s1 * p1.x, bi = s1 * p1.y;
      const float zr = ar + bi, zi = br - ai;
      if (lane == 0) {
        if (k2 >= 1) { re[(32 - k2) & 31] = zr; im[(32 - k2) & 31] = zi; }
      } else {
        re[31 - k2] = zr;
        im[31 - k2] = zi;
      }
    }
  }
  warp_fft1024<1>(re, im, my_tr, s_tw, lane);
#pragma unroll
  for (int p = 0; p < 32; ++p) {
    const float w = s_win[lane + 32 * brev5(p)];
    re[p] *= w;
    im[p] *= w;
  }
}

// syn_pair for a full spectrum: all 513 bins, complex.  As irfft does, the imaginary parts of the DC and
// Nyquist bins are ignored.  Lane l holds Z[l + 32 k2] (k2 = 0..15) in register k2 and the mirrored
// entries Z[1024 - k'] in registers 16..31; lane 0's register 16 is the Nyquist bin Z[512].
__device__ __forceinline__ void syn_pair_full(const SynArgs& a, int clip, int ta, int tb, bool va, bool vb,
                                              float (&re)[32], float (&im)[32], float2* my_tr,
                                              const float2* s_tw, const float* s_win, int lane) {
  const float2* xa = a.ph + ((long long)clip * a.T + (va ? ta : 0)) * AW_NBINS_FULL;
  const float2* xb = a.ph + ((long long)clip * a.T + (vb ? tb : 0)) * AW_NBINS_FULL;
  const float sa = va ? a.scale : 0.f, sb = vb ? a.scale : 0.f;
  const int lm = (32 - lane) & 31;
#pragma unroll
  for (int k2 = 0; k2 < 16; ++k2) {
    {
      float2 p0 = xa[lane + 32 * k2], p1 = xb[lane + 32 * k2];
      if (k2 == 0 && lane == 0) { p0.y = 0.f; p1.y = 0.f; }
      const float ar = sa * p0.x, ai = sa * p0.y, br = sb * p1.x, bi = sb * p1.y;
      re[k2] = ar - bi;
      im[k2] = ai + br;
    }
    {
      const float2 p0 = xa[lm + 32 * k2], p1 = xb[lm + 32 * k2];
      const float ar = sa * p0.x, ai = sa * p0.y, br = sb * p1.x, bi = sb * p1.y;
      const float zr = ar + bi, zi = br - ai;
      if (lane == 0) {
        if (k2 >= 1) { re[32 - k2] = zr; im[32 - k2] = zi; }
      } else {
        re[31 - k2] = zr;
        im[31 - k2] = zi;
      }
    }
  }
  if (lane == 0) {
    re[16] = sa * xa[512].x;
    im[16] = sb * xb[512].x;
  }
  warp_fft1024<1>(re, im, my_tr, s_tw, lane);
#pragma unroll
  for (int p = 0; p < 32; ++p) {
    const float w = s_win[lane + 32 * brev5(p)];
    re[p] *= w;
    im[p] *= w;
  }
}

template <int MODE, int K2LO, int K2HI>
__device__ __forceinline__ void syn_frames(const SynArgs& a, int clip, int ta, int tb, bool va, bool vb,
                                           float (&re)[32], float (&im)[32], float2* my_tr,
                                           const float2* s_tw, const float* s_win, int lane) {
  if (MODE == SYN_FULL)
    syn_pair_full(a, clip, ta, tb, va, vb, re, im, my_tr, s_tw, s_win, lane);
  else
    syn_pair<K2LO, K2HI>(a, clip, ta, tb, va, vb, re, im, my_tr, s_tw, s_win, lane);
}

__device__ __forceinline__ void ola_add(float* s_ola, int off, const float (&v)[32], int lane) {
#pragma unroll
  for (int p = 0; p < 32; ++p) s_ola[off + lane + 32 * brev5(p)] += v[p];
}

// One CTA (4 warps) produces 29 hops of output from 32 frames.  Warp w owns the 8
// consecutive frames f0+8w .. f0+8w+7 (four frame pairs).  Frames 0..4 of a warp lie
// entirely inside the warp's private 2048-sample stripe of the overlap-add buffer and are
// accumulated before the single __syncthreads; frames 5..7 spill into the next warp's stripe
// and are accumulated after it (frame 5 waits in registers across the barrier).  No two
// warps ever add to the same address concurrently, so the accumulation needs no atomics
// and its order is fixed (deterministic).
template <int MODE, int K2LO, int K2HI>
__global__ void __launch_bounds__(128, 2) k_synthesis(SynArgs a) {
  extern __shared__ float smem[];
  float* s_ola = smem;
  float* s_win = s_ola + AW_SYN_OLA;
  float2* s_tw = reinterpret_cast<float2*>(s_win + 1024);
  float2* s_tr = s_tw + 1024;
  __shared__ unsigned long long s_pk[4];

  const int clip = blockIdx.y;
  const int h0 = blockIdx.x * AW_SYN_HOPS;        // first output hop (padded axis)
  const int f0 = h0 - 3;                           // first contributing frame
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = a.T, L = a.L;

  for (int i = tid; i < 1024; i += 128) {
    s_win[i] = a.window[i];
    s_tw[i] = a.twiddle[i];
  }
  for (int i = tid; i < AW_SYN_OLA; i += 128) s_ola[i] = 0.f;
  __syncthreads();

  float2* my_tr = s_tr + warp * (32 * AW_TR_STRIDE);
  const int fw = f0 + 8 * warp;                    // this warp's first frame
  const int ow = AW_HOP * 8 * warp;                // its stripe in s_ola
  float re[32], im[32];
  float hold[32];
  bool hold_valid = false;
#pragma unroll 1
  for (int pr = 0; pr < 3; ++pr) {                 // pairs (0,1) (2,3) (4,5)
    const int ta = fw + 2 * pr, tb = ta + 1;
    const bool va = ta >= 0 && ta < T, vb = tb >= 0 && tb < T;
    if (!(va || vb)) continue;                     // warp-uniform
    syn_frames<MODE, K2LO, K2HI>(a, clip, ta, tb, va, vb, re, im, my_tr, s_tw, s_win, lane);
    if (va) ola_add(s_ola, ow + AW_HOP * (2 * pr), re, lane);
    if (pr < 2) {
      if (vb) ola_add(s_ola, ow + AW_HOP * (2 * pr + 1), im, lane);
    } else if (vb) {                               // frame 5 spills: keep it for after the barrier
#pragma unroll
      for (int p = 0; p < 32; ++p) hold[p] = im[p];
      hold_valid = true;
    }
  }
  __syncthreads();
  if (hold_valid) ola_add(s_ola, ow + AW_HOP * 5, hold, lane);
  {
    const int ta = fw + 6, tb = ta + 1;
    const bool va = ta >= 0 && ta < T, vb = tb >= 0 && tb < T;
    if (va || vb) {
      syn_frames<MODE, K2LO, K2HI>(a, clip, ta, tb, va, vb, re, im, my_tr, s_tw, s_win, lane);
      if (va) ola_add(s_ola, ow + AW_HOP * 6, re, lane);
      if (vb) ola_add(s_ola, ow + AW_HOP * 7, im, lane);
    }
  }
  __syncthreads();

  // ---- epilogue over this tile's output samples ----------------------------
  const int m_lo = AW_HOP * h0;
  const int m_total = AW_HOP * (T - 1) + AW_NFFT;
  int m_hi = m_lo + AW_HOP * AW_SYN_HOPS;
  if (m_hi > m_total) m_hi = m_total;

  if (MODE == SYN_FULL) {
    // output sample n = m - 512 < L; m < m_total bounds it by 256 (T - 1) + 512, past which torch.istft
    // pads with zeros (the caller's job).  The last 512 samples are the tail of the final frame over its
    // small window envelope, as torch computes them.
    float* yc = a.y + (long long)clip * a.x_stride;
    for (int m = m_lo + tid; m < m_hi; m += 128) {
      const int n = m - AW_HALF;
      if (n < 0 || n >= L) continue;
      yc[n] = s_ola[m - AW_HOP * f0] * ola_inv_envelope(m, T, s_win, a.env256);
    }
    return;
  }

  {
    float best = -1.f;
    int best_n = 0;
    float rdx = 1.f;
    const int pk_lo = a.pk_lo, pk_hi = a.pk_hi > 0 ? a.pk_hi : L;
    if (MODE == SYN_OOB) rdx = __fdiv_rn(1.0f, peak_value(a.peak_x[clip]) + 1e-8f);
    const bool interior = h0 >= 3 && h0 + AW_SYN_HOPS <= T - 1 && m_lo >= AW_HALF && m_hi - AW_HALF <= L;
    if (interior) {
      // 4 consecutive samples per thread: float4 traffic, table envelope, no range checks
      const float* so = s_ola + (m_lo - AW_HOP * f0);
      const long long ob = (long long)clip * L + (m_lo - AW_HALF);
      for (int i = tid * 4; i < AW_HOP * AW_SYN_HOPS; i += 512) {
        const float4 o4 = *reinterpret_cast<const float4*>(so + i);
        const float4 e4 = *reinterpret_cast<const float4*>(a.env256 + 256 + (i & 255));
        float yb[4] = {o4.x * e4.x, o4.y * e4.y, o4.z * e4.z, o4.w * e4.w};
        if (MODE == SYN_OOB) {
          const float* xp = a.x + (long long)clip * a.x_stride + (m_lo - AW_HALF) + i;
          const float yo[4] = {xp[0] * rdx - yb[0], xp[1] * rdx - yb[1], xp[2] * rdx - yb[2], xp[3] * rdx - yb[3]};
          *reinterpret_cast<float4*>(a.y_oob + ob + i) = make_float4(yo[0], yo[1], yo[2], yo[3]);
          if (a.z_oob) {
            const float4 v4 = *reinterpret_cast<const float4*>(a.env256 + (i & 255));
            *reinterpret_cast<float4*>(a.z_oob + ob + i) =
                make_float4(yo[0] * v4.x, yo[1] * v4.y, yo[2] * v4.z, yo[3] * v4.w);
          }
        } else {
          const float4 q4 = *reinterpret_cast<const float4*>(a.y_oob + ob + i);
          const float yy[4] = {yb[0] + q4.x, yb[1] + q4.y, yb[2] + q4.z, yb[3] + q4.w};
          *reinterpret_cast<float4*>(a.y + ob + i) = make_float4(yy[0], yy[1], yy[2], yy[3]);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int nn = m_lo - AW_HALF + i + k;
            if (fabsf(yy[k]) > best && nn >= pk_lo && nn < pk_hi) { best = fabsf(yy[k]); best_n = nn; }
          }
        }
      }
    } else {
      for (int m = m_lo + tid; m < m_hi; m += 128) {
        const int n = m - AW_HALF;
        if (n < 0 || n >= L) continue;
        const float yb = s_ola[m - AW_HOP * f0] * ola_inv_envelope(m, T, s_win, a.env256);
        const long long o = (long long)clip * L + n;
        if (MODE == SYN_OOB) {
          const float yo = a.x[(long long)clip * a.x_stride + n] * rdx - yb;
          a.y_oob[o] = yo;
          if (a.z_oob) a.z_oob[o] = __fdiv_rn(yo, ola_inv_envelope(m, T, s_win, a.env256));
        } else {
          const float yy = yb + a.y_oob[o];
          a.y[o] = yy;
          if (fabsf(yy) > best && n >= pk_lo && n < pk_hi) { best = fabsf(yy); best_n = n; }
        }
      }
    }
    if (MODE == SYN_WAVE) {
      // strict '>' in ascending sample order keeps the lowest index per thread; the packed
      // u64 max then keeps the lowest index across threads, warps and tiles
      unsigned long long pk = best >= 0.f ? pack_peak(best, (unsigned)best_n) : 0ull;
      pk = warp_max_u64(pk);
      if (lane == 0) s_pk[warp] = pk;
      __syncthreads();
      if (tid == 0) {
        for (int w = 1; w < 4; ++w) pk = s_pk[w] > pk ? s_pk[w] : pk;
        atomicMax(a.peak_y + clip, pk);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// per-clip peak |x| (utils/audio/waveform.py:19) and final normalise
// ---------------------------------------------------------------------------
// order-preserving int encoding of a float (signed max through an integer atomicMax)
__device__ __forceinline__ int float_ordered(float f) {
  const int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_float(int o) {
  return __int_as_float(o >= 0 ? o : o ^ 0x7fffffff);
}
// One pass over the clip: packed (|x| max, lowest index) and, with `smax`, also the SIGNED max
// (service/embed.py:69 rescales by np.max(audio), not by the peak).  4 samples per load where the
// row is 16-byte aligned.  smax must be pre-set to INT_MIN.
__global__ void __launch_bounds__(256) k_peak(const float* x, long long stride, int n,
                                              unsigned long long* peak, int* smax) {
  const int clip = blockIdx.y;
  const float* p = x + (long long)clip * stride;
  unsigned long long pk = 0ull;
  float sm = -INFINITY;
  const bool vec = ((reinterpret_cast<uintptr_t>(p) & 15) == 0);
  const int n4 = vec ? n >> 2 : 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(p)[i];
    const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned long long q = pack_peak(fabsf(e[k]), (unsigned)(4 * i + k));
      pk = q > pk ? q : pk;
      sm = fmaxf(sm, e[k]);
    }
  }
  for (int i = 4 * n4 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long q = pack_peak(fabsf(p[i]), (unsigned)i);
    pk = q > pk ? q : pk;
    sm = fmaxf(sm, p[i]);
  }
  __shared__ unsigned long long s_pk[8];
  __shared__ float s_sm[8];
  pk = warp_max_u64(pk);
  sm = warp_max(sm);
  if ((threadIdx.x & 31) == 0) { s_pk[threadIdx.x >> 5] = pk; s_sm[threadIdx.x >> 5] = sm; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { pk = s_pk[w] > pk ? s_pk[w] : pk; sm = fmaxf(sm, s_sm[w]); }
    atomicMax(peak + clip, pk);
    if (smax) atomicMax(smax + clip, float_ordered(sm));
  }
}

// out = y / (peak + 1e-8) [* scale[clip]]   (multibit_embedder.py:185-192, service/embed.py:73)
// `smax` (order-encoded signed max of the input, from k_peak) takes the place of `scale`
__global__ void __launch_bounds__(256) k_final_normalize(const float* y, int L,
                                                         const unsigned long long* peak,
                                                         const float* scale, const int* smax, float* out,
                                                         long long out_stride) {
  const int clip = blockIdx.y;
  const float d = peak_value(peak[clip]) + 1e-8f;
  const bool scaled = scale || smax;
  const float s = scale ? scale[clip] : (smax ? ordered_float(smax[clip]) : 1.f);
  const float* yc = y + (long long)clip * L;
  float* oc = out + (long long)clip * out_stride;
  if ((out_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {      // L % 256 == 0
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < (L >> 2); i += gridDim.x * blockDim.x) {
      const float4 t = reinterpret_cast<const float4*>(yc)[i];
      float v[4] = {__fdiv_rn(t.x, d), __fdiv_rn(t.y, d), __fdiv_rn(t.z, d), __fdiv_rn(t.w, d)};
      if (scaled) {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __fmul_rn(s, v[k]);
      }
      reinterpret_cast<float4*>(oc)[i] = make_float4(v[0], v[1], v[2], v[3]);
    }
    return;
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) {
    float v = __fdiv_rn(yc[i], d);
    if (scaled) v = __fmul_rn(s, v);
    oc[i] = v;
  }
}

}  // namespace aw
