// Causal convolution of every clip with a long impulse response (the reverberation and echo attacks,
// DESIGN.md section 7): uniformly partitioned overlap-save with 1024-point transforms and hop 512.
//
//   input block b (b = 0 .. NB-1, NB = ceil(N / 512)) = x[512 (b-1), 512 (b+1)), zero outside [0, N),
//       no window; X_b = its 513-bin real FFT                                               (k_conv_fwd)
//   partition j (j = 0 .. K-1) = h[512 j, 512 j + 512) zero-padded to 1024; H_j = its rfft  (host)
//   Y_b = sum_{j = 0 .. min(K-1, b)} X_{b-j} H_j in ascending j, fp32; samples 512 .. 1023 of
//       irfft(Y_b) are y[512 b, 512 b + 512)                                                (k_conv_mac_inv)
//
// Both kernels reuse the one-warp 1024-point FFT of fft.cuh (two real frames per complex transform).
// The spectra X live in a packed half-spectrum layout of 512 slots per block: the DC and Nyquist bins of a
// real frame are real, so slot 0 holds (X[0], X[512]) and slot k holds X[k] for k = 1 .. 511.  One thread
// of k_conv_mac_inv owns one slot; slot 0's thread multiplies component-wise instead of complex, by the
// same four FMAs with two coefficients zeroed.  No atomics: a clip's output depends only on its own input
// and filter, in a fixed order.
#pragma once
#include "common.cuh"
#include "fft.cuh"

namespace aw {

#define AW_CONV_P 512              // partition length and hop
#define AW_CONV_SLOTS 512          // packed half spectrum per block
#define AW_CONV_MAXPARTS 512
#define AW_CONV_FWD_BLOCKS 16      // input blocks per CTA of k_conv_fwd (4 warps, two blocks per transform)
#define AW_CONV_R 16               // output blocks per CTA of k_conv_mac_inv
#define AW_CONV_FWD_SMEM ((1024 + 4 * 32 * AW_TR_STRIDE) * 8)
#define AW_CONV_INV_SMEM ((AW_CONV_R * AW_CONV_SLOTS + 1024 + (AW_CONV_R / 2) * 32 * AW_TR_STRIDE) * 8)

struct ConvArgs {
  const float* x; long long x_stride;   // input rows
  int n;                                // samples per clip (input and output)
  int nb;                               // blocks per clip, ceil(n / 512)
  float2* X;                            // [clip][nb][512] packed input spectra (workspace)
  const float2* H;                      // [filter][K][513] partition spectra
  int K;                                // partitions per filter
  const int* filter;                    // [clip] filter of each clip, or null (filter 0)
  const float2* twiddle;                // [k1][lane], as fft.cuh
  float* y; long long y_stride;         // output rows
};

// X_b for every block of every clip.  Warp w transforms blocks (b, b+1) as one complex FFT; the second
// half of block b's window is the first half of block b+1's, so a lane loads 48 samples, not 64.
__global__ void __launch_bounds__(128) k_conv_fwd(ConvArgs a) {
  extern __shared__ float2 csm[];
  float2* s_tw = csm;
  float2* s_tr = csm + 1024;
  const int clip = blockIdx.y, b0 = blockIdx.x * AW_CONV_FWD_BLOCKS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < 1024; i += 128) s_tw[i] = a.twiddle[i];
  __syncthreads();
  const float* xc = a.x + (long long)clip * a.x_stride;
  float2* my_tr = s_tr + warp * (32 * AW_TR_STRIDE);
  for (int p = warp; p < AW_CONV_FWD_BLOCKS / 2; p += 4) {
    const int ba = b0 + 2 * p;
    if (ba >= a.nb) break;                                  // warp-uniform
    const bool has_b = ba + 1 < a.nb;
    float re[32], im[32];
    const int base = AW_CONV_P * (ba - 1) + lane;
#pragma unroll
    for (int j = 0; j < 48; ++j) {
      const int m = base + 32 * j;
      const float v = (m >= 0 && m < a.n) ? xc[m] : 0.f;
      if (j < 32) re[j] = v;
      if (j >= 16) im[j - 16] = v;
    }
    warp_fft1024<-1>(re, im, my_tr, s_tw, lane);
    float2* xa = a.X + ((long long)clip * a.nb + ba) * AW_CONV_SLOTS;
    float2* xb = xa + AW_CONV_SLOTS;
    const int src = (32 - lane) & 31;
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) {
      // Z[k], k = lane + 32 k2, is register brev5(k2); its mirror Z[1024-k] is register brev5(31-k2) of
      // lane 32-lane (lane > 0) or register brev5(32-k2) of lane 0 (as k_analysis)
      float mr = __shfl_sync(0xffffffffu, re[brev5(31 - k2)], src);
      float mi = __shfl_sync(0xffffffffu, im[brev5(31 - k2)], src);
      if (lane == 0) {
        mr = re[brev5((32 - k2) & 31)];
        mi = im[brev5((32 - k2) & 31)];
      }
      const float zr = re[brev5(k2)], zi = im[brev5(k2)];
      // block a: (Z[k] + conj Z[N-k]) / 2 ; block b: (Z[k] - conj Z[N-k]) / (2i)
      float2 fa = make_float2(0.5f * (zr + mr), 0.5f * (zi - mi));
      float2 fb = make_float2(0.5f * (zi + mi), 0.5f * (mr - zr));
      if (k2 == 0 && lane == 0) {                           // slot 0: (DC, Nyquist), both real
        fa = make_float2(zr, re[brev5(16)]);
        fb = make_float2(zi, im[brev5(16)]);
      }
      xa[lane + 32 * k2] = fa;
      if (has_b) xb[lane + 32 * k2] = fb;
    }
  }
}

// Steps j = j0 .. j0+R-1 of the partition loop of k_conv_mac_inv (TAIL: only those below jmax) for the
// thread's slot: acc[r] += X_{b0+r-j} H_j, the X blocks read from the register ring w, where X_i sits at
// w[i mod R] (b0 and j0 are multiples of R, so every ring index is a compile-time constant).  After step j
// the ring slot of X_{b0+R-1-j}, no longer needed, takes X_{b0-1-j} (zero before the clip).  hs / hn: the
// thread's slot / the Nyquist bin in partition 0's spectrum (hn is read by slot 0 only).
template <bool TAIL>
__device__ __forceinline__ void conv_mac_steps(float2 (&acc)[AW_CONV_R], float2 (&w)[AW_CONV_R], const float2* hs,
                                               const float2* hn, const float2* xs, int b0, int j0, int jmax,
                                               bool packed) {
  constexpr int R = AW_CONV_R;
#pragma unroll
  for (int u = 0; u < R; ++u) {
    const int j = j0 + u;
    if (TAIL && j >= jmax) break;                           // block-uniform
    float2 h = hs[(long long)j * (AW_CONV_SLOTS + 1)];
    if (packed) h.y = hn[(long long)j * (AW_CONV_SLOTS + 1)].x;
    // complex: (xr hr - xi hi, xr hi + xi hr); slot 0, component-wise: (xr hr, xi hi)
    const float cP = h.x, cQ = packed ? 0.f : -h.y, cS = packed ? 0.f : h.y, cU = packed ? h.y : h.x;
    const int i = b0 - 1 - j;
    const float2 xn = i >= 0 ? xs[(long long)i * AW_CONV_SLOTS] : make_float2(0.f, 0.f);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float2 xv = w[(r - u + R) % R];
      acc[r].x = fmaf(xv.x, cP, acc[r].x);
      acc[r].x = fmaf(xv.y, cQ, acc[r].x);
      acc[r].y = fmaf(xv.x, cS, acc[r].y);
      acc[r].y = fmaf(xv.y, cU, acc[r].y);
    }
    w[(R - 1 - u) % R] = xn;
  }
}

// One CTA = AW_CONV_R consecutive output blocks of one clip; thread s owns slot s and keeps Y_{b0+r}
// (r < R) in registers while j runs over the partitions in ascending order (conv_mac_steps).  Blocks before
// the clip contribute exact zeros; partitions j >= b0 + R meet only such blocks and are skipped.  Then
// warps 0 .. R/2-1 inverse-transform pairs of blocks from shared memory and store the valid halves.
__global__ void __launch_bounds__(512, 1) k_conv_mac_inv(ConvArgs a) {
  constexpr int R = AW_CONV_R;
  extern __shared__ float2 csm[];
  float2* s_y = csm;                                        // [R][512]
  float2* s_tw = s_y + R * AW_CONV_SLOTS;
  float2* s_tr = s_tw + 1024;
  const int clip = blockIdx.y, b0 = blockIdx.x * R;
  const int s = threadIdx.x, lane = s & 31, warp = s >> 5;
  for (int i = s; i < 1024; i += 512) s_tw[i] = a.twiddle[i];

  const int nb = a.nb;
  const int f = a.filter ? a.filter[clip] : 0;
  const float2* H = a.H + (long long)f * a.K * (AW_CONV_SLOTS + 1);
  const float2* xs = a.X + (long long)clip * nb * AW_CONV_SLOTS + s;
  float2 acc[R], w[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    acc[r] = make_float2(0.f, 0.f);
    w[r] = b0 + r < nb ? xs[(long long)(b0 + r) * AW_CONV_SLOTS] : make_float2(0.f, 0.f);
  }
  const int jmax = min(a.K, b0 + R);
  int j0 = 0;
#pragma unroll 1
  for (; j0 + R <= jmax; j0 += R) conv_mac_steps<false>(acc, w, H + s, H + AW_CONV_SLOTS, xs, b0, j0, jmax, s == 0);
  if (j0 < jmax) conv_mac_steps<true>(acc, w, H + s, H + AW_CONV_SLOTS, xs, b0, j0, jmax, s == 0);
#pragma unroll
  for (int r = 0; r < R; ++r) s_y[r * AW_CONV_SLOTS + s] = acc[r];
  __syncthreads();
  if (warp >= R / 2) return;

  // ---- irfft of blocks (ba, ba+1) as one complex transform of Z = Ya + i Yb ----------------------
  const int ba = b0 + 2 * warp;
  if (ba >= nb) return;
  const bool has_b = ba + 1 < nb;
  const float2* ya = s_y + (2 * warp) * AW_CONV_SLOTS;
  const float2* yb = ya + AW_CONV_SLOTS;
  float re[32], im[32];
  const int lm = (32 - lane) & 31;
#pragma unroll
  for (int k2 = 0; k2 < 16; ++k2) {
    {
      float2 p0 = ya[lane + 32 * k2], p1 = yb[lane + 32 * k2];
      if (k2 == 0 && lane == 0) { p0.y = 0.f; p1.y = 0.f; }   // DC: real (slot 0's .y is the Nyquist bin)
      re[k2] = p0.x - p1.y;
      im[k2] = p0.y + p1.x;
    }
    {
      // mirrored entry Z[1024-k'] = conj(Ya[k']) + i conj(Yb[k']), k' = lm + 32 k2: register 31-k2
      // (lane > 0) or 32-k2 (lane 0, k2 >= 1)
      const float2 p0 = ya[lm + 32 * k2], p1 = yb[lm + 32 * k2];
      const float zr = p0.x + p1.y, zi = p1.x - p0.y;
      if (lane == 0) {
        if (k2 >= 1) { re[32 - k2] = zr; im[32 - k2] = zi; }
      } else {
        re[31 - k2] = zr;
        im[31 - k2] = zi;
      }
    }
  }
  if (lane == 0) {                                          // Z[512] = Ya[512] + i Yb[512]
    re[16] = ya[0].y;
    im[16] = yb[0].y;
  }
  warp_fft1024<1>(re, im, s_tr + warp * (32 * AW_TR_STRIDE), s_tw, lane);
  // lane k1, register p holds sample k1 + 32 brev5(p); samples 512 .. 1023 (brev5(p) >= 16, p odd) are valid
  float* yc = a.y + (long long)clip * a.y_stride;
  const float scale = 1.0f / 1024.0f;
#pragma unroll
  for (int p = 1; p < 32; p += 2) {
    const int off = 32 * (brev5(p) - 16) + lane;
    const int na = AW_CONV_P * ba + off, nbb = na + AW_CONV_P;
    if (na < a.n) yc[na] = re[p] * scale;
    if (has_b && nbb < a.n) yc[nbb] = im[p] * scale;
  }
}

}  // namespace aw
