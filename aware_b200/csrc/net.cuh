// Detector front end / head and their adjoints (SURVEY K5-K8, K10-K12, K14, K16;
// reference detection/multibit_detector_net.py:109-140, modules/mel.py:195,
// globalStandardize.py:16-21, BRH.py:16-27, embedding/losses.py:38-42).
// Layouts: spectra [clip][T][nbins]; mel [clip][T][128]; activations channels-last
// [clip * Tp_pad + j][C] with Tp_pad = T' rounded up to 128 rows (pad rows are 0).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "common.cuh"

namespace aw {

// activation element access (float for the fp32 / TF32 paths, bf16 for the bf16 embed path)
__device__ __forceinline__ float act_ld(const float* p) { return *p; }
__device__ __forceinline__ float act_ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void act_st(float* p, float v) { *p = v; }
__device__ __forceinline__ void act_st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void act_ld4(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void act_ld4(const __nv_bfloat16* p, float (&v)[4]) {
  const uint2 t = *reinterpret_cast<const uint2*>(p);
  v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
  v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
}
__device__ __forceinline__ void act_st4(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void act_st4(__nv_bfloat16* p, const float (&v)[4]) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a),
                                            *reinterpret_cast<const uint32_t*>(&b));
}

__device__ __forceinline__ float act_ld(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ void act_st(__half* p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ void act_ld4(const __half* p, float (&v)[4]) {
  const uint2 t = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void act_st4(__half* p, const float (&v)[4]) {
  const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a),
                                            *reinterpret_cast<const uint32_t*>(&b));
}

struct SparseMel {
  // CSR over mel channels (band-relative columns) and CSC over band bins
  const int* rowptr;   // [129]
  const int* col;      // [nnz]
  const float* val;    // [nnz]
  const int* colptr;   // [nbins + 1]
  const int* row;      // [nnz]
  const float* valT;   // [nnz]
};

struct ChanStats {      // per clip, per mel channel (forward, reused by backward)
  float mu, rstd, varratio, pad;   // varratio = var / (var + eps)
};

// ---- mel projection + per-channel sums -------------------------------------
#define AW_MEL_FRAMES 32
// peak_y != null: `mag` is the spectrum of the UN-normalised waveform (spec.cuh) and the two
// stacked peak normalisers (waveform.py:19) are applied here as one factor 1/(d1 d2).
__global__ void __launch_bounds__(128) k_mel(const float* __restrict__ mag, int T, int nb,
                                             SparseMel sm, float* __restrict__ M,
                                             double* __restrict__ chan_part,
                                             const unsigned long long* __restrict__ peak_y) {
  extern __shared__ float s_a[];   // [AW_MEL_FRAMES][nb]
  const int clip = blockIdx.y, t0 = blockIdx.x * AW_MEL_FRAMES, c = threadIdx.x;
  const int nf = min(AW_MEL_FRAMES, T - t0);
  const float* src = mag + ((long long)clip * T + t0) * nb;
  float inv = 1.f;
  if (peak_y) {
    const float p1 = peak_value(peak_y[clip]);
    const float d1 = p1 + 1e-8f;
    const float d2 = __fdiv_rn(p1, d1) + 1e-8f;
    inv = __fdiv_rn(__fdiv_rn(1.0f, d1), d2);
  }
  for (int i = threadIdx.x; i < AW_MEL_FRAMES * nb; i += 128) s_a[i] = i < nf * nb ? src[i] * inv : 0.f;
  __syncthreads();
  // filter taps outermost: each (weight, bin) pair of this channel is fetched once and applied to
  // all 32 staged frames (most channels have 2-5 taps inside the band, many have none)
  const int e0 = sm.rowptr[c], e1 = sm.rowptr[c + 1];
  float acc[AW_MEL_FRAMES];
#pragma unroll
  for (int f = 0; f < AW_MEL_FRAMES; ++f) acc[f] = 0.f;
  for (int e = e0; e < e1; ++e) {
    const float w = sm.val[e];
    const float* col = s_a + sm.col[e];
#pragma unroll
    for (int f = 0; f < AW_MEL_FRAMES; ++f) acc[f] = fmaf(w, col[f * nb], acc[f]);
  }
  double s1 = 0.0, s2 = 0.0;
#pragma unroll
  for (int f = 0; f < AW_MEL_FRAMES; ++f) {
    if (f < nf) {
      M[((long long)clip * T + t0 + f) * AW_NMEL + c] = acc[f];
      s1 += acc[f];
      s2 += (double)acc[f] * acc[f];
    }
  }
  // per-block partial sums, reduced in fixed order by the consumers (deterministic)
  double* p = chan_part + (((long long)clip * gridDim.x + blockIdx.x) * AW_NMEL + c) * 2;
  p[0] = s1;
  p[1] = s2;
}

// Second-level reduction for long clips: [clip][nblk][W] doubles -> [clip][ceil(nblk/G)][W],
// each output the fixed-order sum of G consecutive blocks (deterministic).  W = 256 for the
// per-channel (sum, sum-of-squares) pairs, 1 for scalar partials.
__global__ void __launch_bounds__(256) k_reduce_partials(const double* __restrict__ in, int nblk, int W,
                                                         int G, double* __restrict__ out) {
  const int clip = blockIdx.z, ob = blockIdx.y, nob = gridDim.y;
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const int b0 = ob * G, b1 = min(b0 + G, nblk);
  double s = 0.0;
  for (int b = b0; b < b1; ++b) s += in[((long long)clip * nblk + b) * W + w];
  out[((long long)clip * nob + ob) * W + w] = s;
}

// sum of `nblk` per-block partials [clip][nblk][128][2] for channel c, in block order
__device__ __forceinline__ void sum_partials(const double* __restrict__ part, int clip, int nblk, int c,
                                             double& s1, double& s2) {
  s1 = 0.0;
  s2 = 0.0;
  const double* p = part + ((long long)clip * nblk * AW_NMEL + c) * 2;
  // eight blocks' loads in flight at a time (one CTA per clip: the loop is pure L2 latency otherwise), added
  // in block order
  int b = 0;
  for (; b + 8 <= nblk; b += 8) {
    double2 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __ldg(reinterpret_cast<const double2*>(p + (long long)(b + i) * AW_NMEL * 2));
#pragma unroll
    for (int i = 0; i < 8; ++i) { s1 += v[i].x; s2 += v[i].y; }
  }
  for (; b < nblk; ++b) {
    s1 += p[(long long)b * AW_NMEL * 2];
    s2 += p[(long long)b * AW_NMEL * 2 + 1];
  }
}

// ---- InstanceNorm(128) -> GlobalStandardize -> AvgPool(2,2) -----------------
// GlobalStandardize statistics are taken analytically from the channel
// statistics: after InstanceNorm every channel has mean 0 and second moment
// var/(var+eps), so mean_g = 0 and std_g^2 = T * sum_c var_c/(var_c+eps) / (128 T - 1).
// k_mel_stats reduces the per-block partials ONCE per clip (one CTA per clip, thread = channel);
// k_p0 then only streams.
__global__ void __launch_bounds__(128) k_mel_stats(const double* __restrict__ chan_part, int nblk, int T,
                                                   ChanStats* __restrict__ cs, float* __restrict__ sigma_out) {
  __shared__ double s_red[32];
  const int clip = blockIdx.x, c = threadIdx.x;
  double s1, s2;
  sum_partials(chan_part, clip, nblk, c, s1, s2);
  const double mu = s1 / T;
  double var = s2 / T - mu * mu;
  if (var < 0.0) var = 0.0;
  const double rstd = 1.0 / sqrt(var + AW_IN_EPS);
  const double vr = var / (var + AW_IN_EPS);
  const double tot = block_sum(vr, s_red);
  ChanStats st;
  st.mu = (float)mu; st.rstd = (float)rstd; st.varratio = (float)vr; st.pad = 0.f;
  cs[(long long)clip * AW_NMEL + c] = st;
  if (threadIdx.x == 0) {
    const double n = 128.0 * T;
    sigma_out[clip] = (float)sqrt((double)T * tot / (n - 1.0));
  }
}

#define AW_P0_ROWS 32
template <typename AT>
__global__ void __launch_bounds__(128) k_p0(const float* __restrict__ M, int T, int Tp, int Tp_pad,
                                            const ChanStats* __restrict__ cs,
                                            const float* __restrict__ sigma_in,
                                            AT* __restrict__ P0, int round_tf32) {
  const int clip = blockIdx.y, c = threadIdx.x, j0 = blockIdx.x * AW_P0_ROWS;
  const ChanStats st = cs[(long long)clip * AW_NMEL + c];
  const float fmu = st.mu, fr = st.rstd;
  const float inv = (float)(1.0 / ((double)sigma_in[clip] + 1e-8));
  const float* Mc = M + (long long)clip * T * AW_NMEL + c;
  // 8 pooled rows per batch: 16 independent loads in flight per thread (latency-bound otherwise)
#pragma unroll 1
  for (int jb = j0; jb < min(j0 + AW_P0_ROWS, Tp_pad); jb += 8) {
    float a0[8], a1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int j = jb + i;
      const bool ok = j < Tp;
      a0[i] = ok ? Mc[(long long)(2 * j) * AW_NMEL] : 0.f;
      a1[i] = ok ? Mc[(long long)(2 * j + 1) * AW_NMEL] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int j = jb + i;
      if (j >= Tp_pad) break;
      float p = 0.f;
      if (j < Tp) {
        const float g0 = (a0[i] - fmu) * fr * inv;
        const float g1 = (a1[i] - fmu) * fr * inv;
        p = 0.5f * (g0 + g1);
        if (sizeof(AT) == 4 && round_tf32) p = to_tf32(p);
      }
      act_st(P0 + ((long long)clip * Tp_pad + j) * AW_NMEL + c, p);
    }
  }
}

// ---- InstanceNorm statistics from per-tile partials --------------------------
// part: [clip * tiles + tile][ldp][2] ; stat: [clip][C][2] = (mean, rstd)
// block = 32 channels x 8 tile slices: slice s sums tiles s, s+8, ... and the 8 slice sums are
// combined in fixed order, so long clips (thousands of tiles) are not serialised per channel.
// MODE: 0 forward (mean, rstd), 1 backward (two means), 2 raw float64 sums [clip][C][2] written to
// `raw` (frame-sharded long-form mode: the sums are all-reduced over ranks before k_stat_from_sums)
template <int MODE>
__global__ void __launch_bounds__(256) k_finalize(const float* __restrict__ part, int ldp, int tiles,
                                                  int C, int Tp, float* __restrict__ stat,
                                                  double* __restrict__ raw = nullptr) {
  __shared__ double s_s[8][32][2];
  const int clip = blockIdx.y, cl = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  double s1 = 0.0, s2 = 0.0;
  if (c < C) {
    for (int t = sl; t < tiles; t += 8) {
      const float2 p = *reinterpret_cast<const float2*>(part + (((long long)clip * tiles + t) * ldp + c) * 2);
      s1 += p.x;
      s2 += p.y;
    }
  }
  s_s[sl][cl][0] = s1;
  s_s[sl][cl][1] = s2;
  __syncthreads();
  if (sl != 0 || c >= C) return;
#pragma unroll
  for (int k = 1; k < 8; ++k) { s1 += s_s[k][cl][0]; s2 += s_s[k][cl][1]; }
  if (MODE == 2) {
    raw[((long long)clip * C + c) * 2] = s1;
    raw[((long long)clip * C + c) * 2 + 1] = s2;
  } else if (MODE == 1) {
    // bstat: (mean_j dHhat, mean_j dHhat*Hhat)
    stat[((long long)clip * C + c) * 2] = (float)(s1 / Tp);
    stat[((long long)clip * C + c) * 2 + 1] = (float)(s2 / Tp);
  } else {
    const double mu = s1 / Tp;
    double var = s2 / Tp - mu * mu;
    if (var < 0.0) var = 0.0;
    stat[((long long)clip * C + c) * 2] = (float)mu;
    stat[((long long)clip * C + c) * 2 + 1] = (float)(1.0 / sqrt(var + AW_IN_EPS));
  }
}

// Short clips (a handful of tiles): one thread per channel, no shared memory, C / 256 blocks per clip instead
// of C / 32 -- the slice kernel above spends its time being launched (8 192 blocks of 256 threads for 7 float2
// each at 256 clips x 10 s).  Same float64 summation order (slice sums t = s, s + 8, ..., combined s = 0..7),
// so the statistics are bit-identical to k_finalize's.
template <int MODE>
__global__ void __launch_bounds__(256) k_finalize_small(const float* __restrict__ part, int ldp, int tiles,
                                                        int C, int Tp, float* __restrict__ stat) {
  const int clip = blockIdx.y, c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  const float* p0 = part + (((long long)clip * tiles) * ldp + c) * 2;
  double s1 = 0.0, s2 = 0.0;
  if (tiles <= 8) {
    // one tile per slice: all loads in flight at once, then the same sums in the same (slice) order
    float2 pv[8];
#pragma unroll
    for (int t = 0; t < 8; ++t)
      pv[t] = t < tiles ? __ldg(reinterpret_cast<const float2*>(p0 + (long long)t * ldp * 2)) : make_float2(0.f, 0.f);
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      if (t < tiles) {
        s1 = t == 0 ? (double)pv[t].x : s1 + (double)pv[t].x;
        s2 = t == 0 ? (double)pv[t].y : s2 + (double)pv[t].y;
      }
    }
  } else {
    for (int sl = 0; sl < 8; ++sl) {
      double a1 = 0.0, a2 = 0.0;
      for (int t = sl; t < tiles; t += 8) {
        const float2 p = __ldg(reinterpret_cast<const float2*>(p0 + (long long)t * ldp * 2));
        a1 += p.x;
        a2 += p.y;
      }
      s1 = sl == 0 ? a1 : s1 + a1;
      s2 = sl == 0 ? a2 : s2 + a2;
    }
  }
  if (MODE == 1) {
    stat[((long long)clip * C + c) * 2] = (float)(s1 / Tp);
    stat[((long long)clip * C + c) * 2 + 1] = (float)(s2 / Tp);
  } else {
    const double mu = s1 / Tp;
    double var = s2 / Tp - mu * mu;
    if (var < 0.0) var = 0.0;
    stat[((long long)clip * C + c) * 2] = (float)mu;
    stat[((long long)clip * C + c) * 2 + 1] = (float)(1.0 / sqrt(var + AW_IN_EPS));
  }
}

// statistics from (all-reduced) raw sums; Tp = GLOBAL pooled frame count of the clip
template <bool BWD>
__global__ void __launch_bounds__(256) k_stat_from_sums(const double* __restrict__ raw, int C, int Tp,
                                                        float* __restrict__ stat) {
  const int clip = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double s1 = raw[((long long)clip * C + c) * 2], s2 = raw[((long long)clip * C + c) * 2 + 1];
  if (BWD) {
    stat[((long long)clip * C + c) * 2] = (float)(s1 / Tp);
    stat[((long long)clip * C + c) * 2 + 1] = (float)(s2 / Tp);
  } else {
    const double mu = s1 / Tp;
    double var = s2 / Tp - mu * mu;
    if (var < 0.0) var = 0.0;
    stat[((long long)clip * C + c) * 2] = (float)mu;
    stat[((long long)clip * C + c) * 2 + 1] = (float)(1.0 / sqrt(var + AW_IN_EPS));
  }
}

// ---- row-wise InstanceNorm application, in place --------------------------------
// NORM_FWD: P  = LeakyReLU((H - mean) * rstd)                      (conv1d.py:40-41)
// NORM_BWD: dH = rstd * (dHhat - a1 - Hhat * a2), Hhat recovered from P
// pad rows (j >= Tp) are forced to 0.  One thread owns 4 adjacent channels of one clip for
// AW_NORM_ROWS rows: the per-channel statistics are loaded once into registers and the
// row loop is pure 16-byte streaming with 8 independent loads in flight.
// grid = (Tp_pad / (AW_NORM_ROWS * RL) rounded up, C / (V * 128) rounded up, n_clips), block = 128.
enum { NORM_FWD = 0, NORM_BWD = 1 };
#define AW_NORM_ROWS 32
// 16 bytes per access for every storage type: 4 floats or 8 half / bf16 values
template <typename AT> struct Vec16 { static constexpr int N = 16 / sizeof(AT); };
__device__ __forceinline__ void ld16(const float* p, float (&v)[4]) { act_ld4(p, v); }
__device__ __forceinline__ void st16(float* p, const float (&v)[4]) { act_st4(p, v); }
__device__ __forceinline__ void ld16(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 t = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = __uint_as_float(w[j] << 16);
    v[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
  }
}
__device__ __forceinline__ void st16(__nv_bfloat16* p, const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    w[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ void ld16(const __half* p, float (&v)[8]) {
  const uint4 t = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
    v[2 * j] = f.x; v[2 * j + 1] = f.y;
  }
}
__device__ __forceinline__ void st16(__half* p, const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __half2 h = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
    w[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

template <typename AT, int MODE>
__global__ void __launch_bounds__(128) k_norm_rows(AT* __restrict__ X, const AT* __restrict__ P, int C,
                                                   int Tp, int Tp_pad, const float* __restrict__ stat,
                                                   const float* __restrict__ bstat, int round_tf32) {
  constexpr int V = Vec16<AT>::N;
  const int clip = blockIdx.z;
  // narrow layers (C / V < 128 column groups, e.g. the 64-channel last layer): the block's 128 threads are
  // G column groups x RL row lanes and the block covers AW_NORM_ROWS * RL rows, so every thread still owns
  // AW_NORM_ROWS rows (stride RL) and a warp's access stays contiguous; wide layers: G = 128, RL = 1
  const int G = min(128, C / V), RL = 128 / G;
  const int cgp = threadIdx.x % G, rl = threadIdx.x / G;
  const int c = (blockIdx.y * 128 + cgp) * V;
  if (c >= C) return;
  const int j0 = blockIdx.x * AW_NORM_ROWS * RL + rl;
  float mu[V], rs[V], a1[V], a2[V];
#pragma unroll
  for (int k = 0; k < V; k += 2) {
    const float4 s01 = *reinterpret_cast<const float4*>(stat + ((long long)clip * C + c + k) * 2);
    mu[k] = s01.x; rs[k] = s01.y; mu[k + 1] = s01.z; rs[k + 1] = s01.w;
    if (MODE == NORM_BWD) {
      const float4 b01 = *reinterpret_cast<const float4*>(bstat + ((long long)clip * C + c + k) * 2);
      a1[k] = b01.x; a2[k] = b01.y; a1[k + 1] = b01.z; a2[k + 1] = b01.w;
    }
  }
  AT* x = X + ((long long)clip * Tp_pad + j0) * C + c;
  const AT* p = MODE == NORM_BWD ? P + ((long long)clip * Tp_pad + j0) * C + c : nullptr;
  const long long rstride = (long long)RL * C;           // between two rows of this thread
  constexpr int NB = V == 4 ? 8 : 4;                     // 16-byte loads in flight per tensor
#pragma unroll 1
  for (int r0 = 0; r0 < AW_NORM_ROWS; r0 += NB) {
    if (j0 + r0 * RL >= Tp_pad) break;                   // Tp_pad is a multiple of 128 >= NB * RL rows
    float h[NB][V], a[MODE == NORM_BWD ? NB : 1][V];
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      ld16(x + (r0 + i) * rstride, h[i]);
      if (MODE == NORM_BWD) ld16(p + (r0 + i) * rstride, a[i]);
    }
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      float o[V];
#pragma unroll
      for (int k = 0; k < V; ++k) {
        if (MODE == NORM_FWD) {
          o[k] = leaky((h[i][k] - mu[k]) * rs[k]);
        } else {
          const float av = a[MODE == NORM_BWD ? i : 0][k];
          const float hh = av > 0.f ? av : av * (1.0f / AW_LEAKY);
          o[k] = rs[k] * (h[i][k] - a1[k] - hh * a2[k]);
        }
        if (sizeof(AT) == 4 && round_tf32) o[k] = to_tf32(o[k]);
        if (j0 + (r0 + i) * RL >= Tp) o[k] = 0.f;
      }
      st16(x + (r0 + i) * rstride, o);
    }
  }
}

// ---- BRH head + loss + seed of the backward pass -------------------------------
// P4: [rows][64] (40 live channels) = LeakyReLU(Hhat).  Three kernels so that a long clip is
// not serialised on one CTA:
//   k_head_partial (grid = row tiles x clips): per 128-row tile and channel,
//        S_pos = sum_{P>0} P,  S_neg = sum_{P<=0} P / 0.2 (= Hhat),  n_pos
//   k_head_final   (grid = clips): z = (S_pos + 0.2 S_neg)/T', v = tanh(z_even - z_odd), loss,
//        best / improved, dz, and the InstanceNorm-adjoint means -- both follow from the SAME
//        partial sums because dHhat = LeakyReLU'(P) dz is constant per channel and sign:
//        a1 = dz (n_pos + 0.2 n_neg)/T',  a2 = mean(dHhat Hhat) = dz z
//   k_head_seed    (grid = row tiles x clips): dH4 = gscale rstd (dHhat - a1 - Hhat a2)
template <typename AT>
struct HeadArgs {
  const AT* P4; int Tp, Tp_pad;
  int Tp_glob;               // pooled frames of the WHOLE clip (= Tp unless the clip is frame-sharded)
  const float* stat4;        // [clip][64][2]
  const float* pattern;      // [clip][20] (+-1) or null (detect only)
  float* values;             // [clip][20]
  float* losses;             // [iters][n_clips] or null
  float* best;               // [clip]
  int* improved;             // [clip]
  AT* dH4;                   // [rows][64] or null
  const int* it_ptr; int n_clips;
  int round_tf32;
  float gscale;              // 16-bit modes: target magnitude of the seeded gradient (0.5), else 0
  float* gsc;                // [clip] out: power-of-two loss scale chosen per clip and iteration
  double* hpart;             // [clip][tiles][64][3] partial sums
  float* hcoef;              // [clip][64][4] = (dz, a1, a2, rstd)
};

template <typename AT>
__global__ void __launch_bounds__(256) k_head_partial(HeadArgs<AT> a) {
  __shared__ double s_acc[4][64][3];
  const int tile = blockIdx.x, clip = blockIdx.y, tid = threadIdx.x;
  const int c = tid & 63, g = tid >> 6;
  const AT* P = a.P4 + ((long long)clip * a.Tp_pad + tile * 128) * 64;
  const int rows = min(128, a.Tp - tile * 128);
  double sp = 0.0, sn = 0.0, np_ = 0.0;
#pragma unroll 1
  for (int jb = g; jb < rows; jb += 32) {                  // 8 independent loads per batch
    float p8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) p8[i] = jb + 4 * i < rows ? act_ld(P + (long long)(jb + 4 * i) * 64 + c) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (jb + 4 * i >= rows) break;
      const float p = p8[i];
      if (p > 0.f) { sp += p; np_ += 1.0; } else { sn += (double)(p * (1.0f / AW_LEAKY)); }
    }
  }
  s_acc[g][c][0] = sp; s_acc[g][c][1] = sn; s_acc[g][c][2] = np_;
  __syncthreads();
  if (tid < 64) {
    double* o = a.hpart + (((long long)clip * gridDim.x + tile) * 64 + tid) * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k] = s_acc[0][tid][k] + s_acc[1][tid][k] + s_acc[2][tid][k] + s_acc[3][tid][k];
  }
}

template <typename AT>
__global__ void __launch_bounds__(64) k_head_final(HeadArgs<AT> a, int tiles) {
  __shared__ float s_z[64], s_dz[64];
  const int clip = blockIdx.x, c = threadIdx.x;
  double sp = 0.0, sn = 0.0, np_ = 0.0;
  for (int t0 = 0; t0 < tiles; t0 += 8) {                   // eight tiles' loads in flight, added in tile order
    double o3[8][3];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const double* o = a.hpart + (((long long)clip * tiles + min(t0 + i, tiles - 1)) * 64 + c) * 3;
      o3[i][0] = o[0]; o3[i][1] = o[1]; o3[i][2] = o[2];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (t0 + i < tiles) { sp += o3[i][0]; sn += o3[i][1]; np_ += o3[i][2]; }
  }
  const float z = (float)((sp + (double)AW_LEAKY * sn) / a.Tp_glob);
  s_z[c] = z;
  s_dz[c] = 0.f;
  __syncthreads();
  if (c < 32) {
    float v = 0.f, p = 0.f;
    if (c < AW_NBITS) {
      v = tanhf(s_z[2 * c] - s_z[2 * c + 1]);
      a.values[(long long)clip * AW_NBITS + c] = v;
      if (a.pattern) p = a.pattern[(long long)clip * AW_NBITS + c];
    }
    if (a.pattern) {
      const float se = c < AW_NBITS ? (v - p) * (v - p) : 0.f;
      const float ab = c < AW_NBITS ? fabsf(v) : 0.f;
      const float mse = warp_sum(se) / AW_NBITS, pen = 0.1f * (warp_sum(ab) / AW_NBITS);
      const float loss = mse - pen;
      if (c == 0) {
        const int it = a.it_ptr ? *a.it_ptr : 0;
        if (a.losses) a.losses[(long long)it * a.n_clips + clip] = loss;
        const float b = a.best[clip];
        const int imp = loss < b;
        a.improved[clip] = imp;
        if (imp) a.best[clip] = loss;
      }
      if (c < AW_NBITS) {
        const float sg = v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f);
        const float dv = 2.f * (v - p) / AW_NBITS - 0.1f * sg / AW_NBITS;
        const float dd = dv * (1.f - v * v);
        s_dz[2 * c] = dd / a.Tp_glob;
        s_dz[2 * c + 1] = -dd / a.Tp_glob;
      }
    }
  }
  if (!a.pattern || !a.dH4) return;
  __syncthreads();
  if (c < 32) {
    // per-clip, per-iteration power-of-two loss scale (fp16 gradients): keeps the seeded gradient at
    // a fixed magnitude for any clip length and however far tanh has saturated; a power of two
    // changes no mantissa, and it is removed exactly where dP0 is consumed
    float mx = fmaxf(fabsf(s_dz[c]), fabsf(s_dz[c + 32]));
    mx = warp_max(mx);
    if (c == 0) {
      float gs = 1.0f;
      if (a.gscale > 0.f && mx > 0.f) gs = exp2f(fminf(fmaxf(rintf(log2f(a.gscale / mx)), 0.f), 60.f));
      a.gsc[clip] = gs;
    }
  }
  const float dz = s_dz[c];
  const double nneg = (double)a.Tp_glob - np_;
  const float a1 = (float)((double)dz * (np_ + (double)AW_LEAKY * nneg) / a.Tp_glob);
  const float a2 = dz * z;
  *reinterpret_cast<float4*>(a.hcoef + ((long long)clip * 64 + c) * 4) =
      make_float4(dz, a1, a2, a.stat4[((long long)clip * 64 + c) * 2 + 1]);
}

template <typename AT>
__global__ void __launch_bounds__(256) k_head_seed(HeadArgs<AT> a) {
  const int tile = blockIdx.x, clip = blockIdx.y, tid = threadIdx.x;
  const int c = tid & 63, g = tid >> 6;
  const float4 k = *reinterpret_cast<const float4*>(a.hcoef + ((long long)clip * 64 + c) * 4);
  const float dz = k.x, a1 = k.y, a2 = k.z, rstd = k.w;
  const float gscale = a.gsc[clip];
  const AT* P = a.P4 + ((long long)clip * a.Tp_pad + tile * 128) * 64;
  AT* D = a.dH4 + ((long long)clip * a.Tp_pad + tile * 128) * 64;
#pragma unroll 1
  for (int jb = g; jb < 128; jb += 32) {                   // 8 independent loads per batch
    float p8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) p8[i] = act_ld(P + (long long)(jb + 4 * i) * 64 + c);   // pad rows exist (zeros)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int j = jb + 4 * i;
      float o = 0.f;
      if (tile * 128 + j < a.Tp && c < 2 * AW_NBITS) {
        const float p = p8[i];
        const bool pos = p > 0.f;
        const float dh = pos ? dz : AW_LEAKY * dz;
        o = gscale * (rstd * (dh - a1 - (pos ? p : p * (1.0f / AW_LEAKY)) * a2));
        if (sizeof(AT) == 4 && a.round_tf32) o = to_tf32(o);
      }
      act_st(D + (long long)j * 64 + c, o);
    }
  }
}

// ---- adjoint of pool / GlobalStandardize / InstanceNorm(128) / mel -------------
// pass 1: S1_c = sum_t dG, S2_c = sum_t dG * Mhat   (dG[t] = dP0[t/2]/2, 0 for the odd tail)
#define AW_P0B_FRAMES 64
__global__ void __launch_bounds__(128) k_p0_bwd_reduce(const float* __restrict__ dP0,
                                                       const float* __restrict__ M, int T, int Tp,
                                                       int Tp_pad, const ChanStats* __restrict__ cs,
                                                       double* __restrict__ bpart,
                                                       const float* __restrict__ gsc) {
  const int clip = blockIdx.y, c = threadIdx.x, t0 = blockIdx.x * AW_P0B_FRAMES;
  const float ginv = 1.0f / gsc[clip];                     // exact: the scale is a power of two
  const ChanStats st = cs[(long long)clip * AW_NMEL + c];
  double s1 = 0.0, s2 = 0.0;
  const int t1 = min(t0 + AW_P0B_FRAMES, 2 * Tp);
  // ncu (profiles/r2_ncu_summary.md, front end): this kernel was ISSUE-bound (81 % issue-active, 37 instructions per
  // element), not HBM-bound -- so: one base pointer per tensor and immediate offsets, each pooled row of dP0 loaded
  // once for its two frames, predicates only in the clip's last block.  Same sums in the same order.
  const float* dp = dP0 + ((long long)clip * Tp_pad + (t0 >> 1)) * AW_NMEL + c;      // t0 is even
  const float* mp = M + ((long long)clip * T + t0) * AW_NMEL + c;
  const float hg = 0.5f * ginv;
#pragma unroll 1
  for (int tb = t0; tb < t1; tb += 8, dp += 4 * AW_NMEL, mp += 8 * AW_NMEL) {
    float d4[4], m8[8];
    if (tb + 8 <= t1) {
#pragma unroll
      for (int i = 0; i < 4; ++i) d4[i] = dp[i * AW_NMEL];
#pragma unroll
      for (int i = 0; i < 8; ++i) m8[i] = mp[i * AW_NMEL];
    } else {                                                      // the clip's last block (2 Tp is even: whole pairs)
#pragma unroll
      for (int i = 0; i < 4; ++i) d4[i] = tb + 2 * i < t1 ? dp[i * AW_NMEL] : 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) m8[i] = tb + i < t1 ? mp[i * AW_NMEL] : st.mu;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float dg = hg * d4[i >> 1];                           // masked rows: dg = 0 and mh = 0, as before
      const float mh = (m8[i] - st.mu) * st.rstd;
      s1 += dg;
      s2 += (double)dg * mh;
    }
  }
  double* p = bpart + (((long long)clip * gridDim.x + blockIdx.x) * AW_NMEL + c) * 2;
  p[0] = s1;
  p[1] = s2;
}

// pass 1b: per clip, once: the scalars and per-channel coefficients of the three adjoints
struct P0BwdCoef { float A1, A2; };
struct P0BwdScal { float alpha, beta, meanG, pad; };
__global__ void __launch_bounds__(128) k_p0_bwd_coef(const double* __restrict__ bpart, int nblk, int T,
                                                     const ChanStats* __restrict__ cs,
                                                     const float* __restrict__ sigma_in,
                                                     P0BwdCoef* __restrict__ coef,
                                                     P0BwdScal* __restrict__ scal) {
  __shared__ double s_red[32];
  __shared__ float s_ab[3];
  const int clip = blockIdx.x, c = threadIdx.x;
  double S1, S2;
  sum_partials(bpart, clip, nblk, c, S1, S2);
  const double tS1 = block_sum(S1, s_red);
  __syncthreads();
  const double tS2 = block_sum(S2, s_red);
  if (threadIdx.x == 0) {
    const double n = 128.0 * T, sg = sigma_in[clip];
    s_ab[0] = (float)(1.0 / (sg + 1e-8));                                      // alpha
    s_ab[1] = (float)(tS2 / ((n - 1.0) * sg * (sg + 1e-8) * (sg + 1e-8)));      // beta
    s_ab[2] = (float)(tS1 / n);                                                 // mean dG
    P0BwdScal o;
    o.alpha = s_ab[0]; o.beta = s_ab[1]; o.meanG = s_ab[2]; o.pad = 0.f;
    scal[clip] = o;
  }
  __syncthreads();
  const float alpha = s_ab[0], beta = s_ab[1], meanG = s_ab[2];
  const ChanStats st = cs[(long long)clip * AW_NMEL + c];
  P0BwdCoef k;
  k.A1 = alpha * ((float)(S1 / T) - meanG);
  k.A2 = alpha * (float)(S2 / T) - beta * st.varratio;
  coef[(long long)clip * AW_NMEL + c] = k;
}

// pass 2: dM, then dA~[t][b] = sum_c mel[c][b] dM[t][c]
#define AW_P0A_FRAMES 16
__global__ void __launch_bounds__(128) k_p0_bwd_apply(const float* __restrict__ dP0,
                                                      const float* __restrict__ M, int T, int Tp,
                                                      int Tp_pad, const ChanStats* __restrict__ cs,
                                                      const P0BwdCoef* __restrict__ coef,
                                                      const P0BwdScal* __restrict__ scal,
                                                      SparseMel sm,
                                                      int nb, float* __restrict__ dA,
                                                      const float* __restrict__ mag_un,
                                                      double* __restrict__ s2_part,
                                                      const float* __restrict__ gsc) {
  __shared__ double s_red[32];
  __shared__ float s_dm[AW_P0A_FRAMES][AW_NMEL];
  const int clip = blockIdx.y, c = threadIdx.x, t0 = blockIdx.x * AW_P0A_FRAMES;
  const P0BwdScal sc = scal[clip];
  const float alpha = sc.alpha, beta = sc.beta, meanG = sc.meanG;
  const float ginv = 1.0f / gsc[clip];
  const ChanStats st = cs[(long long)clip * AW_NMEL + c];
  const P0BwdCoef k = coef[(long long)clip * AW_NMEL + c];
  const float A1 = k.A1, A2 = k.A2;
  const int nf = min(AW_P0A_FRAMES, T - t0);
  {
    float d16[AW_P0A_FRAMES], m16[AW_P0A_FRAMES];          // all loads of the tile in flight together
#pragma unroll
    for (int f = 0; f < AW_P0A_FRAMES; ++f) {
      const int t = t0 + f;
      d16[f] = (f < nf && t < 2 * Tp) ? dP0[((long long)clip * Tp_pad + (t >> 1)) * AW_NMEL + c] : 0.f;
      m16[f] = f < nf ? M[((long long)clip * T + t) * AW_NMEL + c] : st.mu;
    }
#pragma unroll
    for (int f = 0; f < AW_P0A_FRAMES; ++f) {
      const float dg = (0.5f * ginv) * d16[f];
      const float mh = (m16[f] - st.mu) * st.rstd;
      const float dmh = alpha * (dg - meanG) - beta * mh;
      s_dm[f][c] = f < nf ? st.rstd * (dmh - A1 - mh * A2) : 0.f;
    }
  }
  __syncthreads();
  // one thread per band bin: its (weight, channel) taps are fetched once and applied to all frames
  double s2 = 0.0;
  for (int b = threadIdx.x; b < nb; b += 128) {
    const int e0 = sm.colptr[b], e1 = sm.colptr[b + 1];
    float acc[AW_P0A_FRAMES];
#pragma unroll
    for (int f = 0; f < AW_P0A_FRAMES; ++f) acc[f] = 0.f;
    for (int e = e0; e < e1; ++e) {
      const float w = sm.valT[e];
      const int r = sm.row[e];
#pragma unroll
      for (int f = 0; f < AW_P0A_FRAMES; ++f) acc[f] = fmaf(w, s_dm[f][r], acc[f]);
    }
#pragma unroll
    for (int f = 0; f < AW_P0A_FRAMES; ++f) {
      if (f < nf) {
        const long long o = ((long long)clip * T + t0 + f) * nb + b;
        dA[o] = acc[f];
        if (mag_un) s2 += (double)(acc[f] * mag_un[o]);
      }
    }
  }
  if (mag_un) {
    // Euler: sum_n dy2[n] y2[n] = sum_{t,b} dA~ A~ (|STFT| is 1-homogeneous); the factor
    // 1/(d1 d2) that turns the un-normalised magnitudes into A~ is applied by k_clip_scalars
    __syncthreads();
    s2 = block_sum(s2, s_red);
    if (threadIdx.x == 0) s2_part[(long long)clip * gridDim.x + blockIdx.x] = s2;
  }
}

// ---- bit decision + BER counters (utils/watermark/decoder.py:51,63; metrics/audio.py:15)
// counters: [0] bit errors, [1] bits compared, [2] clips
__global__ void __launch_bounds__(128) k_decide_count(const float* __restrict__ values,
                                                      const int* __restrict__ ref_bits,
                                                      float thr, int n_clips,
                                                      int* __restrict__ bits_out,
                                                      int* __restrict__ err_per_clip,
                                                      unsigned long long* __restrict__ counters) {
  const int clip = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (clip >= n_clips) return;
  int bit = 0, err = 0;
  if (lane < AW_NBITS) {
    bit = values[(long long)clip * AW_NBITS + lane] > thr ? 1 : 0;
    if (bits_out) bits_out[(long long)clip * AW_NBITS + lane] = bit;
    if (ref_bits) err = bit != ref_bits[(long long)clip * AW_NBITS + lane];
  }
  const unsigned m = __ballot_sync(0xffffffffu, err);
  if (lane == 0 && ref_bits) {
    const int e = __popc(m);
    if (err_per_clip) err_per_clip[clip] = e;
    if (counters) {
      atomicAdd(counters + 0, (unsigned long long)e);
      atomicAdd(counters + 1, (unsigned long long)AW_NBITS);
      atomicAdd(counters + 2, 1ull);
    }
  }
}

// ---- SNR (metrics/audio.py:68-89): per clip 10 log10(sum o^2 / sum (o-t)^2) -------
__global__ void __launch_bounds__(256) k_snr_partial(const float* __restrict__ out, long long so,
                                                     const float* __restrict__ tgt, long long st_,
                                                     int n, double* __restrict__ acc) {
  __shared__ double s_red[32];
  const int clip = blockIdx.y;
  double p = 0.0, e = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float o = out[(long long)clip * so + i], t = tgt[(long long)clip * st_ + i];
    const float d = o - t;
    p += (double)o * o;
    e += (double)d * d;
  }
  p = block_sum(p, s_red);
  __syncthreads();
  e = block_sum(e, s_red);
  if (threadIdx.x == 0) {
    atomicAdd(acc + 2 * clip, p);
    atomicAdd(acc + 2 * clip + 1, e);
  }
}

__global__ void k_snr_final(const double* __restrict__ acc, int n_clips, double* __restrict__ snr,
                            double* __restrict__ snr_sum) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_clips) return;
  const double p = acc[2 * i], e = acc[2 * i + 1];
  const double s = e == 0.0 ? INFINITY : 10.0 * log10(p / e);
  snr[i] = s;
  if (snr_sum && e != 0.0) atomicAdd(snr_sum, s);
}

}  // namespace aw
