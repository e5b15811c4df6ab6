// Tensor-core form of the embedding loop's band-limited transforms (reference
// embedding/multibit_embedder.py:49-67: STFTAssembler -> ISTFT -> normalise x2 -> STFT -> |.|).
//
// Only B = 81 of 513 bins exist at 44.1 kHz, so restricted to the band the transforms are small dense
// contractions, and because the out-of-band part of the waveform never changes (y = y_band(c) + y_oob)
// everything that varies is linear in X = c u (2B real numbers per frame):
//
//   peak GEMM   y_band[h][j] = sum_{r<4}  X[h-r] . G_r[.][j]          (hop h, sample j < 256; K = 4 P)
//               epilogue: + y_oob, max |y| with index and sign -> the peak normalisers; y is never stored
//   comp GEMM   S_band[t]    = sum_{|d|<=3} K_d X[t+d]                  (K = 7 P, N = P)
//               epilogue: + S_oob (constant, fp32), |S| and S/|S|
//   comp^T GEMM dX[t']       = sum_{|d|<=3} K_d^T dS[t'-d]              (adjoint; fp32 out)
//
// with P = 192 (2B = 162 padded), K_d = A_w E S_w shifted by d hops: analysis basis x 1/envelope x
// synthesis basis, built once on the host in float64 (spectc_build).  The A operands are TOEPLITZ views
// of the frame-row arrays X / dS ([T + 6][P] fp16 per clip, three zero rows at either end), expressed as
// a row offset per k-block into the plain 2-D TMA map of the frame rows -- nothing is gathered or copied.  All three GEMMs run on k_gemm_tc (tcgen05,
// kind::f16, fp32 accumulation in TMEM).
//
// What is NOT Toeplitz: the three frames at either end of a clip (edge envelope, reflect padding).  Those
// six frames are recomputed exactly by k_spec in edge mode (forward: overwrite |S|, q; backward: the
// adjoint of those rows, added to the gradient), and the peak-normaliser sub-gradient (one sample) is
// added analytically in k_tc_update.  Operands are fp16 (X is rounded to 11 bits -- the same rounding the
// detector's fp16 activations already apply to everything downstream); this path is used only when the
// loop GEMMs are fp16, the final synthesis and every detect stay on the fp32 FFT kernels.
#pragma once
#include <cuda_fp16.h>
#include <math.h>

#include <vector>

#include "common.cuh"
#include "fft.cuh"
#include "spec.cuh"

namespace aw {

#define AW_TC_P 192            // padded 2 * nbins (frame-row length of X / dS / S)

struct SpecTcMats {
  std::vector<__half> peakB;   // [256][4 P]   G (x 2^10)
  std::vector<__half> compB;   // [P][7 P]     K_d
  std::vector<__half> compBT;  // [P][7 P]     K_d^T
  std::vector<float> fix;      // [768]: [0] 2^-10, [256+j] hop-2 scale, [512+j] hop-T scale
};

// float64 construction of the three B operands from the analysis / synthesis window
static void spectc_build(const float* window, int bin0, int nb, SpecTcMats& m) {
  const int P = AW_TC_P, N = AW_NFFT, W2 = 2 * nb;
  std::vector<double> w(N), env(256), envL(256), envR(256);
  for (int n = 0; n < N; ++n) w[n] = window[n];
  for (int j = 0; j < 256; ++j) {
    env[j] = envL[j] = envR[j] = 0.0;
    for (int r = 0; r < 4; ++r) {
      const double s = w[256 * r + j] * w[256 * r + j];
      env[j] += s;
      if (r <= 2) envL[j] += s;
      if (r >= 1) envR[j] += s;
    }
  }
  // synthesis basis C[n][i] (one frame's waveform per unit of X component i) and analysis basis A[o][n]
  std::vector<double> C((size_t)N * W2), A((size_t)W2 * N);
  for (int b = 0; b < nb; ++b)
    for (int n = 0; n < N; ++n) {
      const int kn = (int)(((long long)(bin0 + b) * n) % N);
      const double th = 2.0 * M_PI * kn / N, cs = cos(th), sn = sin(th);
      C[(size_t)n * W2 + 2 * b] = (2.0 / N) * w[n] * cs;
      C[(size_t)n * W2 + 2 * b + 1] = -(2.0 / N) * w[n] * sn;
      A[(size_t)(2 * b) * N + n] = w[n] * cs;
      A[(size_t)(2 * b + 1) * N + n] = -w[n] * sn;
    }
  m.peakB.assign((size_t)256 * 4 * P, __float2half(0.f));
  for (int j = 0; j < 256; ++j)
    for (int rp = 0; rp < 4; ++rp)
      for (int i = 0; i < W2; ++i)
        m.peakB[(size_t)j * 4 * P + rp * P + i] =
            __float2half((float)(1024.0 * C[(size_t)(256 * (3 - rp) + j) * W2 + i] / env[j]));
  m.fix.assign(768, 0.f);
  m.fix[0] = 1.0f / 1024.0f;
  for (int j = 0; j < 256; ++j) {
    m.fix[256 + j] = (float)(env[j] / envL[j] / 1024.0);
    m.fix[512 + j] = (float)(env[j] / envR[j] / 1024.0);
  }
  m.compB.assign((size_t)P * 7 * P, __float2half(0.f));
  m.compBT.assign((size_t)P * 7 * P, __float2half(0.f));
  std::vector<double> AE((size_t)W2 * N);           // A[o][n] / env[n mod 256]
  for (int o = 0; o < W2; ++o)
    for (int n = 0; n < N; ++n) AE[(size_t)o * N + n] = A[(size_t)o * N + n] / env[n & 255];
  std::vector<double> Kd((size_t)W2 * W2);
  for (int d = -3; d <= 3; ++d) {
    const int n_lo = d > 0 ? 256 * d : 0, n_hi = d < 0 ? N + 256 * d : N;      // 0 <= n - 256 d < N
    for (int o = 0; o < W2; ++o) {
      double* row = &Kd[(size_t)o * W2];
      for (int i = 0; i < W2; ++i) row[i] = 0.0;
      for (int n = n_lo; n < n_hi; ++n) {
        const double a = AE[(size_t)o * N + n];
        const double* c = &C[(size_t)(n - 256 * d) * W2];
        for (int i = 0; i < W2; ++i) row[i] += a * c[i];
      }
    }
    for (int o = 0; o < W2; ++o)
      for (int i = 0; i < W2; ++i) {
        const __half v = __float2half((float)Kd[(size_t)o * W2 + i]);
        m.compB[(size_t)o * 7 * P + (d + 3) * P + i] = v;        // S[t] += K_d X[t + d]
        m.compBT[(size_t)i * 7 * P + (3 - d) * P + o] = v;       // dX[t'] += K_d^T dS[t' - d]
      }
  }
}

// ---- frame-row arrays ---------------------------------------------------------------------------------
// X rows: [clip][T + 6][P] fp16, row t + 3 = (Re, Im) of c u interleaved per bin; other rows / columns 0.
#define AW_TC_FR 16            // frames per block of the element-wise kernels (16 x 81 elements, 256 threads)
__global__ void __launch_bounds__(256) k_tc_xprep(const float* __restrict__ c, const float2* __restrict__ u, int T,
                                                  int nb, __half* __restrict__ X) {
  const int clip = blockIdx.y, t0 = blockIdx.x * AW_TC_FR;
  const int nf = min(AW_TC_FR, T - t0);
  const long long src = ((long long)clip * T + t0) * nb;            // frames t0.. are contiguous in [T][nb]
  for (int e = threadIdx.x; e < nf * nb; e += blockDim.x) {
    const int f = e / nb, b = e - f * nb;
    const float cv = __ldg(c + src + e);
    const float2 uv = __ldg(u + src + e);
    reinterpret_cast<__half2*>(X + ((long long)clip * (T + 6) + t0 + f + 3) * AW_TC_P)[b] =
        __floats2half2_rn(cv * uv.x, cv * uv.y);
  }
}

// per-clip power-of-two scale that brings the largest |dA| of the clip to ~2^9 (fp16 normal range for
// everything within 2^-23 of it, 2^7 of headroom); dmax holds the float bits of max |dA| (atomicMax on
// non-negative floats) in TWO slots [2][n_clips]: iteration `it` scales by slot it & 1, which iteration
// it - 1 accumulated while it wrote its own dS (the first iteration fills slot 0 with k_tc_absmax), and
// accumulates into slot (it + 1) & 1, which k_clip_scalars has just cleared.  |dA| drifts slowly; should
// it ever jump by more than 2^7 between two iterations the overflow shows up as a non-finite gradient,
// the update is skipped and the clip flagged (aw_embed_status).
__device__ __forceinline__ float tc_grad_scale(unsigned dmax_bits) {
  const float mx = __uint_as_float(dmax_bits);
  if (!(mx > 0.f) || !(mx < INFINITY)) return 1.0f;
  return exp2f(fminf(fmaxf(rintf(9.0f - log2f(mx)), -60.f), 100.f));
}

// dS rows: [clip][T + 6][P] fp16, row t + 3 = scale * dA q; the three frames at either end of the clip are
// written as 0 (their adjoint is evaluated exactly by the edge kernel)
__global__ void __launch_bounds__(256) k_tc_absmax(const float* __restrict__ dA, long long per_clip,
                                                   unsigned* __restrict__ dmax) {
  const int clip = blockIdx.y;
  const float* p = dA + (long long)clip * per_clip;
  float mx = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < per_clip; i += (long long)gridDim.x * blockDim.x)
    mx = fmaxf(mx, fabsf(p[i]));
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0 && mx > 0.f && mx < INFINITY) atomicMax(dmax + clip, __float_as_uint(mx));
}

__global__ void __launch_bounds__(256) k_tc_dsprep(const float* __restrict__ dA, const float2* __restrict__ q, int T,
                                                   int nb, unsigned* __restrict__ dmax2, const int* __restrict__ it_ptr,
                                                   int n_clips, __half* __restrict__ dS) {
  __shared__ float s_mx[8];
  const int clip = blockIdx.y, t0 = blockIdx.x * AW_TC_FR;
  const int nf = min(AW_TC_FR, T - t0);
  const long long src = ((long long)clip * T + t0) * nb;
  const int slot = *it_ptr & 1;
  const float s = tc_grad_scale(dmax2[(size_t)slot * n_clips + clip]);
  float mx = 0.f;
  const unsigned long long nb_magic = 0xFFFFFFFFull / (unsigned)nb + 1ull;   // e / nb == (e * magic) >> 32 for e, nb < 2^16
  // a block's AW_TC_FR x nb elements (nb <= 96) are at most U per thread: all loads first, then the stores
  constexpr int U = (AW_TC_FR * 96 + 255) / 256;
  float a0[U];
  float2 qv[U];
#pragma unroll
  for (int k = 0; k < U; ++k) {
    const int e = threadIdx.x + k * 256;
    const bool on = e < nf * nb;
    a0[k] = on ? __ldg(dA + src + e) : 0.f;
    qv[k] = on ? __ldg(q + src + e) : make_float2(0.f, 0.f);
  }
#pragma unroll
  for (int k = 0; k < U; ++k) {
    const int e = threadIdx.x + k * 256;
    if (e >= nf * nb) break;
    const int f = (int)(((unsigned long long)(unsigned)e * nb_magic) >> 32), b = e - f * nb, t = t0 + f;   // e / nb
    mx = fmaxf(mx, fabsf(a0[k]));
    float2 v = make_float2(0.f, 0.f);
    if (t >= 3 && t < T - 3) {
      const float g = a0[k] * s;
      v = make_float2(g * qv[k].x, g * qv[k].y);
    }
    reinterpret_cast<__half2*>(dS + ((long long)clip * (T + 6) + t + 3) * AW_TC_P)[b] = __floats2half2_rn(v.x, v.y);
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) s_mx[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 8; ++w) mx = fmaxf(mx, s_mx[w]);
    if (mx > 0.f && mx < INFINITY) atomicMax(dmax2 + (size_t)(slot ^ 1) * n_clips + clip, __float_as_uint(mx));
  }
}

// ---- NAdam update from the GEMM's gradient ------------------------------------------------------------
struct TcUpdateArgs {
  int T, nb, rpc;
  const float* dX;             // [rows][P] fp32: scale * K^T dS (interleaved Re, Im)
  const unsigned* dmax;        // [2][n_clips]: this iteration's scale sits in slot it & 1
  int n_clips;
  const ClipScal* scal;        // [clip] inv, corr, nstar
  const float* g_edge;         // [clip][12][nb]: exact adjoint of the six edge rows, frames 0..5 and T-6..T-1
  const float2* u;
  float* c; float* m; float* v; float* cbest;
  const float* c0;
  const int* improved;
  int* nonfinite;
  const NadamStep* steps;
  const int* it_ptr;
  float tol_ratio;
  const float* window;         // [1024]
  const float* env256;         // [512]
  int bin0;
  __half* X;                   // next iteration's frame rows
};

__device__ __forceinline__ void tc_nadam(float g, float& m1, float& v1, float& c1, float c0, const NadamStep& st,
                                         float tol_ratio) {
  // NAdam (torch/optim/nadam.py), clamp (:116-117): same arithmetic as k_spec<BWD>
  m1 = __fadd_rn(m1, __fmul_rn(0.1f, __fsub_rn(g, m1)));
  v1 = __fmul_rn(v1, 0.999f);
  v1 = __fadd_rn(v1, __fmul_rn(__fmul_rn(0.001f, g), g));
  float sq, rden;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(__fmul_rn(v1, st.inv_bc2)));
  const float den = __fadd_rn(sq, 1e-8f);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rden) : "f"(den));
  c1 = __fadd_rn(c1, __fmul_rn(__fmul_rn(st.a_g, g), rden));
  c1 = __fadd_rn(c1, __fmul_rn(__fmul_rn(st.a_m, m1), rden));
  const float dl = __fmul_rn(c0, tol_ratio);
  const float lo = fmaxf(0.f, __fsub_rn(c0, dl)), hi = __fadd_rn(c0, dl);
  c1 = fminf(fmaxf(c1, lo), hi);
}

// One thread = one bin of one frame; a block = AW_TC_FR consecutive frames of a clip (contiguous in the
// [T][nb] state arrays).  All loads of an element are issued before its first store.
__global__ void __launch_bounds__(256) k_tc_update(TcUpdateArgs a) {
  const int clip = blockIdx.y, t0 = blockIdx.x * AW_TC_FR, T = a.T, nb = a.nb;
  const int nf = min(AW_TC_FR, T - t0);
  const int it = *a.it_ptr;
  const NadamStep st = a.steps[it];
  const ClipScal cs = a.scal[clip];
  const float gs = cs.inv / tc_grad_scale(a.dmax[(size_t)(it & 1) * a.n_clips + clip]);
  const bool improved = a.improved[clip] != 0;
  const int mstar = cs.nstar + AW_HALF;
  const long long o0 = ((long long)clip * T + t0) * nb;
  const unsigned long long nb_magic = 0xFFFFFFFFull / (unsigned)nb + 1ull;   // (e * magic) >> 32 == e / nb for e, nb < 2^16
  constexpr int U = 2;                                       // elements in flight per thread
  for (int e0 = threadIdx.x; e0 < nf * nb; e0 += U * blockDim.x) {
    float2 uv[U], d2[U];
    float m1[U], v1[U], c1[U], c0[U], ge[U];
    int tt[U], bb[U];
    bool on[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int e = e0 + k * blockDim.x;
      on[k] = e < nf * nb;
      const int ec = on[k] ? e : e0;
      const int f = (int)(((unsigned long long)(unsigned)ec * nb_magic) >> 32);   // ec / nb without the division sequence
      bb[k] = ec - f * nb;
      tt[k] = t0 + f;
      const long long o = o0 + ec;
      uv[k] = __ldg(a.u + o);
      d2[k] = __ldg(reinterpret_cast<const float2*>(a.dX + ((long long)clip * a.rpc + tt[k]) * AW_TC_P + 2 * bb[k]));
      m1[k] = a.m[o]; v1[k] = a.v[o]; c1[k] = a.c[o];
      c0[k] = __ldg(a.c0 + o);
      const int t = tt[k];
      const int er = t < 6 ? t : (t >= T - 6 ? 6 + (t - (T - 6)) : -1);      // row of g_edge, or -1
      ge[k] = er >= 0 ? __ldg(a.g_edge + ((long long)clip * 12 + er) * nb + bb[k]) : 0.f;
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      if (!on[k]) continue;
      const long long o = o0 + e0 + k * blockDim.x;
      float g = gs * (d2[k].x * uv[k].x + d2[k].y * uv[k].y) + ge[k];
      // peak-normaliser sub-gradient (waveform.py:19 twice): dy[n*] -= corr reaches the (at most four) frames
      // that cover sample n*; through the iSTFT adjoint it is one windowed complex exponential per frame
      const int nn = mstar - AW_HOP * tt[k];
      if (cs.corr != 0.f && nn >= 0 && nn < AW_NFFT && cs.nstar >= 0) {
        const float cw = (2.0f / AW_NFFT) * a.window[nn] * (-cs.corr * ola_inv_envelope(mstar, T, a.window, a.env256));
        float sn, cn;
        sincospif((float)(((a.bin0 + bb[k]) * nn) & (AW_NFFT - 1)) * (2.0f / AW_NFFT), &sn, &cn);
        g += cw * (cn * uv[k].x - sn * uv[k].y);
      }
      if ((__float_as_uint(g) & 0x7f800000u) == 0x7f800000u) {
        if (a.nonfinite) a.nonfinite[clip] = 1;
      } else {
        tc_nadam(g, m1[k], v1[k], c1[k], c0[k], st, a.tol_ratio);
        a.m[o] = m1[k];
        a.v[o] = v1[k];
        a.c[o] = c1[k];
        if (improved) a.cbest[o] = c1[k];                  // best (:120-122)
      }
      reinterpret_cast<__half2*>(a.X + ((long long)clip * a.rpc + tt[k] + 3) * AW_TC_P)[bb[k]] =
          __floats2half2_rn(c1[k] * uv[k].x, c1[k] * uv[k].y);
    }
  }
}

}  // namespace aw
