// Fused spectral passes of the embedding loop (SURVEY K13 -> K1/K2/K3 and their adjoints;
// reference embedding/multibit_embedder.py:49-67 forward, :111 backward, :112-122 update).
//
//   SPEC_FWD : c, u  --iSTFT-->  y (+ y_oob)  --STFT-->  |S~| (un-normalised), q = S~/|S~|
//   SPEC_BWD : dA~, q --STFT^T--> dy --peak-normaliser^T, /env--> --iSTFT^T--> g --> NAdam
//
// One CTA owns FA = 58 consecutive analysis frames of one clip.  The waveform segment those
// frames cover (61 hops of the padded axis) never leaves shared memory: 64 synthesis frames
// are inverse-transformed (one frame PAIR per warp per FFT, as in fft.cuh), overlap-added
// with a register-resident sliding accumulator (each warp streams over 8 consecutive frames
// in ascending order -- torch.istft's order -- so completed hops are written with plain
// stores; only the 3-hop seam between two warps is a read-modify-write), transformed
// sample-wise in place (1/envelope, + y_oob, peak / peak-normaliser adjoint, reflect folds
// at the clip ends) and analysed again from shared memory.  Compared with separate
// synthesis / analysis kernels this removes the y and dpad round trips through HBM (7 MB
// per clip and iteration), one launch per direction and the 23 % halo recompute of a
// 32-frame tile (here 64/58 + 58/58 FFT pairs per 58 frames: 5 %).
//
// The peak normalisers (utils/audio/waveform.py:19, applied twice) are linear for a fixed
// peak, so the forward pass analyses the UN-normalised y and the per-clip factor
// 1/(d1 d2) is applied where the magnitudes are consumed (k_mel).  The backward pass
// needs s2 = sum_n dy2[n] y2[n]; |STFT| is homogeneous of degree 1 in y2, so by Euler's
// identity s2 = sum_{t,b} dA~[t,b] A~[t,b], which k_p0_bwd_apply accumulates -- the
// waveform is not needed again.
//
// The radix-32 passes are pruned at compile time: the inverse transform's first pass sees
// only the band's 32-bin groups (6 of 32 inputs non-zero at 44.1 kHz), the forward
// transform's second pass only has to produce those groups.
#pragma once
#include <utility>
#include "fft.cuh"

namespace aw {

// ---------------------------------------------------------------------------
// compile-time pruned radix-2 DIF stages over 32 registers
// ---------------------------------------------------------------------------
// NZ: bit i set = register i may be non-zero on entry.  NEED: bit i set = register i is
// consumed after this stage.  Registers that are zero are never read; registers that are
// not needed are never written (they keep stale values the caller never looks at).
__host__ __device__ constexpr uint32_t nz_after(uint32_t nz, int half) {
  uint32_t o = 0;
  for (int g = 0; g < 32; g += 2 * half)
    for (int j = 0; j < half; ++j) {
      const int i0 = g + j, i1 = i0 + half;
      if (((nz >> i0) | (nz >> i1)) & 1u) o |= (1u << i0) | (1u << i1);
    }
  return o;
}
__host__ __device__ constexpr uint32_t need_before(uint32_t need, int half) {
  uint32_t o = 0;
  for (int g = 0; g < 32; g += 2 * half)
    for (int j = 0; j < half; ++j) {
      const int i0 = g + j, i1 = i0 + half;
      if (((need >> i0) | (need >> i1)) & 1u) o |= (1u << i0) | (1u << i1);
    }
  return o;
}

__host__ __device__ constexpr int brevn(int x, int bits) {
  int r = 0;
  for (int i = 0; i < bits; ++i)
    if ((x >> i) & 1) r |= 1 << (bits - 1 - i);
  return r;
}
// cos / sin(2 pi e / 32) and their ratios as compile-time constants
__host__ __device__ constexpr double tw_cos(int e) {
  constexpr double c[16] = {1.0, 0.98078528040323043, 0.92387953251128674, 0.83146961230254524,
                            0.70710678118654757, 0.55557023301960229, 0.38268343236508984, 0.19509032201612833,
                            0.0, -0.19509032201612819, -0.38268343236508973, -0.55557023301960196,
                            -0.70710678118654746, -0.83146961230254535, -0.92387953251128674, -0.98078528040323043};
  return c[e];
}
__host__ __device__ constexpr double tw_sin(int e) {
  constexpr double s[16] = {0.0, 0.19509032201612825, 0.38268343236508978, 0.55557023301960218,
                            0.70710678118654746, 0.83146961230254524, 0.92387953251128674, 0.98078528040323043,
                            1.0, 0.98078528040323043, 0.92387953251128674, 0.83146961230254546,
                            0.70710678118654757, 0.55557023301960218, 0.38268343236508989, 0.19509032201612861};
  return s[e];
}

// One butterfly of the decimation-in-time network with natural-order input and bit-reversed
// output: stage S pairs registers half = 16 >> S apart inside 2^S groups, and every butterfly of
// group g uses the same twiddle W = exp(SIGN i 2 pi e / 32), e = brev_S(g) * (16 >> S):
//     (a, b) -> (a + W b, a - W b).
// Because W multiplies b BEFORE the add, a non-trivial butterfly is 6 FMAs (Linzer-Feig:
// W b = c (b + i t b) with t = s / c, or the cotangent form when |s| > |c|) instead of the
// 8 operations of the decimation-in-frequency form.
template <int SIGN, int S, uint32_t NZ, uint32_t NEED, int I>
__device__ __forceinline__ void bfly_p(float (&re)[32], float (&im)[32]) {
  constexpr int HALF = 16 >> S;
  constexpr int g = I / HALF, j = I % HALF;
  constexpr int i0 = g * 2 * HALF + j, i1 = i0 + HALF;
  constexpr bool anz = (NZ >> i0) & 1u, bnz = (NZ >> i1) & 1u;
  constexpr bool n0 = (NEED >> i0) & 1u, n1 = (NEED >> i1) & 1u;
  constexpr int e = brevn(g, S) * (16 >> S);
  constexpr float c = (float)tw_cos(e), sn = (float)(SIGN * tw_sin(e));
  if constexpr ((anz || bnz) && (n0 || n1)) {
    if constexpr (!bnz) {                               // b == 0: both outputs are a
      if constexpr (n1) { re[i1] = re[i0]; im[i1] = im[i0]; }
    } else if constexpr (!anz) {                        // a == 0: outputs are +-W b
      const float br = re[i1], bi = im[i1];
      float tr, ti;
      if constexpr (e == 0) { tr = br; ti = bi; }
      else if constexpr (e == 8) { tr = -SIGN * bi; ti = SIGN * br; }
      else { tr = br * c - bi * sn; ti = br * sn + bi * c; }
      if constexpr (n0) { re[i0] = tr; im[i0] = ti; }
      if constexpr (n1) { re[i1] = -tr; im[i1] = -ti; }
    } else {
      const float ar = re[i0], ai = im[i0], br = re[i1], bi = im[i1];
      if constexpr (e == 0) {
        if constexpr (n0) { re[i0] = ar + br; im[i0] = ai + bi; }
        if constexpr (n1) { re[i1] = ar - br; im[i1] = ai - bi; }
      } else if constexpr (e == 8) {                    // W = SIGN i
        if constexpr (n0) { re[i0] = ar - SIGN * bi; im[i0] = ai + SIGN * br; }
        if constexpr (n1) { re[i1] = ar + SIGN * bi; im[i1] = ai - SIGN * br; }
      } else if constexpr (e <= 4 || e >= 12) {         // |s| <= |c|: tangent form
        constexpr float t = (float)(SIGN * tw_sin(e) / tw_cos(e));
        const float t1 = fmaf(-t, bi, br), t2 = fmaf(t, br, bi);
        if constexpr (n0) { re[i0] = fmaf(c, t1, ar); im[i0] = fmaf(c, t2, ai); }
        if constexpr (n1) { re[i1] = fmaf(-c, t1, ar); im[i1] = fmaf(-c, t2, ai); }
      } else {                                          // cotangent form
        constexpr float ct = (float)(tw_cos(e) / (SIGN * tw_sin(e)));
        const float t1 = fmaf(ct, br, -bi), t2 = fmaf(ct, bi, br);
        if constexpr (n0) { re[i0] = fmaf(sn, t1, ar); im[i0] = fmaf(sn, t2, ai); }
        if constexpr (n1) { re[i1] = fmaf(-sn, t1, ar); im[i1] = fmaf(-sn, t2, ai); }
      }
    }
  }
}
template <int SIGN, int S, uint32_t NZ, uint32_t NEED, int... I>
__device__ __forceinline__ void stage_p(float (&re)[32], float (&im)[32], std::integer_sequence<int, I...>) {
  (bfly_p<SIGN, S, NZ, NEED, I>(re, im), ...);
}
// 32-point DFT, natural order in, bit-reversed order out (register p holds X[brev5(p)]).
// NZ = non-zero inputs (natural index), NEED = needed outputs (register index, i.e. brev5 of
// the natural output index).
template <int SIGN, uint32_t NZ, uint32_t NEED>
__device__ __forceinline__ void fft32_p(float (&re)[32], float (&im)[32]) {
  constexpr uint32_t Z1 = nz_after(NZ, 16), Z2 = nz_after(Z1, 8), Z3 = nz_after(Z2, 4), Z4 = nz_after(Z3, 2);
  constexpr uint32_t N4 = need_before(NEED, 1), N3 = need_before(N4, 2), N2 = need_before(N3, 4),
                     N1 = need_before(N2, 8);
  using Q = std::make_integer_sequence<int, 16>;
  stage_p<SIGN, 0, NZ, N1>(re, im, Q{});
  stage_p<SIGN, 1, Z1, N2>(re, im, Q{});
  stage_p<SIGN, 2, Z2, N3>(re, im, Q{});
  stage_p<SIGN, 3, Z3, N4>(re, im, Q{});
  stage_p<SIGN, 4, Z4, NEED>(re, im, Q{});
}

// natural-index set of the 32-bin groups that hold the band and its hermitian mirror:
// direct [LO..HI], mirror [31-HI..31-LO] (lanes > 0) and 32-k2 (lane 0, k2 >= 1).
__host__ __device__ constexpr uint32_t band_groups(int lo, int hi) {
  uint32_t m = 0;
  for (int k2 = lo; k2 <= hi; ++k2) {
    m |= 1u << k2;
    m |= 1u << (31 - k2);
    if (k2 >= 1) m |= 1u << (32 - k2);
  }
  return m;
}
__host__ __device__ constexpr uint32_t brev_mask(uint32_t m) {
  uint32_t o = 0;
  for (int i = 0; i < 32; ++i)
    if ((m >> i) & 1u) o |= 1u << brev5(i);
  return o;
}

#define AW_TR1_STRIDE 36                       // words per row: 16-byte row stores stay conflict-free
#define AW_TR1_FLOATS (32 * AW_TR1_STRIDE)     // per-warp transpose tile, one float plane

// 1024-point complex FFT across one warp (layout as warp_fft1024) with a pruned first
// (NZ1: natural-index non-zero inputs) and second (NEED2: register-index needed outputs)
// radix-32 pass.  The 32x32 transpose goes through a single-plane padded tile, real part
// first, then imaginary part: every lane stores its 32 registers as 8 x 16 bytes in REGISTER
// order and the readers undo the bit reversal with their column index brev5(lane), so the
// transpose costs 8 + 32 instead of 32 + 32 shared-memory instructions per plane.
template <int SIGN, uint32_t NZ1, uint32_t NEED2>
__device__ __forceinline__ void warp_fft1024_p(float (&re)[32], float (&im)[32], float* s_tr,
                                               const float2* s_tw, int lane) {
  fft32_p<SIGN, NZ1, 0xffffffffu>(re, im);
#pragma unroll
  for (int p = 1; p < 32; ++p) {          // p = 0 is k1 = 0: twiddle 1
    const int k1 = brev5(p);
    const float2 w = s_tw[k1 * 32 + lane];
    const float c = w.x, s = SIGN * w.y;
    const float r = re[p], i = im[p];
    re[p] = r * c - i * s;
    im[p] = r * s + i * c;
  }
  float* row = s_tr + lane * AW_TR1_STRIDE;
  const float* col = s_tr + (__brev((unsigned)lane) >> 27);     // register p of lane n2 holds k1 = brev5(p)
#pragma unroll
  for (int i = 0; i < 8; ++i)
    *reinterpret_cast<float4*>(row + 4 * i) = make_float4(re[4 * i], re[4 * i + 1], re[4 * i + 2], re[4 * i + 3]);
  __syncwarp();
#pragma unroll
  for (int n2 = 0; n2 < 32; ++n2) re[n2] = col[n2 * AW_TR1_STRIDE];
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 8; ++i)
    *reinterpret_cast<float4*>(row + 4 * i) = make_float4(im[4 * i], im[4 * i + 1], im[4 * i + 2], im[4 * i + 3]);
  __syncwarp();
#pragma unroll
  for (int n2 = 0; n2 < 32; ++n2) im[n2] = col[n2 * AW_TR1_STRIDE];
  __syncwarp();
  fft32_p<SIGN, 0xffffffffu, NEED2>(re, im);
}

// ---------------------------------------------------------------------------
// per-clip peak of y with the sample's sign: u64 max == (largest |y|, lowest index)
// [63:32] |y| bits, [31:1] 0x7fffffff - index, [0] sign(y) < 0
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long pack_peak_s(float v, unsigned idx) {
  return ((unsigned long long)__float_as_uint(fabsf(v)) << 32) |
         ((unsigned long long)(0x7fffffffu - idx) << 1) | (v < 0.f ? 1ull : 0ull);
}
__device__ __forceinline__ unsigned peak_s_index(unsigned long long p) {
  return 0x7fffffffu - (unsigned)((p & 0xffffffffull) >> 1);
}
__device__ __forceinline__ float peak_s_sign(unsigned long long p) {
  const float v = peak_value(p);
  return v > 0.f ? ((p & 1ull) ? -1.f : 1.f) : 0.f;
}

// Per-clip scalars of the two stacked peak normalisers and their sub-gradient
// (waveform.py:19 twice; SURVEY A.7): written once per iteration by k_clip_scalars.
struct ClipScal {
  float inv;     // 1 / (d1 d2)
  float corr;    // sign(y*) (s2/d2 + s1) / d1 : subtracted from dy at the arg-max sample
  int nstar;     // arg-max sample
  float pad;
};

// s2_part: [clip][nblk] partial sums of dA~ * A~(un-normalised), fixed-order reduction
// n_base: sample index of this rank's local sample 0 in the whole clip (frame-sharded mode packs
// GLOBAL indices into the peak word; 0 otherwise)
__global__ void __launch_bounds__(128) k_clip_scalars(const unsigned long long* __restrict__ peak_y,
                                                      const double* __restrict__ s2_part, int nblk,
                                                      int n_clips, ClipScal* __restrict__ out, int n_base = 0,
                                                      unsigned* __restrict__ dmax2 = nullptr,
                                                      const int* __restrict__ it_ptr = nullptr) {
  const int clip = blockIdx.x * blockDim.x + threadIdx.x;
  if (clip >= n_clips) return;
  // spectc.cuh: the slot that this iteration's k_tc_dsprep accumulates max |dA| into (next iteration's scale)
  if (dmax2) dmax2[(size_t)((*it_ptr + 1) & 1) * n_clips + clip] = 0u;
  const unsigned long long pk = peak_y[clip];
  const float p1 = peak_value(pk);
  const float d1 = p1 + 1e-8f;
  const float d2 = __fdiv_rn(p1, d1) + 1e-8f;
  ClipScal cs;
  cs.inv = __fdiv_rn(__fdiv_rn(1.0f, d1), d2);
  double s2d = 0.0;
  {
    // eight partials in flight at a time (one thread per clip: pure L2 latency otherwise), added in block order
    const double* sp = s2_part + (long long)clip * nblk;
    int i = 0;
    for (; i + 8 <= nblk; i += 8) {
      double v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = __ldg(sp + i + k);
#pragma unroll
      for (int k = 0; k < 8; ++k) s2d += v[k];
    }
    for (; i < nblk; ++i) s2d += sp[i];
  }
  const float s2 = (float)(s2d * (double)cs.inv);
  const float s1 = s2 * 1e-8f / d2;
  cs.corr = peak_s_sign(pk) * (s2 / d2 + s1) / d1;
  cs.nstar = (int)peak_s_index(pk) - n_base;
  cs.pad = 0.f;
  out[clip] = cs;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// ---------------------------------------------------------------------------
enum { SPEC_FWD = 0, SPEC_BWD = 1 };

struct SpecArgs {
  int n_clips, T, L, bin0, nbins, tiles;
  const float* window;         // [1024]
  const float2* twiddle;       // [k1][lane]
  const float* env256;         // [512]: envelope, reciprocal
  const float* amp;            // [clip][T][nbins]  FWD: c       BWD: dA~
  const float2* ph;            // [clip][T][nbins]  FWD: u       BWD: q
  // FWD
  const float* z_oob;          // [clip][L]  y_oob * overlap-add envelope (k_synthesis<SYN_OOB>)
  unsigned long long* peak_y;  // [clip] (atomicMax, pack_peak_s)
  float* mag;                  // [clip][T][nbins] out: |S~| of the un-normalised y
  float2* q;                   // [clip][T][nbins] out
  // BWD
  const ClipScal* scal;        // [clip]
  const float2* u;
  float* c; float* m; float* v; float* cbest;
  const float* c0;
  const int* improved;         // [clip]
  int* nonfinite;              // [clip] set to 1 when a gradient of the clip was inf / NaN (update skipped)
  const NadamStep* steps;
  const int* it_ptr;
  float tol_ratio;
  // frame-sharded long-form mode: only samples [pk_lo, pk_hi) of the local (halo-extended) segment
  // compete for the peak, and the index packed with it is global (local + idx_base).  pk_hi = 0: all.
  int pk_lo, pk_hi, idx_base;
  // edge mode (spectc.cuh): only the three frames at either end of every clip are evaluated -- item =
  // (clip, side).  FWD overwrites |S|, q of frames 0..2 / T-3..T-1 (no peak).  BWD takes dA of those
  // frames only, applies no peak correction, and writes the gradient it induces on frames 0..5 /
  // T-6..T-1 to g_edge [clip][12][nbins] instead of stepping the optimiser.
  int edge_mode;
  float* g_edge;
};

#define AW_SP_FA 58                        // analysis frames per tile
#define AW_SP_NSYN 64                      // synthesis frames per tile (FA + 6)
#define AW_SP_HOPS 61                      // padded-axis hops held in shared memory (FA + 3)
#define AW_SP_WARPS 8
#define AW_SP_BUF (AW_SP_HOPS * AW_HOP)
#define AW_SP_SMEM ((AW_SP_BUF + 1024 + 256 + 2048 + AW_SP_WARPS * AW_TR1_FLOATS) * 4)

template <int MODE, int K2LO, int K2HI>
__global__ void __launch_bounds__(32 * AW_SP_WARPS, 2) k_spec(SpecArgs a) {
  extern __shared__ float smem[];
  float* s_buf = smem;                                   // [61 hops][256]
  float* s_win = s_buf + AW_SP_BUF;                      // [1024]
  float* s_ienv = s_win + 1024;                          // [256] interior 1/envelope
  float2* s_tw = reinterpret_cast<float2*>(s_ienv + 256);
  float* s_tr = reinterpret_cast<float*>(s_tw + 1024);
  __shared__ unsigned long long s_pk[AW_SP_WARPS];

  constexpr uint32_t GROUPS = band_groups(K2LO, K2HI);
  constexpr uint32_t NEED_OUT = brev_mask(GROUPS);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = a.T, L = a.L, nb = a.nbins;
  for (int i = tid; i < 1024; i += 32 * AW_SP_WARPS) {
    s_win[i] = a.window[i];
    s_tw[i] = a.twiddle[i];
  }
  if (tid < 256) s_ienv[tid] = a.env256[256 + tid];
  float* my_tr = s_tr + warp * AW_TR1_FLOATS;
  const int lm = (32 - lane) & 31;
  const int n_items = a.edge_mode ? a.n_clips * 2 : a.n_clips * a.tiles;

  NadamStep st;
  if (MODE == SPEC_BWD) st = a.steps[*a.it_ptr];

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    int clip = item / a.tiles, tile = item - clip * a.tiles;
    // Frames [t_lo, t_hi) are written by this tile.  The frames that touch the right-hand
    // reflect seam (t >= T-5) must sit in a tile whose buffer reaches hop T+2, so the last
    // tile always owns at least the final 8 frames: a shorter last tile is pulled back and
    // its predecessor stops at T-8.
    bool is_last = tile == a.tiles - 1;
    const bool short_last = T > 8 && T - (a.tiles - 1) * AW_SP_FA < 8;
    int t_lo = tile * AW_SP_FA, t_hi = min(T, t_lo + AW_SP_FA);
    if (short_last && is_last) t_lo = T - 8;
    if (short_last && tile == a.tiles - 2) t_hi = T - 8;
    int ta0 = t_lo;
    int e_lo = -8, e_hi = T + 8;                          // synthesis frames that carry input (edge mode)
    if (a.edge_mode) {                                   // needs T >= 16
      clip = item >> 1;
      is_last = (item & 1) != 0;
      if (!is_last) {
        ta0 = 0; t_lo = 0; t_hi = MODE == SPEC_FWD ? 3 : 6;
        e_hi = MODE == SPEC_FWD ? 5 : 2;
      } else {
        ta0 = T - 8; t_lo = MODE == SPEC_FWD ? T - 3 : T - 6; t_hi = T;
        e_lo = MODE == SPEC_FWD ? T - 6 : T - 3;
      }
    }
    const int m0 = AW_HOP * ta0;                         // padded-axis origin of s_buf
    const long long fbase = (long long)clip * T;
    __syncthreads();                                     // tables / previous item done with s_buf

    // ---------------- phase 1: inverse transforms + streaming overlap-add ----------------
    {
      const int fs = ta0 - 3 + 8 * warp;                 // this warp's first synthesis frame
      if (MODE == SPEC_FWD) {
        // The constant out-of-band waveform (pre-multiplied by the overlap-add envelope) is
        // copied asynchronously into exactly the 8 hops this warp will store, and the stores
        // below accumulate onto it: no global load sits on the sample-wise phase.
        const float* zo = a.z_oob + (long long)clip * L;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int hr = fs - ta0 + i;                   // hop inside s_buf
          if (hr < 0 || hr >= AW_SP_HOPS) continue;
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const int r = hr * AW_HOP + (lane + 32 * k) * 4;
            const int n = m0 + r - AW_HALF;
            if (n >= 0 && n + 3 < L) cp_async16(s_buf + r, zo + n);
          }
        }
      }
      float acc[3][8];
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[i][e] = 0.f;
      const float scale = MODE == SPEC_FWD ? 1.0f / AW_NFFT : 0.5f;
      constexpr int NK = K2HI - K2LO + 1;
      float pa_[NK], pb_[NK];
      float2 qa_[NK], qb_[NK];
      auto fetch = [&](int pr) {
        const int ta = fs + 2 * pr, tb = ta + 1;
        const bool va = ta >= 0 && ta < T && ta >= e_lo && ta <= e_hi, vb = tb >= 0 && tb < T && tb >= e_lo && tb <= e_hi;
        const long long oa = (fbase + (va ? ta : 0)) * nb, ob = (fbase + (vb ? tb : 0)) * nb;
#pragma unroll
        for (int k2 = K2LO; k2 <= K2HI; ++k2) {
          const int b = lane + 32 * k2 - a.bin0;
          const int bc = (b >= 0 && b < nb) ? b : 0;
          pa_[k2 - K2LO] = a.amp[oa + bc]; pb_[k2 - K2LO] = a.amp[ob + bc];
          qa_[k2 - K2LO] = a.ph[oa + bc]; qb_[k2 - K2LO] = a.ph[ob + bc];
        }
      };
#pragma unroll 1
      for (int pr = 0; pr < 4; ++pr) {
        const int ta = fs + 2 * pr, tb = ta + 1;
        const bool va = ta >= 0 && ta < T && ta >= e_lo && ta <= e_hi, vb = tb >= 0 && tb < T && tb >= e_lo && tb <= e_hi;
        fetch(pr);
        float re[32], im[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) { re[j] = 0.f; im[j] = 0.f; }
        {
          const float sa = va ? scale : 0.f, sb = vb ? scale : 0.f;
          float mr[NK + 1], mi[NK + 1];
          mr[NK] = 0.f; mi[NK] = 0.f;
#pragma unroll
          for (int k2 = K2LO; k2 <= K2HI; ++k2) {
            const int b = lane + 32 * k2 - a.bin0;
            const bool ok = b >= 0 && b < nb;
            const float s0 = ok ? sa * pa_[k2 - K2LO] : 0.f, s1 = ok ? sb * pb_[k2 - K2LO] : 0.f;
            const float2 p0 = qa_[k2 - K2LO], p1 = qb_[k2 - K2LO];
            const float ar = s0 * p0.x, ai = s0 * p0.y, br = s1 * p1.x, bi = s1 * p1.y;
            re[k2] = ar - bi;                            // Z[k] = Xa + i Xb
            im[k2] = ai + br;
            // Z[1024-k] = conj(Xa) + i conj(Xb), needed by lane (32-lane)&31
            mr[k2 - K2LO] = __shfl_sync(0xffffffffu, ar + bi, lm);
            mi[k2 - K2LO] = __shfl_sync(0xffffffffu, br - ai, lm);
          }
          // mirror of group k2 lives in register 31-k2 (lane > 0) or 32-k2 (lane 0, k2 >= 1):
          // register 31-j takes M(j) on lanes > 0 and M(j+1) on lane 0
#pragma unroll
          for (int j = K2LO - (K2LO >= 1 ? 1 : 0); j <= K2HI; ++j) {
            const float r_hi = j >= K2LO ? mr[j - K2LO] : 0.f, i_hi = j >= K2LO ? mi[j - K2LO] : 0.f;
            const float r_l0 = j + 1 <= K2HI ? mr[j + 1 - K2LO] : 0.f, i_l0 = j + 1 <= K2HI ? mi[j + 1 - K2LO] : 0.f;
            re[31 - j] = lane ? r_hi : r_l0;
            im[31 - j] = lane ? i_hi : i_l0;
          }
        }
        if (va || vb)                                    // warp-uniform
          warp_fft1024_p<1, GROUPS, 0xffffffffu>(re, im, my_tr, s_tw, lane);
        // sliding overlap-add with the synthesis window folded into the accumulation:
        // frame A = re (t = ta), frame B = im (t = ta + 1); sample n = lane + 32 q sits in
        // register brev5(q); quarter i of a frame is q in [8i, 8i+8)
        float o0[8], o1[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float w0 = s_win[lane + 32 * e], w1 = s_win[lane + 32 * (8 + e)];
          const float w2 = s_win[lane + 32 * (16 + e)], w3 = s_win[lane + 32 * (24 + e)];
          o0[e] = fmaf(re[brev5(e)], w0, acc[0][e]);
          o1[e] = fmaf(im[brev5(e)], w0, fmaf(re[brev5(8 + e)], w1, acc[1][e]));
          acc[0][e] = fmaf(im[brev5(8 + e)], w1, fmaf(re[brev5(16 + e)], w2, acc[2][e]));
          acc[1][e] = fmaf(im[brev5(16 + e)], w2, re[brev5(24 + e)] * w3);
          acc[2][e] = im[brev5(24 + e)] * w3;
        }
        if (MODE == SPEC_FWD && pr == 0) {
          cp_async_wait_all();
          __syncwarp();
        }
        const int h0r = ta - ta0, h1r = h0r + 1;         // hop index inside s_buf
        if (h0r >= 0 && h0r < AW_SP_HOPS) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float* d = s_buf + h0r * AW_HOP + lane + 32 * e;
            *d = MODE == SPEC_FWD ? *d + o0[e] : o0[e];
          }
        }
        if (h1r >= 0 && h1r < AW_SP_HOPS) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float* d = s_buf + h1r * AW_HOP + lane + 32 * e;
            *d = MODE == SPEC_FWD ? *d + o1[e] : o1[e];
          }
        }
      }
      __syncthreads();
      // seam: this warp's 3 trailing partial hops are the next warp's 3 leading hops
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const int hr = fs + 8 + i - ta0;
        if (hr >= 0 && hr < AW_SP_HOPS && warp < AW_SP_WARPS - 1) {
#pragma unroll
          for (int e = 0; e < 8; ++e) s_buf[hr * AW_HOP + lane + 32 * e] += acc[i][e];
        }
      }
    }
    __syncthreads();

    // ---------------- phase 2: sample-wise transform in place -----------------------------
    const bool left_edge = ta0 == 0;
    const bool right_edge = is_last;
    if (MODE == SPEC_BWD && (left_edge || right_edge)) {
      // adjoint of the reflect padding: fold the pad samples back onto the signal
      if (left_edge)
        for (int m = tid; m < AW_HALF; m += 32 * AW_SP_WARPS) s_buf[AW_NFFT - m] += s_buf[m];
      if (right_edge)
        for (int m = L + AW_HALF + tid; m < L + AW_NFFT; m += 32 * AW_SP_WARPS) {
          const int r = m - m0, rt = 2 * L + 1022 - m - m0;
          if (r >= 0 && r < AW_SP_BUF && rt >= 0) s_buf[rt] += s_buf[r];
        }
      __syncthreads();
    }
    {
      float inv = 1.f, corr = 0.f;
      int nstar = -1;
      if (MODE == SPEC_BWD) {
        const ClipScal cs = a.scal[clip];
        inv = cs.inv; corr = cs.corr; nstar = cs.nstar;
      }
      float best = 0.f;
      int best_n = -1;
      const int pk_lo = a.pk_lo, pk_hi = a.pk_hi > 0 ? a.pk_hi : L;
      for (int r4 = tid * 4; r4 < AW_SP_BUF; r4 += 4 * 32 * AW_SP_WARPS) {
        const int m = m0 + r4, n = m - AW_HALF, hop = m >> 8;
        float4 s4 = *reinterpret_cast<float4*>(s_buf + r4);
        float vv[4] = {s4.x, s4.y, s4.z, s4.w};
        if (n >= 0 && n + 3 < L) {                       // all four samples are signal samples
          float ie[4];
          if (hop >= 3 && hop <= T - 1) {
            const float4 e4 = *reinterpret_cast<const float4*>(s_ienv + (m & 255));
            ie[0] = e4.x; ie[1] = e4.y; ie[2] = e4.z; ie[3] = e4.w;
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) ie[k] = ola_inv_envelope(m + k, T, s_win, a.env256);
          }
          if (MODE == SPEC_FWD) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              vv[k] = vv[k] * ie[k];                     // (ola + y_oob * env) / env
              if ((fabsf(vv[k]) > fabsf(best) || best_n < 0) && (n + k >= pk_lo && n + k < pk_hi)) {
                best = vv[k];
                best_n = n + k;
              }
            }
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              float dy = vv[k] * inv;
              if (n + k == nstar && !a.edge_mode) dy -= corr;
              vv[k] = dy * ie[k];
            }
          }
        } else {
          vv[0] = vv[1] = vv[2] = vv[3] = 0.f;           // pad region (L % 4 == 0: never mixed)
        }
        *reinterpret_cast<float4*>(s_buf + r4) = make_float4(vv[0], vv[1], vv[2], vv[3]);
      }
      if (MODE == SPEC_FWD) {
        unsigned long long pk = best_n >= 0 ? pack_peak_s(best, (unsigned)(best_n + a.idx_base)) : 0ull;
        pk = warp_max_u64(pk);
        if (lane == 0) s_pk[warp] = pk;
      }
    }
    __syncthreads();
    if (MODE == SPEC_FWD) {
      if (tid == 0 && !a.edge_mode) {
        unsigned long long pk = s_pk[0];
        for (int w = 1; w < AW_SP_WARPS; ++w) pk = s_pk[w] > pk ? s_pk[w] : pk;
        atomicMax(a.peak_y + clip, pk);
      }
      if (left_edge || right_edge) {
        // reflect padding of y (torch.stft center=True, pad_mode='reflect')
        if (left_edge)
          for (int m = tid; m < AW_HALF; m += 32 * AW_SP_WARPS) s_buf[m] = s_buf[AW_NFFT - m];
        if (right_edge)
          for (int m = L + AW_HALF + tid; m < L + AW_NFFT; m += 32 * AW_SP_WARPS) {
            const int r = m - m0, rs = 2 * L + 1022 - m - m0;
            if (r >= 0 && r < AW_SP_BUF) s_buf[r] = rs >= 0 ? s_buf[rs] : 0.f;
          }
        __syncthreads();
      }
    }

    // ---------------- phase 3: forward transforms from shared memory ----------------------
    bool improved = false;
    if (MODE == SPEC_BWD) improved = a.improved[clip] != 0;
#pragma unroll 1
    for (int p = warp; p < AW_SP_FA / 2; p += AW_SP_WARPS) {
      const int ta = ta0 + 2 * p, tb = ta + 1;
      if (ta >= t_hi || tb < t_lo) continue;             // warp-uniform
      float re[32], im[32];
      const float* fa = s_buf + AW_HOP * (2 * p) + lane;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float w = s_win[32 * j + lane];
        re[j] = fa[32 * j] * w;
        im[j] = fa[32 * j + AW_HOP] * w;
      }
      warp_fft1024_p<-1, 0xffffffffu, NEED_OUT>(re, im, my_tr, s_tw, lane);
      const bool wa = ta >= t_lo, wb = tb < t_hi;
      constexpr int NK = K2HI - K2LO + 1;
      constexpr int G = NK < 3 ? NK : 3;                 // bin groups handled per batch
#pragma unroll
      for (int g0 = K2LO; g0 <= K2HI; g0 += G) {
        float fr[G][2], fi[G][2];
        bool okb[G];
        long long ob_[G];
#pragma unroll
        for (int gi = 0; gi < G; ++gi) {
          const int k2 = g0 + gi;
          okb[gi] = false;
          fr[gi][0] = fr[gi][1] = fi[gi][0] = fi[gi][1] = 0.f;
          ob_[gi] = 0;
          if (k2 > K2HI) continue;
          // Z[k], k = lane + 32 k2, is register brev5(k2); its mirror Z[1024-k] is register
          // brev5(31-k2) of lane 32-lane (lane > 0) or register brev5(32-k2) of lane 0
          float mr = __shfl_sync(0xffffffffu, re[brev5(31 - k2)], lm);
          float mi = __shfl_sync(0xffffffffu, im[brev5(31 - k2)], lm);
          if (k2 >= 1 && lane == 0) {
            mr = re[brev5((32 - k2) & 31)];
            mi = im[brev5((32 - k2) & 31)];
          }
          const int b = lane + 32 * k2 - a.bin0;
          okb[gi] = b >= 0 && b < nb;
          ob_[gi] = (fbase + ta) * nb + (okb[gi] ? b : 0);
          const float zr = re[brev5(k2)], zi = im[brev5(k2)];
          // frame a: (Z[k] + conj Z[N-k]) / 2 ; frame b: (Z[k] - conj Z[N-k]) / (2i)
          fr[gi][0] = 0.5f * (zr + mr); fr[gi][1] = 0.5f * (zi + mi);
          fi[gi][0] = 0.5f * (zi - mi); fi[gi][1] = 0.5f * (mr - zr);
        }
        if (MODE == SPEC_FWD) {
#pragma unroll
          for (int gi = 0; gi < G; ++gi)
#pragma unroll
            for (int f = 0; f < 2; ++f) {
              if (!okb[gi] || (f == 0 ? !wa : !wb)) continue;
              const long long o = ob_[gi] + (long long)f * nb;
              const float sr = fr[gi][f], si = fi[gi][f];
              // |S| and S/|S| from one reciprocal square root (MUFU, <= 2 ulp): inside the loop the
              // magnitudes only feed the detector and the phasor only weights the gradient
              const float p2 = sr * sr + si * si;
              const float iv = p2 > 0.f ? rsqrtf(p2) : 0.f;
              a.mag[o] = p2 * iv;
              a.q[o] = make_float2(sr * iv, si * iv);
            }
        } else {
          // all state of the batch is requested before any of it is consumed
          float2 uu[G][2];
          float mm[G][2], vv[G][2], cc[G][2], c0[G][2];
#pragma unroll
          for (int gi = 0; gi < G; ++gi)
#pragma unroll
            for (int f = 0; f < 2; ++f) {
              const bool on = okb[gi] && (f == 0 ? wa : wb);
              const long long o = on ? ob_[gi] + (long long)f * nb : fbase * nb;   // any valid address
              uu[gi][f] = a.u[o]; mm[gi][f] = a.m[o]; vv[gi][f] = a.v[o];
              cc[gi][f] = a.c[o]; c0[gi][f] = a.c0[o];
            }
#pragma unroll
          for (int gi = 0; gi < G; ++gi)
#pragma unroll
            for (int f = 0; f < 2; ++f) {
              if (!okb[gi] || (f == 0 ? !wa : !wb)) continue;
              const long long o = ob_[gi] + (long long)f * nb;
              // dX = (2/N) DFT(.) ; g = Re(dX conj(u))     (multibit_embedder.py:111)
              const float g = (2.0f / AW_NFFT) * (fr[gi][f] * uu[gi][f].x + fi[gi][f] * uu[gi][f].y);
              if (a.edge_mode) {                          // gradient induced by the edge rows only, no update
                const int t = ta + f;
                const int er = !is_last ? t : 6 + (t - (T - 6));
                a.g_edge[((long long)clip * 12 + er) * nb + (o - (fbase + t) * nb)] = g;
                continue;
              }
              // an overflowed reduced-precision gradient must not poison m / v (NaN would pin the
              // coefficient to its lower bound for good): skip the step and flag the clip
              if ((__float_as_uint(g) & 0x7f800000u) == 0x7f800000u) {
                if (a.nonfinite) a.nonfinite[clip] = 1;
                continue;
              }
              // NAdam (torch/optim/nadam.py), clamp (:116-117), best (:120-122)
              float m1 = mm[gi][f], v1 = vv[gi][f], c1 = cc[gi][f];
              m1 = __fadd_rn(m1, __fmul_rn(0.1f, __fsub_rn(g, m1)));
              v1 = __fmul_rn(v1, 0.999f);
              v1 = __fadd_rn(v1, __fmul_rn(__fmul_rn(0.001f, g), g));
              // sqrt / reciprocal on the special-function unit (<= 1 ulp each): 2e-7 relative on a
              // step of at most lr = 0.1, far below the 1e-4 one-step parity gate
              float sq, rden;
              asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(__fmul_rn(v1, st.inv_bc2)));
              const float den = __fadd_rn(sq, 1e-8f);
              asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rden) : "f"(den));
              c1 = __fadd_rn(c1, __fmul_rn(__fmul_rn(st.a_g, g), rden));
              c1 = __fadd_rn(c1, __fmul_rn(__fmul_rn(st.a_m, m1), rden));
              const float dl = __fmul_rn(c0[gi][f], a.tol_ratio);
              const float lo = fmaxf(0.f, __fsub_rn(c0[gi][f], dl)), hi = __fadd_rn(c0[gi][f], dl);
              c1 = fminf(fmaxf(c1, lo), hi);
              a.m[o] = m1;
              a.v[o] = v1;
              a.c[o] = c1;
              if (improved) a.cbest[o] = c1;
            }
        }
      }
    }
  }
}

}  // namespace aw
