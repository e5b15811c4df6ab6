// Detector conv stack as GEMMs (SURVEY K9, K10, K14; reference
// detection/modules/conv1d.py:38-42).  A 1x1 Conv1d over pooled frames is
//     D[row][n] = sum_k A[row][k] * B[n][k]
// with A = activations, channels-last [rows][K] (rows = clip-major pooled frames,
// each clip padded to a multiple of 128 rows), B = weights [N][K] (PyTorch's own
// (C_out, C_in) layout forward; the transposed copy for the input-gradient GEMM).
//
// k_gemm_tc: persistent tcgen05 GEMM (kind::tf32, or kind::f16 with fp16 / bf16 operands),
//   operands staged by TMA into 128B-swizzled shared tiles, fp32 accumulator double-buffered
//   in TMEM, warp-specialised (TMA producer / MMA issuer / 8 epilogue warps).  The epilogue
//   fuses the InstanceNorm statistics (forward) or the LeakyReLU' / InstanceNorm-adjoint
//   statistics (backward) and does all of its global traffic in a coalesced layout.
// k_gemm_exact: fp32 CUDA-core GEMM with the same epilogues (precision mode
//   "fp32": used to separate tensor-core rounding from logic errors in the
//   parity tests, and for detection at margins below TF32 resolution).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "common.cuh"

namespace aw {

// EPI_*_STATS / EPI_*_APPLY: two-pass form for the small-K layers (K <= 128), whose GEMM is cheaper than
// one round trip of its output.  STATS runs the GEMM for the InstanceNorm column sums only (no store);
// APPLY runs it again and normalises in the epilogue, so the raw H / dHhat tensor never exists in HBM.
// EPI_PEAK / EPI_SPEC: epilogues of the tensor-core spectral path (spectc.cuh): the band-limited
// iSTFT as a GEMM whose epilogue adds the constant out-of-band waveform and reduces max|y| (nothing is
// stored), and the band-limited STFT o iSTFT composite whose epilogue adds the constant out-of-band
// spectrum and writes |S| and S/|S|.
enum { EPI_PLAIN = 0, EPI_FWD = 1, EPI_BWD = 2, EPI_FWD_STATS = 3, EPI_FWD_APPLY = 4, EPI_BWD_STATS = 5,
       EPI_BWD_APPLY = 6, EPI_PEAK = 7, EPI_SPEC = 8 };
__host__ __device__ constexpr bool epi_is_bwd(int e) { return e == EPI_BWD || e == EPI_BWD_STATS || e == EPI_BWD_APPLY; }
__host__ __device__ constexpr bool epi_is_fwd(int e) { return e == EPI_FWD || e == EPI_FWD_STATS || e == EPI_FWD_APPLY; }
__host__ __device__ constexpr bool epi_has_stats(int e) { return e == EPI_FWD || e == EPI_BWD || e == EPI_FWD_STATS || e == EPI_BWD_STATS; }
__host__ __device__ constexpr bool epi_stores(int e) { return e != EPI_FWD_STATS && e != EPI_BWD_STATS && e != EPI_PEAK && e != EPI_SPEC; }
__host__ __device__ constexpr bool epi_applies(int e) { return e == EPI_FWD_APPLY || e == EPI_BWD_APPLY; }

struct EpiArgs {
  float* out;            // [rows][ldo]
  int ldo;
  int n_valid;           // columns < n_valid are stored
  float* part;           // [row_tiles][ldp][2] per-tile column partial sums (FWD/BWD)
  int ldp;
  const float* act;      // BWD: P_{l-1} [rows][ldo] (post-LeakyReLU activations)
};

// ------------------------------ PTX wrappers --------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug traps (-> CUDA error at the next sync) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) {
      printf("aware_b200: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y,
             threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// ---- CTA-pair (cta_group::2) helpers ----------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose transaction bytes are counted on a barrier of the LEADER CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t leader_bar,
                                                 int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
// commit of the leader's MMAs, arriving on the barrier at the same offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
template <int KIND_F16>
__device__ __forceinline__ void tc_mma_pair(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  if (KIND_F16)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d),
        "l"(a), "l"(b), "r"(idesc), "r"(acc)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d),
        "l"(a), "l"(b), "r"(idesc), "r"(acc)
        : "memory");
}

__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Asynchronous TMEM load (no wait) and a wait that names the destination registers as in/out
// operands, so the compiler cannot schedule their consumers above it.
__device__ __forceinline__ void tc_ld32_async(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]),
                 "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]),
                 "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]),
                 "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]),
                 "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// K-major, 128B-swizzled shared tile descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) = 1 | SBO>>4 [32,46) = 1024>>4 | version=1 [46,48)
// | layout_type = SWIZZLE_128B (2) [61,64)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffff) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Column sums of a 32(lanes = rows) x 32(registers = columns) block in 31 shuffles:
// after the call lane l holds the sum over the warp's 32 rows of column l.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int h = 16; h >= 1; h >>= 1) {
    const bool up = (lane & h) != 0;
#pragma unroll
    for (int i = 0; i < h; ++i) {
      const float keep = up ? v[i + h] : v[i];
      const float send = up ? v[i] : v[i + h];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, h);
    }
  }
  return v[0];
}

#define AW_GEMM_STAGES 4                  // BN <= 128; the 256-wide tile runs 3 stages (see gemm_stages)
#define AW_EPI_STRIDE 36                  // words per staged row: 16-byte accesses stay conflict-free
#define AW_EPI_STAGE_WORDS (32 * AW_EPI_STRIDE)
// Three warpgroups: 0 = TMA producer (warp 0), MMA issuer (warp 1) and two idle warps; 1 and 2 = the eight
// epilogue warps.  Whole warpgroups so that `setmaxnreg` can move registers from the two single-thread roles
// to the epilogue: with 12 warps ptxas caps a thread at 168 registers, which is what made every attempt to
// keep more epilogue loads in flight spill (profiles/r2_ncu_summary.md); after the hand-over the epilogue
// warps own 232 each and hold a ring of prefetched operand chunks.
#define AW_GEMM_THREADS 384
// Epilogues that hold an operand ring in registers run the three-warpgroup layout; the others keep the
// compact one (warp 0 TMA, warp 1 MMA, warps 2..9 epilogue; 320 threads, no register hand-over).
__host__ __device__ constexpr bool gemm_big_epi(int e) {
  return e == EPI_PEAK || e == EPI_SPEC || e == EPI_BWD || e == EPI_BWD_STATS;
}
__host__ __device__ constexpr int gemm_threads(int e) { return gemm_big_epi(e) ? AW_GEMM_THREADS : 320; }
#define AW_GEMM_REGS_LIGHT 56
#define AW_GEMM_REGS_EPI 224

// Operand element: float -> kind::tf32 (32 elements per 128-byte swizzle row, K=8 per MMA),
// __nv_bfloat16 -> kind::f16 (64 elements per row, K=16 per MMA).  Either way one k-block is
// 128 bytes wide and one MMA consumes 32 bytes of it.
template <typename T> struct GemmElem;
template <> struct GemmElem<float> {
  static constexpr int BK = 32;
  static constexpr uint32_t FMT = 2;       // TF32
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc,
                                             uint32_t acc) {
    tc_mma_tf32(d, a, b, idesc, acc);
  }
};
template <> struct GemmElem<__nv_bfloat16> {
  static constexpr int BK = 64;
  static constexpr uint32_t FMT = 1;       // BF16
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc,
                                             uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d),
        "l"(a), "l"(b), "r"(idesc), "r"(acc)
        : "memory");
  }
};

// fp16 operands: same 10-bit mantissa as TF32 at half the bytes and twice the MMA rate
template <> struct GemmElem<__half> {
  static constexpr int BK = 64;
  static constexpr uint32_t FMT = 0;       // F16
  static __device__ __forceinline__ void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc,
                                             uint32_t acc) {
    GemmElem<__nv_bfloat16>::mma(d, a, b, idesc, acc);   // kind::f16 covers both 16-bit formats
  }
};

__device__ __forceinline__ void act_ld4g(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void act_ld4g(const __nv_bfloat16* p, float (&v)[4]) {
  const uint2 t = *reinterpret_cast<const uint2*>(p);
  v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
  v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
}
__device__ __forceinline__ void act_ld4g(const __half* p, float (&v)[4]) {
  const uint2 t = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void act_st4g(__half* p, const float (&v)[4]) {
  const __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a),
                                            *reinterpret_cast<const uint32_t*>(&b));
}
__device__ __forceinline__ void act_st4g(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void act_st4g(__nv_bfloat16* p, const float (&v)[4]) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a),
                                            *reinterpret_cast<const uint32_t*>(&b));
}

// Four activations as loaded (converted when consumed): what the epilogue's prefetch ring holds, so that a
// 2-byte activation chunk in flight costs 16 registers instead of 32.
template <typename OT> struct ActRaw { uint2 v; };
template <> struct ActRaw<float> { float4 v; };
__device__ __forceinline__ void act_ldraw(const float* p, ActRaw<float>& r) {
  r.v = __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ void act_ldraw(const __half* p, ActRaw<__half>& r) {
  r.v = __ldg(reinterpret_cast<const uint2*>(p));
}
__device__ __forceinline__ void act_ldraw(const __nv_bfloat16* p, ActRaw<__nv_bfloat16>& r) {
  r.v = __ldg(reinterpret_cast<const uint2*>(p));
}
__device__ __forceinline__ void act_cvt(const ActRaw<float>& r, float (&v)[4]) {
  v[0] = r.v.x; v[1] = r.v.y; v[2] = r.v.z; v[3] = r.v.w;
}
__device__ __forceinline__ void act_cvt(const ActRaw<__nv_bfloat16>& r, float (&v)[4]) {
  v[0] = __uint_as_float(r.v.x << 16); v[1] = __uint_as_float(r.v.x & 0xffff0000u);
  v[2] = __uint_as_float(r.v.y << 16); v[3] = __uint_as_float(r.v.y & 0xffff0000u);
}
__device__ __forceinline__ void act_cvt(const ActRaw<__half>& r, float (&v)[4]) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.v.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.v.y));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

template <typename OT>
struct EpiArgsT {
  OT* out;               // [rows][ldo]
  int ldo;
  float* part;           // [row_tiles][ldp][2] per-tile column partial sums (FWD/BWD)
  int ldp;
  const OT* act;         // BWD: P_{l-1} [rows][ldo] (post-LeakyReLU activations)
  // *_APPLY: per-clip column statistics [clip][ldo][2] = (mean, rstd) / (a1, a2), rows per clip
  const float* stat;
  const float* bstat;
  int tiles_per_clip;    // 128-row tiles per clip (Tp_pad / 128)
  int Tp;                // valid pooled frames per clip: rows beyond are written as 0
  int round_tf32;
  // Toeplitz A operand (spectral path): map_a is the plain 2-D map of an array of frame rows
  // [rows + pad][P]; k-block kb of GEMM row r is elements (kb % (P/BK)) * BK .. of frame row
  // r + kb / (P/BK), i.e. GEMM row r is the concatenation of K / P consecutive frame rows.  0 = ordinary.
  int toep_P;
  // EPI_PEAK / EPI_SPEC
  int rpc;               // GEMM rows per clip (T + 6: three zero frame rows at either end)
  int total_rows;        // n_clips * rpc
  int T, L, nb;
  const float* aux;      // PEAK: y_oob [clip][L]      SPEC: S_oob [clip][T][nb] (float2)
  const float* fix;      // PEAK: [256..512) hop-2 scale, [512..768) hop-T scale per sample of the hop
  float fix0;            // PEAK: interior scale
  unsigned long long* peak;  // PEAK: [clip] packed peak (pack_peak_s), atomicMax
  float* mag;            // SPEC: [clip][T][nb]
  float2* qph;           // SPEC: [clip][T][nb]
};

// packed peak word with sign: see spec.cuh (declared here for the EPI_PEAK epilogue)
__device__ __forceinline__ unsigned long long gemm_pack_peak_s(float v, unsigned idx) {
  return ((unsigned long long)__float_as_uint(fabsf(v)) << 32) |
         ((unsigned long long)(0x7fffffffu - idx) << 1) | (v < 0.f ? 1ull : 0ull);
}


template <int BN>
__host__ __device__ constexpr int gemm_stages() { return BN == 256 ? 3 : AW_GEMM_STAGES; }
template <int BN>
__host__ __device__ constexpr int gemm_tmem_cols() { return BN == 192 ? 512 : 2 * BN; }   // power of two >= 2 BN
// CTA pair: every CTA stages its own 128 rows of A and HALF of the B tile, so a stage is a third smaller
template <int BN>
__host__ __device__ constexpr int gemm_stages_pair() { return BN == 256 ? 5 : 6; }
template <int BN>
constexpr int gemm_tc_smem_pair() {
  return gemm_stages_pair<BN>() * (128 * 128 + BN / 2 * 128) + 1024 + 256 + 2 * 2 * 4 * BN * 4 +
         8 * AW_EPI_STAGE_WORDS * 4;
}
template <int BN>
constexpr int gemm_tc_smem() {
  return gemm_stages<BN>() * (128 * 128 + BN * 128) + 1024 /*align*/ + 256 /*barriers*/ +
         2 * 2 * 4 * BN * 4 /*double-buffered column partials*/ +
         8 * AW_EPI_STAGE_WORDS * 4 /*per-warp epilogue transpose tiles*/;
}

// Tile index -> (128-row tile, column tile), column tile fastest
template <int CG>
__device__ __forceinline__ void gemm_tile_rc(int tile, int n_col_tiles, uint32_t rank, int& row_tile, int& col_tile) {
  row_tile = (tile / n_col_tiles) * CG + (int)rank;
  col_tile = tile % n_col_tiles;
}

// Persistent tcgen05 GEMM.  grid = min(#tiles, #SMs); every CTA walks tiles
// blockIdx.x, blockIdx.x + gridDim.x, ... (column tile fastest, so the CTAs that run
// concurrently share A row tiles in L2).  The fp32 accumulator is double-buffered in TMEM
// (2 x BN columns): while the 8 epilogue warps drain tile i, the MMA warp already
// accumulates tile i+1 and the TMA warp prefetches tile i+2's operands.
// CG = 1: one CTA per 128 x BN tile.  CG = 2: a CTA PAIR (cluster of 2, cta_group::2) per 256 x BN tile --
// each CTA stages its own 128 rows of A and half of the B tile (the weight tile is shared by the pair:
// half the shared-memory and L2 operand traffic per CTA), the leader issues one M = 256 MMA for both,
// each CTA's TMEM holds and each CTA's epilogue warps drain its own 128 rows.
template <typename T, typename OT, int BN, int EPI, int CG>
__device__ __forceinline__ void gemm_tc_body(const CUtensorMap& map_a, const CUtensorMap& map_b,
                                             int K, int n_row_tiles, int n_col_tiles, const EpiArgsT<OT>& ep) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by POINTER arithmetic on the __shared__ array: a round trip through uintptr_t made
  // the compiler forget the address space, every epilogue staging access became a generic LD.E / ST.E on the
  // long scoreboard, and a chunk's math then waited for the global prefetches queued behind them (ncu source
  // view, round 2)
#ifdef AW_GENERIC_SMEM
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
#else
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
#endif
  constexpr int BK = GemmElem<T>::BK;
  constexpr int NSTAGE = CG == 2 ? gemm_stages_pair<BN>() : gemm_stages<BN>();
  constexpr int A_BYTES = 128 * 128, B_BYTES = BN / CG * 128, STAGE = A_BYTES + B_BYTES;
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
  const int unit = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;          // tile walker: CTA or CTA pair
  const int n_units = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  uint8_t* tiles = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NSTAGE * STAGE);
  uint64_t* empty = full + NSTAGE;
  uint64_t* tfull = empty + NSTAGE;     // [2] accumulator ready
  uint64_t* tempty = tfull + 2;                 // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* s_part = reinterpret_cast<float*>(smem + NSTAGE * STAGE + 256);  // [2][2][4][BN]
  float* s_stage = s_part + 2 * 2 * 4 * BN;                                       // [8 warps][32][36]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = K / BK;
  const int n_tiles = n_row_tiles / CG * n_col_tiles;                            // CG = 2: tiles of 256 rows

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull + b, 1);
      mbar_init(tempty + b, 8 * CG);                 // the leader's: epilogue warps of both CTAs arrive
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (CG == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(tmem_slot)),
                   "n"(gemm_tmem_cols<BN>())
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(tmem_slot)),
                   "n"(gemm_tmem_cols<BN>())
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();                   // both CTAs' barriers exist before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t leader_full = CG == 2 ? mapa_u32(smem_u32(full), 0) : 0u;
  const uint32_t leader_tempty = CG == 2 ? mapa_u32(smem_u32(tempty), 0) : 0u;
  // register hand-over between warpgroups (see AW_GEMM_THREADS); each setmaxnreg sits at the head of the
  // branch it governs, which is how ptxas learns the register budget of that branch
  constexpr bool BIG = gemm_big_epi(EPI);
  constexpr int EW0 = BIG ? 4 : 2;                   // first epilogue warp
  if (warp < EW0) {
  if (BIG) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AW_GEMM_REGS_LIGHT));
  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = unit; tile < n_tiles; tile += n_units) {
        int rt_, ct_;
        gemm_tile_rc<CG>(tile, n_col_tiles, rank, rt_, ct_);
        const int row0 = rt_ * 128, n0 = ct_ * BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(empty + s, ph ^ 1);
          if (CG == 2) {
            // both CTAs' bytes are counted on the LEADER's barrier (it issues the MMA for the pair)
            if (rank == 0) mbar_expect_tx(full + s, 2 * STAGE);
            const int arow = ep.toep_P > 0 ? row0 + kb / (ep.toep_P / BK) : row0;
            const int acol = ep.toep_P > 0 ? (kb % (ep.toep_P / BK)) * BK : kb * BK;
            tma_load_2d_pair(tiles + s * STAGE, &map_a, leader_full + 8 * s, acol, arow);
            tma_load_2d_pair(tiles + s * STAGE + A_BYTES, &map_b, leader_full + 8 * s, kb * BK, n0 + (int)rank * (BN / 2));
            if (++s == NSTAGE) { s = 0; ph ^= 1; }
            continue;
          }
          mbar_expect_tx(full + s, STAGE);
          if (ep.toep_P > 0) {
            // Toeplitz operand: GEMM row r, k-block kb = the ordinary 2-D box of the frame-row array at
            // frame row r + kb / kpf, columns (kb % kpf) * BK .. -- a row offset per k-block, nothing else
            const int kpf = ep.toep_P / BK;                 // k-blocks per frame row
            tma_load_2d(tiles + s * STAGE, &map_a, full + s, (kb % kpf) * BK, row0 + kb / kpf);
          } else
            tma_load_2d(tiles + s * STAGE, &map_a, full + s, kb * BK, row0);
          tma_load_2d(tiles + s * STAGE + A_BYTES, &map_b, full + s, kb * BK, n0);
          if (++s == NSTAGE) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -------------------------------
    if (lane == 0 && rank == 0) {
      // instruction descriptor: D=F32 [4,6)=1, A/B format [7,10),[10,13), K-major A/B,
      // N>>3 at [17,23), M>>4 at [24,29)  (M = 256 for the CTA pair)
      const uint32_t idesc = (1u << 4) | (GemmElem<T>::FMT << 7) | (GemmElem<T>::FMT << 10) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((128 * CG) >> 4) << 24);
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int tile = unit; tile < n_tiles; tile += n_units, ++it) {
        const int ab = it & 1;
        mbar_wait(tempty + ab, ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(ab * BN);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(full + s, ph);
          tc_fence_after();
          const uint64_t ad = make_sw128_desc(smem_u32(tiles + s * STAGE));
          const uint64_t bd = make_sw128_desc(smem_u32(tiles + s * STAGE + A_BYTES));
#pragma unroll
          for (int k = 0; k < 4; ++k) {  // 4 x 32 bytes per 128-byte swizzle row
            if (CG == 2)
              tc_mma_pair<(GemmElem<T>::BK == 64)>(d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kb | k) != 0);
            else
              GemmElem<T>::mma(d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kb | k) != 0);
          }
          if (CG == 2) tc_commit_pair(empty + s); else tc_commit(empty + s);
          if (++s == NSTAGE) { s = 0; ph ^= 1; }
        }
        if (CG == 2) tc_commit_pair(tfull + ab); else tc_commit(tfull + ab);
      }
    }
  }
  } else {
    // -------------------------------- epilogue --------------------------------
    if (BIG) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(AW_GEMM_REGS_EPI));
    const int e = warp - EW0;
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    const int half = e >> 2;                        // which half of the BN columns
    constexpr int CHUNKS = BN / 64;                 // 32-column chunks per warp
    // Backward epilogues read the layer's activations P (LeakyReLU', IN-adjoint sums) and the *_APPLY ones
    // the per-clip column statistics: both are loaded ONE chunk ahead -- across the tile boundary -- into a
    // two-slot register ring, and the loads of chunk c + 1 are issued right after chunk c's registers have
    // been consumed.  (Issuing further ahead does not help: the hardware scoreboards are few, the wait for
    // chunk c's data then also waits for the younger loads queued on the same scoreboard -- ncu source view.)
    constexpr bool PF = (EPI == EPI_BWD || EPI == EPI_BWD_STATS) && CHUNKS == 4;
    constexpr bool SPF = EPI == EPI_FWD_APPLY && CHUNKS == 4;
    constexpr int NB = 2;
    ActRaw<OT> gr[PF ? NB : 1][8];
    float4 stq[SPF ? NB : 1][4];                    // (mean, rstd) x 4 columns, (a1, a2) x 4 columns
    const int sr_ = lane >> 3, cg_ = (lane & 7) * 4;
    auto act_tile_base = [&](int tile_) -> const OT* {
      int rt, ct;
      gemm_tile_rc<CG>(tile_, n_col_tiles, rank, rt, ct);
      return ep.act + (long long)(rt * 128 + q * 32 + sr_) * ep.ldo + ct * BN + half * (BN / 2) + cg_;
    };
    auto stat_tile_base = [&](int tile_) -> long long {
      int rt, ct;
      gemm_tile_rc<CG>(tile_, n_col_tiles, rank, rt, ct);
      return ((long long)(rt / ep.tiles_per_clip) * ep.ldo + ct * BN + half * (BN / 2) + cg_) * 2;
    };
    auto stat_load = [&](long long sb, float4 (&dst)[4]) {
      dst[0] = __ldg(reinterpret_cast<const float4*>(ep.stat + sb));
      dst[1] = __ldg(reinterpret_cast<const float4*>(ep.stat + sb + 4));
      if (EPI == EPI_BWD_APPLY) {
        dst[2] = __ldg(reinterpret_cast<const float4*>(ep.bstat + sb));
        dst[3] = __ldg(reinterpret_cast<const float4*>(ep.bstat + sb + 4));
      }
    };
    if (unit < n_tiles) {
      if (PF) {
        const OT* ab0 = act_tile_base(unit);
#pragma unroll
        for (int i = 0; i < 8; ++i) act_ldraw(ab0 + (long long)(4 * i) * ep.ldo, gr[0][i]);
      }
      if (SPF) stat_load(stat_tile_base(unit), stq[0]);
    }
    int it = 0;
    for (int tile = unit; tile < n_tiles; tile += n_units, ++it) {
      const int ab = it & 1;
      int row_tile, col_tile;
      gemm_tile_rc<CG>(tile, n_col_tiles, rank, row_tile, col_tile);
      const int n0 = col_tile * BN;
      const bool has_next = tile + n_units < n_tiles;
      const OT* abase_next = PF && has_next ? act_tile_base(tile + n_units) : nullptr;
      const long long sbase_next = SPF && has_next ? stat_tile_base(tile + n_units) : 0;
      // Global traffic goes through a per-warp 32 x 32 transpose tile: TMEM hands every lane
      // one ROW (32 columns in registers), but a warp-wide access is only coalesced when
      // adjacent lanes touch adjacent columns.  Staged, one 16-byte instruction covers 4 rows
      // x 128 contiguous bytes (4 wavefronts) instead of 32 rows x 16 bytes (32 wavefronts).
      float* s_st = s_stage + e * AW_EPI_STAGE_WORDS;
      const int sr = lane >> 3, cg = (lane & 7) * 4;  // staged access: row 4 i + sr, columns cg .. cg+3
      const long long grow = (long long)(row_tile * 128 + q * 32 + sr) * ep.ldo + n0 + half * (BN / 2) + cg;
      OT* obase = epi_stores(EPI) ? ep.out + grow : nullptr;
      const OT* abase = epi_is_bwd(EPI) ? ep.act + grow : nullptr;
      float* sp = s_part + ab * (2 * 4 * BN);
      float ga[8][4];
      // EPI_PEAK / EPI_SPEC: everything that depends only on the ROW is computed once per tile (the
      // epilogue warps are few -- two per scheduler -- so their instruction count is what bounds these
      // epilogues): GEMM row -> (clip, frame row), validity, the row's base pointer / offset
      const int sp_clip0 = EPI == EPI_PEAK ? (row_tile * 128) / ep.rpc : 0;   // a 128-row tile spans <= 2 clips
      // (32-bit element offsets: y_oob and the band spectra of one wave stay far below 2^31 elements)
      unsigned sp_yoff[8];           // PEAK: clip * L + 256 (hop - 2) into y_oob
      int sp_n0[8], sp_kind[8];      // PEAK: sample index of the hop's first sample; kind: 0 interior, 1 hop 2, 2 hop T,
                                     //       bit 4 clip slot, bit 8 = the row is a valid hop
      int sp_base[8];                // SPEC: (clip * T + t) * nb, or -1
      // PEAK: per clip slot (a tile spans <= 2 clips) the largest |y| so far, its signed value and sample index
      float sp_ba0 = -1.f, sp_ba1 = -1.f, sp_bv0 = 0.f, sp_bv1 = 0.f;
      int sp_bn0 = 0x7fffffff, sp_bn1 = 0x7fffffff;
      if (EPI == EPI_PEAK || EPI == EPI_SPEC) {
        const int r0 = row_tile * 128 + q * 32 + sr;
        const int c0_ = r0 / ep.rpc, t0_ = r0 - c0_ * ep.rpc;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          int ti = t0_ + 4 * i, ci = c0_;
          if (ti >= ep.rpc) { ti -= ep.rpc; ++ci; }
          const bool in = r0 + 4 * i < ep.total_rows;
          if (EPI == EPI_PEAK) {
            const bool ok = in && ti >= 2 && ti <= ep.T;
            sp_n0[i] = AW_HOP * (ti - 2);
            sp_yoff[i] = ok ? (unsigned)ci * (unsigned)ep.L + (unsigned)sp_n0[i] : 0u;
            sp_kind[i] = (ti == 2 ? 1 : (ti == ep.T ? 2 : 0)) | ((ci - sp_clip0) << 4) | (ok ? 256 : 0);
          } else {
            sp_base[i] = in && ti < ep.T ? (ci * ep.T + ti) * ep.nb : -1;
          }
        }
      }
      // *_APPLY: this tile's clip, its first row inside the clip, and the statistics base
      const int clip_ = epi_applies(EPI) ? row_tile / ep.tiles_per_clip : 0;
      const int jrow0 = epi_applies(EPI) ? (row_tile - clip_ * ep.tiles_per_clip) * 128 + q * 32 + sr : 0;
      const long long sbase = epi_applies(EPI) ? ((long long)clip_ * ep.ldo + n0 + half * (BN / 2) + cg) * 2 : 0;
      if (epi_is_bwd(EPI) && !PF) {                   // overlaps the wait for the accumulator
#pragma unroll
        for (int i = 0; i < 8; ++i) act_ld4g(abase + (long long)(4 * i) * ep.ldo, ga[i]);
      }
      // EPI_PEAK / EPI_SPEC: the constant operand (y_oob / S_oob) of chunk c + 1 is loaded while chunk c is
      // processed (two register buffers; chunk 0 overlaps the wait for the accumulator)
      float4 yo[EPI == EPI_PEAK ? 2 : 1][8];
      float2 so[EPI == EPI_SPEC ? 2 : 1][8][2];
      auto peak_load = [&](int c_, float4 (&dst)[8]) {
        const int j0_ = half * (BN / 2) + c_ * 32 + cg;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          dst[i] = (sp_kind[i] & 256) ? __ldg(reinterpret_cast<const float4*>(ep.aux + sp_yoff[i] + j0_))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      auto spec_load = [&](int c_, float2 (&dst)[8][2]) {
        const int b0_ = (half * (BN / 2) + c_ * 32 + cg) >> 1;
        const float2* aux2 = reinterpret_cast<const float2*>(ep.aux);
        const bool v0 = b0_ < ep.nb, v1 = b0_ + 1 < ep.nb;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float2* ap = aux2 + (sp_base[i] < 0 ? 0 : sp_base[i]) + b0_;
          dst[i][0] = v0 ? __ldg(ap) : make_float2(0.f, 0.f);          // row / bin validity only gates the stores
          dst[i][1] = v1 ? __ldg(ap + 1) : make_float2(0.f, 0.f);
        }
      };
      if (EPI == EPI_PEAK) peak_load(0, yo[0]);
      if (EPI == EPI_SPEC) spec_load(0, so[0]);
      mbar_wait(tfull + ab, (it >> 1) & 1);
      tc_fence_after();
      // the TMEM load of chunk c+1 is in flight while chunk c is processed
      uint32_t vbuf[2][32];
      tc_ld32_async(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * BN + half * (BN / 2)), vbuf[0]);
#pragma unroll
      for (int c = 0; c < CHUNKS; ++c) {
        const int c0 = half * (BN / 2) + c * 32;    // column inside the tile
        if (EPI == EPI_PEAK && c + 1 < CHUNKS) peak_load(c + 1, yo[EPI == EPI_PEAK ? ((c + 1) & 1) : 0]);
        if (EPI == EPI_SPEC && c + 1 < CHUNKS) spec_load(c + 1, so[EPI == EPI_SPEC ? ((c + 1) & 1) : 0]);
        {
          uint32_t (&v)[32] = vbuf[c & 1];
          tc_wait_ld(v);
          if (c + 1 < CHUNKS)
            tc_ld32_async(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * BN + c0 + 32), vbuf[(c + 1) & 1]);
          if (c == CHUNKS - 1) {                    // accumulator fully read: hand it back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (CG == 2) mbar_arrive_cluster(leader_tempty + 8 * ab);
              else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(tempty + ab)) : "memory");
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i)
            *reinterpret_cast<uint4*>(s_st + lane * AW_EPI_STRIDE + 4 * i) =
                make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        }
        __syncwarp();
        // from here on a lane owns columns cg..cg+3 of rows 4 i + sr: the layout of the
        // coalesced global accesses, so the activation / gradient math needs no second transpose
        float w[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 t4 = *reinterpret_cast<const float4*>(s_st + (4 * i + sr) * AW_EPI_STRIDE + cg);
          w[i][0] = t4.x; w[i][1] = t4.y; w[i][2] = t4.z; w[i][3] = t4.w;
        }
        __syncwarp();
        if (EPI == EPI_PEAK) {
          // y = y_band (this GEMM, scaled) + y_oob; only max |y| with its sample index and sign survives.
          // Straight-line code: the chunk's loads first (read-only path), then compare / select per row --
          // the epilogue warps are two per scheduler, so instruction count and branches are what it costs.
          const int j0 = half * (BN / 2) + c * 32 + cg;          // sample inside the hop (N = 256: one column tile)
          const float f0 = ep.fix0;
          float4 (&yc)[8] = yo[EPI == EPI_PEAK ? (c & 1) : 0];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 sc = make_float4(f0, f0, f0, f0);
            if (sp_kind[i] & 3)                                 // hop 2 / hop T of a clip: edge envelope (rare)
              sc = __ldg(reinterpret_cast<const float4*>(ep.fix + ((sp_kind[i] & 3) << 8) + j0));
            const float v0 = fmaf(w[i][0], sc.x, yc[i].x), v1 = fmaf(w[i][1], sc.y, yc[i].y);
            const float v2 = fmaf(w[i][2], sc.z, yc[i].z), v3 = fmaf(w[i][3], sc.w, yc[i].w);
            // largest |v| of the four, lowest index on ties
            const bool p1 = fabsf(v1) > fabsf(v0);
            const float a01 = p1 ? v1 : v0;
            const bool p3 = fabsf(v3) > fabsf(v2);
            const float a23 = p3 ? v3 : v2;
            const bool ph = fabsf(a23) > fabsf(a01);
            const float bv = ph ? a23 : a01;
            const int n = sp_n0[i] + j0 + (ph ? (p3 ? 3 : 2) : (p1 ? 1 : 0));
            const float ab = (sp_kind[i] & 256) ? fabsf(bv) : -2.f;
            const bool s1 = (sp_kind[i] & 16) != 0;
            const bool t0 = !s1 && (ab > sp_ba0 || (ab == sp_ba0 && n < sp_bn0));
            const bool t1 = s1 && (ab > sp_ba1 || (ab == sp_ba1 && n < sp_bn1));
            sp_ba0 = t0 ? ab : sp_ba0; sp_bv0 = t0 ? bv : sp_bv0; sp_bn0 = t0 ? n : sp_bn0;
            sp_ba1 = t1 ? ab : sp_ba1; sp_bv1 = t1 ? bv : sp_bv1; sp_bn1 = t1 ? n : sp_bn1;
          }
          continue;
        }
        if (EPI == EPI_SPEC) {
          // S = S_band (this GEMM) + S_oob; |S| and the phasor S/|S| of two bins per lane and row.
          // Loads of the whole chunk first, through the read-only path (no aliasing with the stores).
          const int b0 = (half * (BN / 2) + c * 32 + cg) >> 1;
          const bool v0 = b0 < ep.nb, v1 = b0 + 1 < ep.nb;
          float2 (&sc2)[8][2] = so[EPI == EPI_SPEC ? (c & 1) : 0];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float xr0 = w[i][0] + sc2[i][0].x, xi0 = w[i][1] + sc2[i][0].y;
            const float xr1 = w[i][2] + sc2[i][1].x, xi1 = w[i][3] + sc2[i][1].y;
            const float p0 = fmaf(xr0, xr0, xi0 * xi0), p1 = fmaf(xr1, xr1, xi1 * xi1);
            float r0, r1;                                              // MUFU reciprocal square root (<= 2 ulp), 0 -> inf
            asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(p0));
            asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(p1));
            r0 = p0 > 0.f ? r0 : 0.f;
            r1 = p1 > 0.f ? r1 : 0.f;
            if (sp_base[i] >= 0) {
              float* mrow = ep.mag + sp_base[i] + b0;
              float2* qrow = ep.qph + sp_base[i] + b0;
              if (v0) { mrow[0] = p0 * r0; qrow[0] = make_float2(xr0 * r0, xi0 * r0); }
              if (v1) { mrow[1] = p1 * r1; qrow[1] = make_float2(xr1 * r1, xi1 * r1); }
            }
          }
          continue;
        }
        float s1c[4] = {0.f, 0.f, 0.f, 0.f}, s2c[4] = {0.f, 0.f, 0.f, 0.f};
        float st_mu[4], st_rs[4], st_a1[4], st_a2[4];
        if (epi_applies(EPI)) {
          float4 s01, s23, b01 = make_float4(0.f, 0.f, 0.f, 0.f), b23 = b01;
          if (SPF) {
            s01 = stq[SPF ? (c & 1) : 0][0]; s23 = stq[SPF ? (c & 1) : 0][1];
            if (EPI == EPI_BWD_APPLY) { b01 = stq[SPF ? (c & 1) : 0][2]; b23 = stq[SPF ? (c & 1) : 0][3]; }
          } else {
            s01 = *reinterpret_cast<const float4*>(ep.stat + sbase + c * 64);
            s23 = *reinterpret_cast<const float4*>(ep.stat + sbase + c * 64 + 4);
            if (EPI == EPI_BWD_APPLY) {
              b01 = *reinterpret_cast<const float4*>(ep.bstat + sbase + c * 64);
              b23 = *reinterpret_cast<const float4*>(ep.bstat + sbase + c * 64 + 4);
            }
          }
          st_mu[0] = s01.x; st_rs[0] = s01.y; st_mu[1] = s01.z; st_rs[1] = s01.w;
          st_mu[2] = s23.x; st_rs[2] = s23.y; st_mu[3] = s23.z; st_rs[3] = s23.w;
          if (EPI == EPI_BWD_APPLY) {
            st_a1[0] = b01.x; st_a2[0] = b01.y; st_a1[1] = b01.z; st_a2[1] = b01.w;
            st_a1[2] = b23.x; st_a2[2] = b23.y; st_a1[3] = b23.z; st_a2[3] = b23.w;
          }
        }
        float gaf[PF ? 8 : 1][4];
        if (PF) {
#pragma unroll
          for (int i = 0; i < 8; ++i) act_cvt(gr[PF ? (c & 1) : 0][i], gaf[i]);
        }
        // chunk c's operands are in plain registers now: queue the loads of the next chunk
        if (PF) {
          const OT* src = c + 1 < CHUNKS ? abase + (c + 1) * 32 : abase_next;
          if (src) {
#pragma unroll
            for (int i = 0; i < 8; ++i) act_ldraw(src + (long long)(4 * i) * ep.ldo, gr[PF ? ((c + 1) & 1) : 0][i]);
          }
        }
        if (SPF) {
          if (c + 1 < CHUNKS) stat_load(sbase + (c + 1) * 64, stq[SPF ? ((c + 1) & 1) : 0]);
          else if (has_next) stat_load(sbase_next, stq[0]);
        }
        if (epi_is_bwd(EPI)) {
          // d(IN out) = dP * LeakyReLU'(P);  IN out recovered from P
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float gai[4];
            if (PF) { gai[0] = gaf[PF ? i : 0][0]; gai[1] = gaf[PF ? i : 0][1]; gai[2] = gaf[PF ? i : 0][2]; gai[3] = gaf[PF ? i : 0][3]; }
            else { gai[0] = ga[i][0]; gai[1] = ga[i][1]; gai[2] = ga[i][2]; gai[3] = ga[i][3]; }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float pv = gai[k];
              const bool pos = pv > 0.f;
              const float g = pos ? w[i][k] : AW_LEAKY * w[i][k];
              const float hh = pos ? pv : pv * (1.0f / AW_LEAKY);
              if (EPI == EPI_BWD_APPLY) {               // dH = rstd (dHhat - a1 - Hhat a2), pad rows 0 (k_norm_rows<BWD>)
                float o = st_rs[k] * (g - st_a1[k] - hh * st_a2[k]);
                if (sizeof(OT) == 4 && ep.round_tf32) o = to_tf32(o);   // TF32 mode stores float activations
                w[i][k] = jrow0 + 4 * i < ep.Tp ? o : 0.f;
              } else {
                w[i][k] = g;
                s1c[k] += g;
                s2c[k] = fmaf(hh, g, s2c[k]);
              }
            }
          }
          if (!PF && c + 1 < CHUNKS) {              // prefetch the next chunk's activations
#pragma unroll
            for (int i = 0; i < 8; ++i) act_ld4g(abase + (c + 1) * 32 + (long long)(4 * i) * ep.ldo, ga[i]);
          }
        } else if (EPI == EPI_FWD_APPLY) {            // P = LeakyReLU((H - mean) rstd), pad rows 0 (k_norm_rows<FWD>)
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              float o = leaky((w[i][k] - st_mu[k]) * st_rs[k]);
              if (sizeof(OT) == 4 && ep.round_tf32) o = to_tf32(o);   // TF32 mode stores float activations
              w[i][k] = jrow0 + 4 * i < ep.Tp ? o : 0.f;
            }
        } else if (epi_is_fwd(EPI)) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              s1c[k] += w[i][k];
              s2c[k] = fmaf(w[i][k], w[i][k], s2c[k]);
            }
        }
        if (epi_stores(EPI)) {
#pragma unroll
          for (int i = 0; i < 8; ++i) act_st4g(obase + c * 32 + (long long)(4 * i) * ep.ldo, w[i]);
        }
        if (epi_has_stats(EPI)) {
          // the 4 lanes that share (lane & 7) hold the same columns for different rows
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            s1c[k] += __shfl_xor_sync(0xffffffffu, s1c[k], 8);
            s2c[k] += __shfl_xor_sync(0xffffffffu, s2c[k], 8);
            s1c[k] += __shfl_xor_sync(0xffffffffu, s1c[k], 16);
            s2c[k] += __shfl_xor_sync(0xffffffffu, s2c[k], 16);
          }
          if (sr == 0) {
            *reinterpret_cast<float4*>(sp + (0 * 4 + q) * BN + c0 + cg) = make_float4(s1c[0], s1c[1], s1c[2], s1c[3]);
            *reinterpret_cast<float4*>(sp + (1 * 4 + q) * BN + c0 + cg) = make_float4(s2c[0], s2c[1], s2c[2], s2c[3]);
          }
        }
      }
      if (EPI == EPI_PEAK) {
        const unsigned long long m0 = sp_ba0 >= 0.f ? gemm_pack_peak_s(sp_bv0, (unsigned)sp_bn0) : 0ull;
        const unsigned long long m1 = sp_ba1 >= 0.f ? gemm_pack_peak_s(sp_bv1, (unsigned)sp_bn1) : 0ull;
        const unsigned long long w0 = warp_max_u64(m0), w1 = warp_max_u64(m1);
        if (lane == 0 && w0) atomicMax(ep.peak + sp_clip0, w0);
        if (lane == 0 && w1) atomicMax(ep.peak + sp_clip0 + 1, w1);
      }
      if (epi_has_stats(EPI)) {
        asm volatile("bar.sync 1, 256;" ::: "memory");                // the 8 epilogue warps
        const int t = threadIdx.x - 32 * EW0;                         // 0..255
        for (int cc = t; cc < BN; cc += 256) {
          float s1 = 0.f, s2 = 0.f;
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            s1 += sp[(0 * 4 + w) * BN + cc];
            s2 += sp[(1 * 4 + w) * BN + cc];
          }
          float* p = ep.part + ((long long)row_tile * ep.ldp + n0 + cc) * 2;
          p[0] = s1;
          p[1] = s2;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();                   // the peer may still be draining its half of the pair's TMEM
  if (warp == 1) {
    if (CG == 2)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(gemm_tmem_cols<BN>())
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(gemm_tmem_cols<BN>())
                   : "memory");
  }
}

template <typename T, typename OT, int BN, int EPI>
__global__ void __launch_bounds__(gemm_threads(EPI), 1)
k_gemm_tc(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
          int K, int n_row_tiles, int n_col_tiles, EpiArgsT<OT> ep) {
  gemm_tc_body<T, OT, BN, EPI, 1>(map_a, map_b, K, n_row_tiles, n_col_tiles, ep);
}

// CTA-pair form: map_b's box holds BN / 2 rows; n_row_tiles must be even; grid = 2 x #pairs
template <typename T, typename OT, int BN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(gemm_threads(EPI), 1)
k_gemm_tc_pair(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               int K, int n_row_tiles, int n_col_tiles, EpiArgsT<OT> ep) {
  gemm_tc_body<T, OT, BN, EPI, 2>(map_a, map_b, K, n_row_tiles, n_col_tiles, ep);
}

// ---------------------------------------------------------------------------
// exact fp32 GEMM (CUDA cores) + standalone epilogue with the same semantics
// ---------------------------------------------------------------------------
// D[rows][ldo] = A[rows][K] * B[N][K]^T ; 64x64 tile, 256 threads, 4x4 per thread.
// Products and sums are carried in float64 so the result is the correctly rounded fp32 of
// the exact dot product (better than any fp32 summation order): this path is the
// validation yardstick, not the fast path.
__global__ void __launch_bounds__(256) k_gemm_exact(const float* __restrict__ A,
                                                    const float* __restrict__ B, int K, int N,
                                                    float* __restrict__ D, int ldo) {
  __shared__ float sa[16][64 + 1], sb[16][64 + 1];
  const int r0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      const int r = i >> 4, k = i & 15;
      sa[k][r] = A[(long long)(r0 + r) * K + k0 + k];
      sb[k][r] = (c0 + r < N) ? B[(long long)(c0 + r) * K + k0 + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sa[k][ty * 4 + i]; b[i] = sb[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + tx * 4 + j;
      if (c < N) D[(long long)(r0 + ty * 4 + i) * ldo + c] = (float)acc[i][j];
    }
}

// Per 128-row tile column statistics (and the BWD transform), for the exact path.
// grid = (row_tiles, ceil(ncols/128)), block = 128 (one column per thread).
template <int EPI>
__global__ void __launch_bounds__(128) k_epilogue_exact(EpiArgs ep, int ncols) {
  const int row_tile = blockIdx.x;
  const int c = blockIdx.y * 128 + threadIdx.x;
  if (c >= ncols) return;
  float s1 = 0.f, s2 = 0.f;
  for (int r = 0; r < 128; ++r) {
    const long long o = (long long)(row_tile * 128 + r) * ep.ldo + c;
    float v = ep.out[o];
    if (EPI == EPI_BWD) {
      const float p = ep.act[o];
      const bool pos = p > 0.f;
      v = pos ? v : AW_LEAKY * v;
      ep.out[o] = v;
      s1 += v;
      s2 += (pos ? p : p * (1.0f / AW_LEAKY)) * v;
    } else {
      s1 += v;
      s2 += v * v;
    }
  }
  float* p = ep.part + ((long long)row_tile * ep.ldp + c) * 2;
  p[0] = s1;
  p[1] = s2;
}

}  // namespace aw
