// aware_b200 C ABI (include/aware_b200.h): context, workspace and the batched
// detect / embed / attack pipelines built from the kernels in this directory.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <math.h>
#include <stdarg.h>
#include <limits.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "../../include/aware_b200.h"
#include "attacks.cuh"
#include "common.cuh"
#include "conv.cuh"
#include "fft.cuh"
#include "gemm.cuh"
#include "gemm64.cuh"
#include "net.cuh"
#include "spec.cuh"
#include "spectc.cuh"
#include "stoi.cuh"
#include "vocoder.cuh"

namespace aw {
thread_local char g_err[512] = "";
int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
}  // namespace aw

using namespace aw;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static const int kC[5] = {128, 512, 1024, 1024, 40};     // channel widths (detector_net.py:58)
static const int kCp[5] = {128, 512, 1024, 1024, 64};    // padded to GEMM tiles

struct MelCfg {
  int bin0, nbins, nnz;
  int *rowptr, *col, *colptr, *row;
  float *val, *valT;
};

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
};

struct aw_ctx {
  int device = 0, prec = AW_PREC_TF32;
  int64_t launches = 0;
  float* d_w[4] = {};    // forward weights  [kCp[l+1]][kCp[l]]
  float* d_wt[4] = {};   // transposed       [kCp[l]][kCp[l+1]]
  __nv_bfloat16* d_w16[4] = {};    // bf16 copies (embed loop in bf16)
  __nv_bfloat16* d_wt16[4] = {};
  __half* d_w16h[4] = {};          // fp16 copies (AW_PREC_FP16)
  __half* d_wt16h[4] = {};
  int num_sms = 148;
  float* d_window = nullptr;
  float2* d_twiddle = nullptr;   // [k1][lane] = exp(2 pi i lane k1 / 1024)
  float* d_env256 = nullptr;     // interior overlap-add envelope sum_r w^2[j + 256 r]
  std::vector<float> h_mel, h_window;
  float band_lo = 500.f, band_hi = 4000.f, tol_db = 6.f, threshold = 0.f;
  std::vector<MelCfg> mels;
  PFN_encodeTiled encode = nullptr;
  CUtensorMap tm_w[4], tm_wt[4], tm_w16[4], tm_wt16[4], tm_w16h[4], tm_wt16h[4];
  // the same weights with a 128-row box: every CTA of a CTA pair stages half of the 256-wide B tile
  CUtensorMap tm_w_p[4], tm_wt_p[4], tm_w16_p[4], tm_wt16_p[4], tm_w16h_p[4], tm_wt16h_p[4];
  bool pair_gemm = true;           // K >= 512 layers on CTA pairs (cta_group::2); AW_B200_NO_PAIR=1 / AW_OPT_PAIR_GEMM: off
  // workspace (grow-only)
  Buf scal, zoob, p0coef, p0scal, hpart, hcoef, red_a, red_b, red_c;
  // CUDA-graph replay of the optimisation iteration (AW_B200_NO_GRAPH=1 disables): the ~50 launches
  // of one iteration are captured once on a context-owned stream and replayed iters-1 times
  bool graphs = true;
  cudaStream_t gstream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  Buf accum, peakx, mag, ph_u, ph_q, c0, c, m, v, cbest, dA, yoob, y, M, cs, sigma;
  Buf act[5], ga, gb, dh4, dp0, part, stat[5], bstat, values, best, improved, pattern, itc, steps;
  Buf gsc;               // [clip] per-clip loss scale of the back-propagated gradient (16-bit modes)
  Buf nonfinite;         // [n_clips of the last embed call] 1 = a non-finite gradient was skipped
  Buf smax;              // [clip] signed max of the input, order-preserving int encoding (scale_mode 1)
  Buf lowm;              // [1 + n_clips] low-margin count + per-clip flags (aw_detect_batch re-evaluation)
  int* h_lowm = nullptr; // pinned host mirror of lowm
  size_t h_lowm_cap = 0;
  double exact_margin = 1e-3;      // AW_OPT_EXACT_MARGIN
  bool two_pass = true;            // small-K layers as statistics pass + apply pass (AW_B200_ONE_PASS=1: off)
  bool bwd64_stream = true;        // 16-bit loops: the backward K = 64 layer on k_gemm_bwd64 (TMA-streamed activations, AW_OPT_BWD64_STREAM)
  // tensor-core spectral path of the fp16 embed loop (spectc.cuh; AW_B200_FFT_SPEC=1: off)
  bool tc_spec = true;
  int tc_min_frames = 24 * 1024;   // n_clips * frames from which the tensor-core path is used (AW_OPT_TC_SPECTRAL value > 1 sets it)
  struct TcMats {
    int bin0 = -1, nb = 0;
    __half *peakB = nullptr, *compB = nullptr, *compBT = nullptr;
    float* fix = nullptr;
    CUtensorMap tm_peakB, tm_compB, tm_compBT;
  } tcm;
  Buf tc_X, tc_dS, tc_soob, tc_dX, tc_gedge, tc_dmax, tc_ones;
  CUtensorMap tm_tcX, tm_tcdS;     // plain 2-D maps of the frame-row arrays (Toeplitz by row offset per k-block)
  void *tc_map_x = nullptr, *tc_map_ds = nullptr;
  long long tc_map_rows = 0;
  bool tc_active = false;          // set while an embed wave runs on the tensor-core spectral path
  int64_t stat_detect_clips = 0, stat_reeval_clips = 0;
  int last_embed_clips = 0;
  // frame-sharded long-form mode (aw_*_sharded): this context holds a halo-extended segment of ONE
  // clip; per-clip statistics are all-reduced over the ranks through the caller's callbacks
  struct Shard {
    aw_comm comm;
    int e0;                    // global index of the segment's first frame
    int own_lo, own_hi;        // frames this rank owns, LOCAL indices into the segment
    int64_t n_allreduce = 0, n_allgather = 0;
  };
  Shard* sh = nullptr;
  int ws_rows = 0;
  // activation tensor maps, [0] = float32 view, [1] = bf16 view of the same buffers
  CUtensorMap tm_act[2][4], tm_dh4[2], tm_ga1024[2], tm_ga512[2], tm_gb1024[2];
  Buf cvt_a, cvt_b;    // aw_gemm bf16 test hook
  Buf stoi_ws;         // aw_stoi_batch workspace
  Buf conv_x, conv_idx;  // aw_attack_convolve: packed input block spectra, per-clip filter index
  bool stoi_edges_set = false;
  // state of the last embed wave (for aw_embed_state)
  int last_n = 0, last_T = 0, last_nb = 0;
  // optional CUDA-event timing of the GEMM launches (aw_profile_*)
  struct ProfRec { int n, k, epi; cudaEvent_t a, b; };
  std::vector<const void*> smem_attr_done;   // kernels whose dynamic-smem limit was raised on this device
  bool prof_on = false;
  std::vector<ProfRec> prof;
  // every-launch timeline: an event before each launch; a kernel's time = next mark - its mark
  struct Mark { const char* label; cudaEvent_t e; };
  std::vector<Mark> marks;
  std::vector<cudaEvent_t> ev_pool;
};

static cudaEvent_t prof_event(aw_ctx* ctx) {
  cudaEvent_t e;
  if (!ctx->ev_pool.empty()) {
    e = ctx->ev_pool.back();
    ctx->ev_pool.pop_back();
  } else {
    cudaEventCreate(&e);
  }
  return e;
}

// Timeline mark in front of a launch (label = nullptr closes the previous interval).
static void prof_mark(aw_ctx* ctx, cudaStream_t st, const char* label) {
  if (!ctx->prof_on) return;
  cudaEvent_t e = prof_event(ctx);
  cudaEventRecord(e, st);
  ctx->marks.push_back({label, e});
}

// interned "gemm_<epi>_n<N>_k<K>" labels (pointers stay valid for the process lifetime)
static const char* gemm_label(int epi, int n, int k) {
  static char table[32][32];
  static int used = 0;
  char buf[32];
  static const char* kind[9] = {"plain", "fwd", "bwd", "fwd_stats", "fwd_apply", "bwd_stats", "bwd_apply", "peak", "spec"};
  snprintf(buf, sizeof(buf), "gemm_%s_n%d_k%d", epi >= 0 && epi < 9 ? kind[epi] : "other", n, k);
  for (int i = 0; i < used; ++i)
    if (strcmp(table[i], buf) == 0) return table[i];
  if (used == 32) return "gemm_other";
  strcpy(table[used], buf);
  return table[used++];
}

// cudaFuncSetAttribute is per device: remember it per context, not per process
static int raise_smem_limit(aw_ctx* ctx, const void* func, int bytes) {
  for (const void* f : ctx->smem_attr_done)
    if (f == func) return 0;
  AW_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  ctx->smem_attr_done.push_back(func);
  return 0;
}

static int ensure(Buf& b, size_t bytes) {
  if (bytes <= b.cap) return 0;
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  AW_CUDA(cudaMalloc(&b.p, bytes));
  b.cap = bytes;
  return 0;
}

// Long clips produce thousands of per-block partial sums per clip; reduce them in groups first so
// the per-clip consumers (one CTA per clip) stay short.  Returns the array / block count to read.
static int reduce_if_long(aw_ctx* ctx, Buf& scratch, const double*& part, int& nblk, int n_clips, int W,
                          cudaStream_t st) {
  if (nblk <= 512) return 0;
  const int G = 64, nob = (nblk + G - 1) / G;
  if (ensure(scratch, (size_t)n_clips * nob * W * sizeof(double))) return 1;
  prof_mark(ctx, st, "reduce_partials");
  k_reduce_partials<<<dim3((W + 255) / 256, nob, n_clips), 256, 0, st>>>(part, nblk, W, G, (double*)scratch.p);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  part = (const double*)scratch.p;
  nblk = nob;
  return 0;
}

// ---- frame-sharded mode: reductions over ranks ------------------------------------------------
// arena layout (caller-owned device buffer): [0, 32 KB) reduction operand, [32 KB, 64 KB) halo send,
// [64 KB, 64 KB + world * 32 KB) halo receive
#define AW_ARENA_RED 0
#define AW_ARENA_SEND (32 << 10)
#define AW_ARENA_RECV (64 << 10)
#define AW_HALO 8
static int sh_allreduce(aw_ctx* ctx, int64_t count, int dtype, int op, cudaStream_t st) {
  aw_ctx::Shard* sh = ctx->sh;
  prof_mark(ctx, st, "allreduce");
  if (sh->comm.allreduce(sh->comm.user, AW_ARENA_RED, count, dtype, op, (void*)st))
    return set_error("frame-sharded mode: all-reduce callback failed");
  sh->n_allreduce++;
  prof_mark(ctx, st, nullptr);
  return 0;
}
// [nblk][W] float64 partials of the single clip -> arena[0..W) (fixed order), all-reduced (sum)
static int sh_reduce_sum(aw_ctx* ctx, Buf& scratch, const double* part, int nblk, int W, cudaStream_t st) {
  if (reduce_if_long(ctx, scratch, part, nblk, 1, W, st)) return 1;
  double* red = (double*)((uint8_t*)ctx->sh->comm.d_arena + AW_ARENA_RED);
  prof_mark(ctx, st, "reduce_partials");
  k_reduce_partials<<<dim3((W + 255) / 256, 1, 1), 256, 0, st>>>(part, nblk, W, nblk, red);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return sh_allreduce(ctx, W, AW_COMM_F64, AW_COMM_SUM, st);
}
static const double* sh_red(aw_ctx* ctx) { return (const double*)((uint8_t*)ctx->sh->comm.d_arena + AW_ARENA_RED); }
// per-clip packed peak word: max over ranks (the u64 word never has bit 63 set: int64 max == u64 max)
static int sh_peak_max(aw_ctx* ctx, unsigned long long* peak, cudaStream_t st) {
  void* red = (uint8_t*)ctx->sh->comm.d_arena + AW_ARENA_RED;
  AW_CUDA(cudaMemcpyAsync(red, peak, 8, cudaMemcpyDeviceToDevice, st));
  if (sh_allreduce(ctx, 1, AW_COMM_I64, AW_COMM_MAX, st)) return 1;
  AW_CUDA(cudaMemcpyAsync(peak, red, 8, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// boundary frames of a [T_seg][nb] float array: own frames [own_lo, own_lo+H) and [own_hi-H, own_hi)
// -> send[2][H][nb]; after the all-gather the neighbours' pieces land in this rank's halos
__global__ void k_halo_pack(const float* __restrict__ a, int nb, int own_lo, int own_hi, int H,
                            float* __restrict__ send) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, per = H * nb;
  if (i >= 2 * per) return;
  const int side = i / per, r = i - side * per;
  const int frame = side == 0 ? own_lo + r / nb : own_hi - H + r / nb;
  send[i] = a[(long long)frame * nb + r % nb];
}
__global__ void k_halo_unpack(const float* __restrict__ recv, int nb, int own_lo, int own_hi, int H, int rank,
                              int world, int stride_floats, float* __restrict__ a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, per = H * nb;
  if (i >= 2 * per) return;
  const int side = i / per, r = i - side * per;
  if (side == 0) {                     // left halo <- left neighbour's LAST H own frames
    if (rank == 0) return;
    a[(long long)(own_lo - H + r / nb) * nb + r % nb] = recv[(long long)(rank - 1) * stride_floats + per + r];
  } else {                             // right halo <- right neighbour's FIRST H own frames
    if (rank == world - 1) return;
    a[(long long)(own_hi + r / nb) * nb + r % nb] = recv[(long long)(rank + 1) * stride_floats + r];
  }
}
static int sh_halo_exchange(aw_ctx* ctx, float* arr, int nb, cudaStream_t st) {
  aw_ctx::Shard* sh = ctx->sh;
  if (sh->comm.world == 1) return 0;
  float* send = (float*)((uint8_t*)sh->comm.d_arena + AW_ARENA_SEND);
  float* recv = (float*)((uint8_t*)sh->comm.d_arena + AW_ARENA_RECV);
  const int per = AW_HALO * nb, tot = 2 * per;
  prof_mark(ctx, st, "halo_pack");
  k_halo_pack<<<(tot + 255) / 256, 256, 0, st>>>(arr, nb, sh->own_lo, sh->own_hi, AW_HALO, send);
  prof_mark(ctx, st, "allgather");
  if (sh->comm.allgather(sh->comm.user, AW_ARENA_SEND, AW_ARENA_RECV, (int64_t)tot * 4, (void*)st))
    return set_error("frame-sharded mode: all-gather callback failed");
  sh->n_allgather++;
  prof_mark(ctx, st, "halo_unpack");
  k_halo_unpack<<<(tot + 255) / 256, 256, 0, st>>>(recv, nb, sh->own_lo, sh->own_hi, AW_HALO, sh->comm.rank,
                                                   sh->comm.world, tot, arr);
  ctx->launches += 2;
  AW_LAUNCH_CHECK();
  prof_mark(ctx, st, nullptr);
  return 0;
}

// ---- the places where the frame-sharded mode differs from a batch; no-ops for whole clips
static int sync_peak(aw_ctx* ctx, unsigned long long* peak, cudaStream_t st) {
  return ctx->sh ? sh_peak_max(ctx, peak, st) : 0;
}
static int sync_halo(aw_ctx* ctx, float* arr, int nb, cudaStream_t st) {
  return ctx->sh ? sh_halo_exchange(ctx, arr, nb, st) : 0;
}
// [clip][nblk][W] partial sums -> what a per-clip consumer reads: grouped when long (whole clips), or
// summed over the whole clip into one block (frame-sharded mode)
static int clip_sums(aw_ctx* ctx, Buf& scratch, const double*& part, int& nblk, int n_clips, int W, cudaStream_t st) {
  if (!ctx->sh) return reduce_if_long(ctx, scratch, part, nblk, n_clips, W, st);
  if (sh_reduce_sum(ctx, scratch, part, nblk, W, st)) return 1;
  part = sh_red(ctx);
  nblk = 1;
  return 0;
}

// 2-D K-major tensor map with 128-byte swizzle; one box row = 128 bytes of K.
static int make_map(aw_ctx* ctx, CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t K,
                    uint32_t box_rows, bool bf16) {
  const uint64_t esz = bf16 ? 2 : 4;
  cuuint64_t gdim[2] = {K, rows};
  cuuint64_t gstr[1] = {K * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ctx->encode(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                           2, (void*)ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error("cuTensorMapEncodeTiled failed: %d", (int)r);
  return 0;
}

static int bn_for(int n) { return n >= 256 ? 256 : (n >= 128 ? 128 : 64); }

template <typename T, typename OT, int BN, int EPI>
static int launch_tc(aw_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mb, int rows, int n,
                     int k, const EpiArgsT<OT>& ep, cudaStream_t st) {
  if (raise_smem_limit(ctx, (const void*)k_gemm_tc<T, OT, BN, EPI>, gemm_tc_smem<BN>())) return 1;
  const int n_row_tiles = rows / 128, n_col_tiles = n / BN;
  const int tiles = n_row_tiles * n_col_tiles;
  const int grid = std::min(tiles, ctx->num_sms);
  aw_ctx::ProfRec pr;
  if (ctx->prof_on) {
    pr.n = n; pr.k = k; pr.epi = EPI;
    pr.a = prof_event(ctx); pr.b = prof_event(ctx);
    cudaEventRecord(pr.a, st);
  }
  prof_mark(ctx, st, gemm_label(EPI, n, k));
  k_gemm_tc<T, OT, BN, EPI><<<grid, gemm_threads(EPI), gemm_tc_smem<BN>(), st>>>(ma, mb, k, n_row_tiles,
                                                                                 n_col_tiles, ep);
  if (ctx->prof_on) {
    cudaEventRecord(pr.b, st);
    ctx->prof.push_back(pr);
  }
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

// CTA-pair form (cta_group::2): 256 x 256 tiles, `mb_half` = the weight map with a 128-row box
template <typename T, typename OT, int EPI>
static int launch_tc_pair(aw_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mb_half, int rows, int n,
                          int k, const EpiArgsT<OT>& ep, cudaStream_t st) {
  constexpr int BN = 256;
  if (raise_smem_limit(ctx, (const void*)k_gemm_tc_pair<T, OT, BN, EPI>, gemm_tc_smem_pair<BN>())) return 1;
  const int n_row_tiles = rows / 128, n_col_tiles = n / BN;
  const int pairs = n_row_tiles / 2 * n_col_tiles;
  const int grid = 2 * std::min(pairs, ctx->num_sms / 2);
  aw_ctx::ProfRec pr;
  if (ctx->prof_on) {
    pr.n = n; pr.k = k; pr.epi = EPI;
    pr.a = prof_event(ctx); pr.b = prof_event(ctx);
    cudaEventRecord(pr.a, st);
  }
  prof_mark(ctx, st, gemm_label(EPI, n, k));
  k_gemm_tc_pair<T, OT, BN, EPI><<<grid, gemm_threads(EPI), gemm_tc_smem_pair<BN>(), st>>>(ma, mb_half, k, n_row_tiles,
                                                                                           n_col_tiles, ep);
  if (ctx->prof_on) {
    cudaEventRecord(pr.b, st);
    ctx->prof.push_back(pr);
  }
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}
// Measured (256 clips x 10 s, profiles/r2_pair_gemm.txt): the pair wins where operand staging bounds the
// tile -- K bytes per row >= 2 KB (TF32 K >= 512: -16 %, fp16 K = 1024: -5..10 %); at fp16 K = 512 the
// tile is epilogue-bound and coupling the two CTAs' drains costs 15 %, so that layer stays on single CTAs.
static bool pair_ok(aw_ctx* ctx, int rows, int n, int k, int elem_bytes) {
  return ctx->pair_gemm && (rows / 128) % 2 == 0 && n % 256 == 0 && k * elem_bytes >= 2048;
}

// backward K = 64 layer as a streaming kernel (gemm64.cuh): activations in through a TMA ring, dH out through TMA
template <typename T, int EPI>
static int launch_bwd64(aw_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mb128, const CUtensorMap& mact,
                        const CUtensorMap& mout, int rows, int n, int k, const Gemm64Args& ga, cudaStream_t st) {
  if (raise_smem_limit(ctx, (const void*)k_gemm_bwd64<T, EPI>, gemm64_smem<EPI>())) return 1;
  const int n_row_tiles = rows / 128, n_col_tiles = n / AW_G64_BN;
  const int grid = std::min(n_row_tiles * n_col_tiles, ctx->num_sms);
  aw_ctx::ProfRec pr;
  if (ctx->prof_on) {
    pr.n = n; pr.k = k; pr.epi = EPI;
    pr.a = prof_event(ctx); pr.b = prof_event(ctx);
    cudaEventRecord(pr.a, st);
  }
  prof_mark(ctx, st, gemm_label(EPI, n, k));
  k_gemm_bwd64<T, EPI><<<grid, 320, gemm64_smem<EPI>(), st>>>(ma, mb128, mact, mout, k,
                                                              n_row_tiles, n_col_tiles, ga);
  if (ctx->prof_on) {
    cudaEventRecord(pr.b, st);
    ctx->prof.push_back(pr);
  }
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

// tensor-core GEMM, operands of type T, output/activation type OT
template <typename T, typename OT, int EPI>
static int launch_tc_bn(aw_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mb, int rows, int n,
                        int k, const EpiArgsT<OT>& ep, cudaStream_t st) {
  switch (bn_for(n)) {
    case 256: return launch_tc<T, OT, 256, EPI>(ctx, ma, mb, rows, n, k, ep, st);
    case 128: return launch_tc<T, OT, 128, EPI>(ctx, ma, mb, rows, n, k, ep, st);
    default: return launch_tc<T, OT, 64, EPI>(ctx, ma, mb, rows, n, k, ep, st);
  }
}

// exact fp32 path: CUDA-core GEMM + stand-alone epilogue kernel
template <int EPI>
static int launch_exact(aw_ctx* ctx, const float* a, const float* b, int rows, int n, int k,
                        const EpiArgsT<float>& ept, cudaStream_t st) {
  EpiArgs ep;
  ep.out = ept.out; ep.ldo = ept.ldo; ep.n_valid = n; ep.part = ept.part; ep.ldp = ept.ldp; ep.act = ept.act;
  dim3 grid(rows / 64, (n + 63) / 64);
  prof_mark(ctx, st, "gemm_exact");
  k_gemm_exact<<<grid, 256, 0, st>>>(a, b, k, n, ep.out, ep.ldo);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  if (EPI != EPI_PLAIN) {
    dim3 g2(rows / 128, (n + 127) / 128);
    prof_mark(ctx, st, "epilogue_exact");
    k_epilogue_exact<EPI><<<g2, 128, 0, st>>>(ep, n);
    ctx->launches++;
    AW_LAUNCH_CHECK();
  }
  return 0;
}

// ---------------------------------------------------------------------------
extern "C" const char* aw_last_error(void) { return g_err; }
extern "C" const char* aw_version(void) { return "aware_b200 0.1 (sm_100a)"; }

extern "C" int aw_ctx_create(aw_ctx** out, int device, const aw_model* model) {
  AW_REQUIRE(out && model, "aw_ctx_create: null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error("aw_ctx_create: no CUDA device (this library has no CPU fallback)");
  AW_REQUIRE(device >= 0 && device < ndev, "aw_ctx_create: bad device %d", device);
  AW_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  AW_CUDA(cudaGetDeviceProperties(&prop, device));
  AW_REQUIRE(prop.major == 10, "aw_ctx_create: device is sm_%d%d, this build targets sm_100a",
             prop.major, prop.minor);
  aw_ctx* ctx = new aw_ctx();
  ctx->device = device;
  ctx->band_lo = model->band_lo_hz;
  ctx->band_hi = model->band_hi_hz;
  ctx->tol_db = model->tolerance_db;
  ctx->threshold = model->threshold;
  ctx->h_mel.assign(model->mel_basis, model->mel_basis + AW_NMEL * 513);
  ctx->h_window.assign(model->window, model->window + 1024);
  {
    const char* e = getenv("AW_B200_NO_GRAPH");
    ctx->graphs = !(e && e[0] == '1');
    const char* e2 = getenv("AW_B200_ONE_PASS");
    ctx->two_pass = !(e2 && e2[0] == '1');
    const char* e3 = getenv("AW_B200_FFT_SPEC");
    ctx->tc_spec = !(e3 && e3[0] == '1');
    const char* e4 = getenv("AW_B200_NO_PAIR");
    ctx->pair_gemm = !(e4 && e4[0] == '1');
  }

  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  AW_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  AW_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
  ctx->encode = (PFN_encodeTiled)fn;

  // weights: zero-padded forward copies and transposed copies for the input-gradient GEMMs
  for (int l = 0; l < 4; ++l) {
    const int co = kC[l + 1], ci = kC[l], cop = kCp[l + 1], cip = kCp[l];
    std::vector<float> w((size_t)cop * cip, 0.f), wt((size_t)cip * cop, 0.f);
    for (int o = 0; o < co; ++o)
      for (int i = 0; i < ci; ++i) {
        const float x = model->w[l][(size_t)o * ci + i];
        w[(size_t)o * cip + i] = x;
        wt[(size_t)i * cop + o] = x;
      }
    AW_CUDA(cudaMalloc(&ctx->d_w[l], w.size() * 4));
    AW_CUDA(cudaMalloc(&ctx->d_wt[l], wt.size() * 4));
    AW_CUDA(cudaMemcpy(ctx->d_w[l], w.data(), w.size() * 4, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(ctx->d_wt[l], wt.data(), wt.size() * 4, cudaMemcpyHostToDevice));
    if (make_map(ctx, &ctx->tm_w[l], ctx->d_w[l], cop, cip, bn_for(cop), false)) return 1;
    if (make_map(ctx, &ctx->tm_wt[l], ctx->d_wt[l], cip, cop, bn_for(cip), false)) return 1;
    std::vector<__nv_bfloat16> w16(w.size()), wt16(wt.size());
    for (size_t i = 0; i < w.size(); ++i) w16[i] = __float2bfloat16_rn(w[i]);
    for (size_t i = 0; i < wt.size(); ++i) wt16[i] = __float2bfloat16_rn(wt[i]);
    AW_CUDA(cudaMalloc(&ctx->d_w16[l], w16.size() * 2));
    AW_CUDA(cudaMalloc(&ctx->d_wt16[l], wt16.size() * 2));
    AW_CUDA(cudaMemcpy(ctx->d_w16[l], w16.data(), w16.size() * 2, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(ctx->d_wt16[l], wt16.data(), wt16.size() * 2, cudaMemcpyHostToDevice));
    if (make_map(ctx, &ctx->tm_w16[l], ctx->d_w16[l], cop, cip, bn_for(cop), true)) return 1;
    if (make_map(ctx, &ctx->tm_wt16[l], ctx->d_wt16[l], cip, cop, bn_for(cip), true)) return 1;
    // fp16 copies; the tensor maps only move bytes, so the 16-bit (bf16-typed) encoding serves both
    std::vector<__half> w16h(w.size()), wt16h(wt.size());
    for (size_t i = 0; i < w.size(); ++i) w16h[i] = __float2half_rn(w[i]);
    for (size_t i = 0; i < wt.size(); ++i) wt16h[i] = __float2half_rn(wt[i]);
    AW_CUDA(cudaMalloc(&ctx->d_w16h[l], w16h.size() * 2));
    AW_CUDA(cudaMalloc(&ctx->d_wt16h[l], wt16h.size() * 2));
    AW_CUDA(cudaMemcpy(ctx->d_w16h[l], w16h.data(), w16h.size() * 2, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(ctx->d_wt16h[l], wt16h.data(), wt16h.size() * 2, cudaMemcpyHostToDevice));
    if (make_map(ctx, &ctx->tm_w16h[l], ctx->d_w16h[l], cop, cip, bn_for(cop), true)) return 1;
    if (make_map(ctx, &ctx->tm_wt16h[l], ctx->d_wt16h[l], cip, cop, bn_for(cip), true)) return 1;
    if (cop >= 256) {
      if (make_map(ctx, &ctx->tm_w_p[l], ctx->d_w[l], cop, cip, 128, false)) return 1;
      if (make_map(ctx, &ctx->tm_w16_p[l], ctx->d_w16[l], cop, cip, 128, true)) return 1;
      if (make_map(ctx, &ctx->tm_w16h_p[l], ctx->d_w16h[l], cop, cip, 128, true)) return 1;
    }
    if (cip >= 256) {
      if (make_map(ctx, &ctx->tm_wt_p[l], ctx->d_wt[l], cip, cop, 128, false)) return 1;
      if (make_map(ctx, &ctx->tm_wt16_p[l], ctx->d_wt16[l], cip, cop, 128, true)) return 1;
      if (make_map(ctx, &ctx->tm_wt16h_p[l], ctx->d_wt16h[l], cip, cop, 128, true)) return 1;
    }
  }
  ctx->num_sms = prop.multiProcessorCount;
  AW_CUDA(cudaMalloc(&ctx->d_window, 1024 * 4));
  AW_CUDA(cudaMemcpy(ctx->d_window, model->window, 1024 * 4, cudaMemcpyHostToDevice));
  std::vector<float2> tw(1024);
  for (int k1 = 0; k1 < 32; ++k1)
    for (int l = 0; l < 32; ++l) {
      const double a = 2.0 * M_PI * (double)(l * k1) / 1024.0;
      tw[k1 * 32 + l] = make_float2((float)cos(a), (float)sin(a));
    }
  AW_CUDA(cudaMalloc(&ctx->d_twiddle, 1024 * sizeof(float2)));
  AW_CUDA(cudaMemcpy(ctx->d_twiddle, tw.data(), 1024 * sizeof(float2), cudaMemcpyHostToDevice));
  std::vector<float> env(512);           // [0,256): envelope, [256,512): its reciprocal
  for (int j = 0; j < 256; ++j) {
    float e = 0.f;                       // same order as ola_envelope: ascending frame index
    for (int r = 3; r >= 0; --r) e = fmaf(model->window[j + 256 * r], model->window[j + 256 * r], e);
    env[j] = e;
    env[256 + j] = 1.0f / e;
  }
  AW_CUDA(cudaMalloc(&ctx->d_env256, 512 * 4));
  AW_CUDA(cudaMemcpy(ctx->d_env256, env.data(), 512 * 4, cudaMemcpyHostToDevice));
  AW_CUDA(cudaStreamCreateWithFlags(&ctx->gstream, cudaStreamNonBlocking));
  AW_CUDA(cudaEventCreateWithFlags(&ctx->ev_in, cudaEventDisableTiming));
  AW_CUDA(cudaEventCreateWithFlags(&ctx->ev_out, cudaEventDisableTiming));
  *out = ctx;
  return 0;
}

static std::vector<Buf*> all_bufs(aw_ctx* ctx) {
  return {&ctx->accum, &ctx->peakx, &ctx->mag, &ctx->ph_u, &ctx->ph_q, &ctx->c0, &ctx->c,
                 &ctx->m, &ctx->v, &ctx->cbest, &ctx->dA, &ctx->yoob, &ctx->y, &ctx->M,
                 &ctx->cs, &ctx->sigma, &ctx->act[0], &ctx->act[1], &ctx->act[2], &ctx->act[3],
                 &ctx->act[4], &ctx->ga, &ctx->gb, &ctx->dh4, &ctx->dp0, &ctx->part, &ctx->stat[0],
                 &ctx->stat[1], &ctx->stat[2], &ctx->stat[3], &ctx->stat[4], &ctx->bstat,
                 &ctx->values, &ctx->best, &ctx->improved, &ctx->pattern, &ctx->itc, &ctx->steps,
                 &ctx->scal, &ctx->zoob, &ctx->p0coef, &ctx->p0scal, &ctx->hpart, &ctx->hcoef, &ctx->red_a, &ctx->red_b, &ctx->red_c,
                 &ctx->gsc, &ctx->nonfinite, &ctx->smax, &ctx->lowm, &ctx->tc_X, &ctx->tc_dS, &ctx->tc_soob,
                 &ctx->tc_dX, &ctx->tc_gedge, &ctx->tc_dmax, &ctx->tc_ones, &ctx->stoi_ws,
                 &ctx->conv_x, &ctx->conv_idx};
}

extern "C" int aw_ctx_destroy(aw_ctx* ctx) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  for (int l = 0; l < 4; ++l) {
    cudaFree(ctx->d_w[l]);
    cudaFree(ctx->d_wt[l]);
    cudaFree(ctx->d_w16[l]);
    cudaFree(ctx->d_wt16[l]);
    cudaFree(ctx->d_w16h[l]);
    cudaFree(ctx->d_wt16h[l]);
  }
  if (ctx->gstream) cudaStreamDestroy(ctx->gstream);
  if (ctx->ev_in) cudaEventDestroy(ctx->ev_in);
  if (ctx->ev_out) cudaEventDestroy(ctx->ev_out);
  if (ctx->h_lowm) cudaFreeHost(ctx->h_lowm);
  cudaFree(ctx->tcm.peakB); cudaFree(ctx->tcm.compB); cudaFree(ctx->tcm.compBT); cudaFree(ctx->tcm.fix);
  cudaFree(ctx->d_window);
  cudaFree(ctx->d_twiddle);
  cudaFree(ctx->d_env256);
  for (auto& mc : ctx->mels) {
    cudaFree(mc.rowptr); cudaFree(mc.col); cudaFree(mc.val);
    cudaFree(mc.colptr); cudaFree(mc.row); cudaFree(mc.valT);
  }
  for (Buf* b : all_bufs(ctx))
    if (b->p) cudaFree(b->p);
  delete ctx;
  return 0;
}

extern "C" int aw_ctx_set_precision(aw_ctx* ctx, int prec) {
  AW_REQUIRE(ctx, "null ctx");
  if (ctx) cudaSetDevice(ctx->device);
  AW_REQUIRE(prec == AW_PREC_TF32 || prec == AW_PREC_FP32 || prec == AW_PREC_BF16 || prec == AW_PREC_FP16,
             "unknown precision %d", prec);
  ctx->prec = prec;
  return 0;
}

extern "C" int64_t aw_launch_count(aw_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int aw_ctx_set_option(aw_ctx* ctx, int option, double value) {
  AW_REQUIRE(ctx, "null ctx");
  switch (option) {
    case AW_OPT_THRESHOLD: ctx->threshold = (float)value; return 0;
    case AW_OPT_EXACT_MARGIN:
      AW_REQUIRE(value >= 0.0, "aw_ctx_set_option: margin must be >= 0");
      ctx->exact_margin = value;
      return 0;
    case AW_OPT_TC_SPECTRAL:
      ctx->tc_spec = value != 0.0;
      if (value > 1.0) ctx->tc_min_frames = (int)value;      // 1 = on with the default batch threshold
      return 0;
    case AW_OPT_TWO_PASS: ctx->two_pass = value != 0.0; return 0;
    case AW_OPT_PAIR_GEMM: ctx->pair_gemm = value != 0.0; return 0;
    case AW_OPT_BWD64_STREAM: ctx->bwd64_stream = value != 0.0; return 0;
    default: return set_error("aw_ctx_set_option: unknown option %d", option);
  }
}

extern "C" int aw_ctx_get_stat(aw_ctx* ctx, int which, int64_t* out) {
  AW_REQUIRE(ctx && out, "null argument");
  switch (which) {
    case AW_STAT_DETECT_CLIPS: *out = ctx->stat_detect_clips; return 0;
    case AW_STAT_REEVAL_CLIPS: *out = ctx->stat_reeval_clips; return 0;
    default: return set_error("aw_ctx_get_stat: unknown statistic %d", which);
  }
}

// per-clip flags of the last aw_embed_batch call: 1 = a non-finite gradient was met (its NAdam
// update was skipped); a reduced-precision loop that flags a clip should be re-run in TF32
extern "C" int aw_embed_status(aw_ctx* ctx, int32_t* d_flags, int n_clips, void* stream) {
  AW_REQUIRE(ctx && d_flags, "null argument");
  AW_REQUIRE(n_clips == ctx->last_embed_clips && ctx->nonfinite.p, "aw_embed_status: last embed had %d clips, asked for %d",
             ctx->last_embed_clips, n_clips);
  cudaSetDevice(ctx->device);
  AW_CUDA(cudaMemcpyAsync(d_flags, ctx->nonfinite.p, (size_t)n_clips * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

extern "C" int aw_profile_enable(aw_ctx* ctx, int on) {
  AW_REQUIRE(ctx, "null ctx");
  if (ctx) cudaSetDevice(ctx->device);
  ctx->prof_on = on != 0;
  return 0;
}

// Sum the recorded tensor-core GEMM launches by (n, k, epilogue); waits for their events.
extern "C" int aw_profile_read(aw_ctx* ctx, int max_classes, int* n_classes, int* cls_n, int* cls_k,
                               int* cls_epi, int64_t* cls_count, double* cls_ms) {
  AW_REQUIRE(ctx && n_classes, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  int nc = 0;
  for (auto& r : ctx->prof) {
    AW_CUDA(cudaEventSynchronize(r.b));
    float ms = 0.f;
    AW_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    int c = 0;
    for (; c < nc; ++c)
      if (cls_n[c] == r.n && cls_k[c] == r.k && cls_epi[c] == r.epi) break;
    if (c == nc) {
      if (nc >= max_classes) continue;
      cls_n[c] = r.n; cls_k[c] = r.k; cls_epi[c] = r.epi; cls_count[c] = 0; cls_ms[c] = 0.0;
      ++nc;
    }
    cls_count[c] += 1;
    cls_ms[c] += ms;
    ctx->ev_pool.push_back(r.a);
    ctx->ev_pool.push_back(r.b);
  }
  ctx->prof.clear();
  *n_classes = nc;
  return 0;
}

// Per-kernel-class device time of everything launched since the last read (every launch is
// bracketed by events on the launching stream).  names: [max_classes][32] chars.
extern "C" int aw_profile_read_named(aw_ctx* ctx, int max_classes, int* n_classes, char* names,
                                     int64_t* cls_count, double* cls_ms) {
  AW_REQUIRE(ctx && n_classes && names && cls_count && cls_ms, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  int nc = 0;
  for (size_t i = 0; i + 1 < ctx->marks.size(); ++i) {
    const aw_ctx::Mark& a = ctx->marks[i];
    if (!a.label) continue;
    AW_CUDA(cudaEventSynchronize(ctx->marks[i + 1].e));
    float ms = 0.f;
    AW_CUDA(cudaEventElapsedTime(&ms, a.e, ctx->marks[i + 1].e));
    int c = 0;
    for (; c < nc; ++c)
      if (strncmp(names + 32 * c, a.label, 31) == 0) break;
    if (c == nc) {
      if (nc >= max_classes) continue;
      strncpy(names + 32 * c, a.label, 31);
      names[32 * c + 31] = 0;
      cls_count[c] = 0; cls_ms[c] = 0.0;
      ++nc;
    }
    cls_count[c] += 1;
    cls_ms[c] += ms;
  }
  for (auto& m : ctx->marks) ctx->ev_pool.push_back(m.e);
  ctx->marks.clear();
  *n_classes = nc;
  return 0;
}

// embedding/multibit_embedder.py:43-47: bins k with band_lo <= k*sr/1024 <= band_hi,
// frequencies evaluated like np.fft.rfftfreq (k * (sr / 1024) in float64).
extern "C" int aw_band_bins(aw_ctx* ctx, int sample_rate, int* bin0, int* nbins) {
  AW_REQUIRE(ctx && bin0 && nbins, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  int lo = -1, hi = -1;
  const double val = 1.0 / (1024.0 * (1.0 / sample_rate));
  for (int k = 0; k <= 512; ++k) {
    const double f = k * val;
    if (f >= ctx->band_lo && f <= ctx->band_hi) {
      if (lo < 0) lo = k;
      hi = k;
    }
  }
  AW_REQUIRE(lo >= 1 && hi <= 511 && hi - lo + 1 <= AW_MAX_BINS,
             "embedding band [%g,%g] Hz at %d Hz maps to unsupported bins [%d,%d]", ctx->band_lo,
             ctx->band_hi, sample_rate, lo, hi);
  *bin0 = lo;
  *nbins = hi - lo + 1;
  return 0;
}

static int get_mel(aw_ctx* ctx, int bin0, int nbins, SparseMel* out) {
  for (auto& mc : ctx->mels)
    if (mc.bin0 == bin0 && mc.nbins == nbins) {
      *out = SparseMel{mc.rowptr, mc.col, mc.val, mc.colptr, mc.row, mc.valT};
      return 0;
    }
  std::vector<int> rowptr(AW_NMEL + 1, 0), col, colptr(nbins + 1, 0), row;
  std::vector<float> val, valT;
  for (int c = 0; c < AW_NMEL; ++c) {
    for (int b = 0; b < nbins; ++b) {
      const float w = ctx->h_mel[(size_t)c * 513 + bin0 + b];
      if (w != 0.f) { col.push_back(b); val.push_back(w); }
    }
    rowptr[c + 1] = (int)col.size();
  }
  for (int b = 0; b < nbins; ++b) {
    for (int c = 0; c < AW_NMEL; ++c) {
      const float w = ctx->h_mel[(size_t)c * 513 + bin0 + b];
      if (w != 0.f) { row.push_back(c); valT.push_back(w); }
    }
    colptr[b + 1] = (int)row.size();
  }
  MelCfg mc;
  mc.bin0 = bin0; mc.nbins = nbins; mc.nnz = (int)col.size();
  const size_t nz = col.size() ? col.size() : 1;
  AW_CUDA(cudaMalloc(&mc.rowptr, rowptr.size() * 4));
  AW_CUDA(cudaMalloc(&mc.col, nz * 4));
  AW_CUDA(cudaMalloc(&mc.val, nz * 4));
  AW_CUDA(cudaMalloc(&mc.colptr, colptr.size() * 4));
  AW_CUDA(cudaMalloc(&mc.row, nz * 4));
  AW_CUDA(cudaMalloc(&mc.valT, nz * 4));
  AW_CUDA(cudaMemcpy(mc.rowptr, rowptr.data(), rowptr.size() * 4, cudaMemcpyHostToDevice));
  AW_CUDA(cudaMemcpy(mc.colptr, colptr.data(), colptr.size() * 4, cudaMemcpyHostToDevice));
  if (!col.empty()) {
    AW_CUDA(cudaMemcpy(mc.col, col.data(), col.size() * 4, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(mc.val, val.data(), val.size() * 4, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(mc.row, row.data(), row.size() * 4, cudaMemcpyHostToDevice));
    AW_CUDA(cudaMemcpy(mc.valT, valT.data(), valT.size() * 4, cudaMemcpyHostToDevice));
  }
  ctx->mels.push_back(mc);
  *out = SparseMel{mc.rowptr, mc.col, mc.val, mc.colptr, mc.row, mc.valT};
  return 0;
}

// ---------------------------------------------------------------------------
// workspace
// ---------------------------------------------------------------------------
struct Dims {
  int n, N, T, L, Tp, Tp_pad, tiles, rows, bin0, nb;
  int T_clip, Tp_clip;   // frames / pooled frames per-clip statistics divide by: the whole clip's, also for a shard
};

static void set_frames(Dims* d, int T) {
  d->T = T;
  d->L = AW_HOP * (T - 1);
  d->Tp = T / 2;
  d->Tp_pad = (d->Tp + AW_ROW_TILE - 1) / AW_ROW_TILE * AW_ROW_TILE;
  d->tiles = d->Tp_pad / AW_ROW_TILE;
  d->rows = d->n * d->Tp_pad;
  d->T_clip = T;
  d->Tp_clip = d->Tp;
}

static int make_dims(aw_ctx* ctx, int n, int N, int sr, Dims* d) {
  AW_REQUIRE(n >= 1, "n_clips must be >= 1");
  AW_REQUIRE(N > 1024, "clips must be longer than 1024 samples (got %d)", N);
  d->n = n; d->N = N;
  set_frames(d, 1 + N / AW_HOP);
  return aw_band_bins(ctx, sr, &d->bin0, &d->nb);
}

// per-clip peak of the synthesised waveform (u64 atomicMax, order independent) is the only
// accumulator cleared per pass; every sum is a per-block partial reduced in fixed order.
struct Acc {
  unsigned long long* peak_y; double* s2_part; double* chan_part; double* bpart;
  int mel_blocks, syn_tiles, p0b_blocks;
};
static Acc acc_view(aw_ctx* ctx, const struct Dims& d);

__global__ void k_iter_begin(unsigned long long* peak, int n, int* it, unsigned* dmax = nullptr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) peak[i] = 0ull;
  if (i < n && dmax) dmax[i] = 0u;
  if (i == 0 && it) *it += 1;
}
__global__ void k_fill_u64(unsigned long long* p, unsigned long long v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

static int mel_blocks(const Dims& d) { return (d.T + AW_MEL_FRAMES - 1) / AW_MEL_FRAMES; }
static int syn_tiles(const Dims& d) { return (d.T + 3 + AW_SYN_HOPS - 1) / AW_SYN_HOPS; }
static int p0b_blocks(const Dims& d) { return (2 * d.Tp + AW_P0B_FRAMES - 1) / AW_P0B_FRAMES; }
static int p0a_blocks(const Dims& d) { return (d.T + AW_P0A_FRAMES - 1) / AW_P0A_FRAMES; }
static int s2_slots(const Dims& d) { return p0a_blocks(d); }
static size_t acc_doubles(const Dims& d) {
  return (size_t)d.n * (1 + s2_slots(d) + 256 * (size_t)mel_blocks(d) + 256 * (size_t)p0b_blocks(d)) + 1;   // + alignment pad
}
static Acc acc_view(aw_ctx* ctx, const Dims& d) {
  Acc a;
  a.mel_blocks = mel_blocks(d); a.syn_tiles = syn_tiles(d); a.p0b_blocks = p0b_blocks(d);
  double* base = (double*)ctx->accum.p;
  a.peak_y = (unsigned long long*)base;
  a.s2_part = base + d.n;
  // (sum, sum of squares) pairs are read as double2: 16-byte aligned
  a.chan_part = base + (((size_t)d.n * (1 + s2_slots(d)) + 1) & ~(size_t)1);
  a.bpart = a.chan_part + (size_t)d.n * 256 * a.mel_blocks;
  return a;
}

// ds: the frames the spectra span, d: the frames the detector net runs on (the same dims for whole
// clips; a shard's segment and its own frames)
static int ensure_net_ws(aw_ctx* ctx, const Dims& ds, const Dims& d, bool backward) {
  const size_t n = d.n, R = d.rows;
  if (ensure(ctx->accum, acc_doubles(ds) * 8)) return 1;
  if (ensure(ctx->peakx, n * 8)) return 1;
  if (ensure(ctx->mag, n * ds.T * ds.nb * 4)) return 1;
  if (ensure(ctx->M, n * d.T * AW_NMEL * 4)) return 1;
  if (ensure(ctx->cs, n * AW_NMEL * sizeof(ChanStats))) return 1;
  if (ensure(ctx->sigma, n * 4)) return 1;
  if (ensure(ctx->hpart, n * d.tiles * 64 * 3 * sizeof(double)) || ensure(ctx->hcoef, n * 64 * 4 * sizeof(float))) return 1;
  if (ensure(ctx->p0coef, n * AW_NMEL * sizeof(P0BwdCoef)) || ensure(ctx->p0scal, n * sizeof(P0BwdScal))) return 1;
  bool remap = false;
  for (int l = 0; l < 5; ++l) {
    void* before = ctx->act[l].p;
    if (ensure(ctx->act[l], R * kCp[l] * 4)) return 1;
    if (ensure(ctx->stat[l], n * kCp[l] * 2 * 4)) return 1;
    remap |= before != ctx->act[l].p;
  }
  if (ensure(ctx->part, (R / 128) * 1024 * 2 * 4)) return 1;
  if (ensure(ctx->values, n * AW_NBITS * 4)) return 1;
  if (ensure(ctx->best, n * 4)) return 1;
  if (ensure(ctx->improved, n * 4)) return 1;
  if (ensure(ctx->itc, 4)) return 1;
  if (ensure(ctx->gsc, n * 4)) return 1;
  if (backward) {
    void *b0 = ctx->ga.p, *b1 = ctx->gb.p, *b2 = ctx->dh4.p;
    if (ensure(ctx->ga, R * 1024 * 4)) return 1;
    if (ensure(ctx->gb, R * 1024 * 4)) return 1;
    if (ensure(ctx->dh4, R * 64 * 4)) return 1;
    if (ensure(ctx->dp0, R * 128 * 4)) return 1;
    if (ensure(ctx->bstat, n * 1024 * 2 * 4)) return 1;
    remap |= b0 != ctx->ga.p || b1 != ctx->gb.p || b2 != ctx->dh4.p;
  }
  if (remap || ctx->ws_rows != d.rows) {
    for (int b = 0; b < 2; ++b) {
      for (int l = 0; l < 4; ++l)
        if (make_map(ctx, &ctx->tm_act[b][l], ctx->act[l].p, R, kCp[l], 128, b)) return 1;
      if (ctx->ga.p) {
        if (make_map(ctx, &ctx->tm_dh4[b], ctx->dh4.p, R, 64, 128, b)) return 1;
        if (make_map(ctx, &ctx->tm_ga1024[b], ctx->ga.p, R, 1024, 128, b)) return 1;
        if (make_map(ctx, &ctx->tm_ga512[b], ctx->ga.p, R, 512, 128, b)) return 1;
        if (make_map(ctx, &ctx->tm_gb1024[b], ctx->gb.p, R, 1024, 128, b)) return 1;
      }
    }
    ctx->ws_rows = d.rows;
  }
  return 0;
}

// ---------------------------------------------------------------------------
// detector forward from band magnitudes (ctx->mag) to values (+ optional backward seed)
// ---------------------------------------------------------------------------
// AT = activation storage type: float (fp32 / TF32 modes) or bf16 (bf16 mode)
template <typename AT, int EPI>
static int gemm_layer(aw_ctx* ctx, const CUtensorMap& ma, const void* a, const CUtensorMap& mb,
                      const void* b, int rows, int n, int k, const EpiArgsT<AT>& ep, cudaStream_t st);

template <>
int gemm_layer<float, EPI_FWD>(aw_ctx* ctx, const CUtensorMap& ma, const void* a, const CUtensorMap& mb,
                               const void* b, int rows, int n, int k, const EpiArgsT<float>& ep, cudaStream_t st) {
  if (ctx->prec == AW_PREC_FP32) return launch_exact<EPI_FWD>(ctx, (const float*)a, (const float*)b, rows, n, k, ep, st);
  return launch_tc_bn<float, float, EPI_FWD>(ctx, ma, mb, rows, n, k, ep, st);
}
template <>
int gemm_layer<float, EPI_BWD>(aw_ctx* ctx, const CUtensorMap& ma, const void* a, const CUtensorMap& mb,
                               const void* b, int rows, int n, int k, const EpiArgsT<float>& ep, cudaStream_t st) {
  if (ctx->prec == AW_PREC_FP32) return launch_exact<EPI_BWD>(ctx, (const float*)a, (const float*)b, rows, n, k, ep, st);
  return launch_tc_bn<float, float, EPI_BWD>(ctx, ma, mb, rows, n, k, ep, st);
}
template <>
int gemm_layer<__nv_bfloat16, EPI_FWD>(aw_ctx* ctx, const CUtensorMap& ma, const void*, const CUtensorMap& mb,
                                       const void*, int rows, int n, int k, const EpiArgsT<__nv_bfloat16>& ep,
                                       cudaStream_t st) {
  if (n >= 256) return launch_tc<__nv_bfloat16, __nv_bfloat16, 256, EPI_FWD>(ctx, ma, mb, rows, n, k, ep, st);
  return launch_tc<__nv_bfloat16, __nv_bfloat16, 64, EPI_FWD>(ctx, ma, mb, rows, n, k, ep, st);
}
template <>
int gemm_layer<__nv_bfloat16, EPI_BWD>(aw_ctx* ctx, const CUtensorMap& ma, const void*, const CUtensorMap& mb,
                                       const void*, int rows, int n, int k, const EpiArgsT<__nv_bfloat16>& ep,
                                       cudaStream_t st) {
  return launch_tc<__nv_bfloat16, __nv_bfloat16, 256, EPI_BWD>(ctx, ma, mb, rows, n, k, ep, st);
}

template <>
int gemm_layer<__half, EPI_FWD>(aw_ctx* ctx, const CUtensorMap& ma, const void*, const CUtensorMap& mb,
                                const void*, int rows, int n, int k, const EpiArgsT<__half>& ep, cudaStream_t st) {
  if (n >= 256) return launch_tc<__half, __half, 256, EPI_FWD>(ctx, ma, mb, rows, n, k, ep, st);
  return launch_tc<__half, __half, 64, EPI_FWD>(ctx, ma, mb, rows, n, k, ep, st);
}
template <>
int gemm_layer<__half, EPI_BWD>(aw_ctx* ctx, const CUtensorMap& ma, const void*, const CUtensorMap& mb,
                                const void*, int rows, int n, int k, const EpiArgsT<__half>& ep, cudaStream_t st) {
  return launch_tc<__half, __half, 256, EPI_BWD>(ctx, ma, mb, rows, n, k, ep, st);
}

// B: activation tensor-map view (0 = 4-byte, 1 = 2-byte elements); weight copies per type
template <typename AT> struct ModeOf {
  static constexpr int B = 0;
  static const CUtensorMap& w(aw_ctx* c, int l) { return c->tm_w[l]; }
  static const CUtensorMap& wP(aw_ctx* c, int l) { return c->tm_w_p[l]; }
  static const CUtensorMap& wt(aw_ctx* c, int l) { return c->tm_wt[l]; }
  static const CUtensorMap& wtP(aw_ctx* c, int l) { return c->tm_wt_p[l]; }
  static const void* wp(aw_ctx* c, int l) { return c->d_w[l]; }
  static const void* wtp(aw_ctx* c, int l) { return c->d_wt[l]; }
  static constexpr float GSCALE = 1.0f;
};
template <> struct ModeOf<__nv_bfloat16> {
  static constexpr int B = 1;
  static const CUtensorMap& w(aw_ctx* c, int l) { return c->tm_w16[l]; }
  static const CUtensorMap& wP(aw_ctx* c, int l) { return c->tm_w16_p[l]; }
  static const CUtensorMap& wt(aw_ctx* c, int l) { return c->tm_wt16[l]; }
  static const CUtensorMap& wtP(aw_ctx* c, int l) { return c->tm_wt16_p[l]; }
  static const void* wp(aw_ctx* c, int l) { return c->d_w16[l]; }
  static const void* wtp(aw_ctx* c, int l) { return c->d_wt16[l]; }
  static constexpr float GSCALE = 1.0f;
};
template <> struct ModeOf<__half> {
  static constexpr int B = 1;
  static const CUtensorMap& w(aw_ctx* c, int l) { return c->tm_w16h[l]; }
  static const CUtensorMap& wP(aw_ctx* c, int l) { return c->tm_w16h_p[l]; }
  static const CUtensorMap& wt(aw_ctx* c, int l) { return c->tm_wt16h[l]; }
  static const CUtensorMap& wtP(aw_ctx* c, int l) { return c->tm_wt16h_p[l]; }
  static const void* wp(aw_ctx* c, int l) { return c->d_w16h[l]; }
  static const void* wtp(aw_ctx* c, int l) { return c->d_wt16h[l]; }
  // gradients are ~1e-4 .. 1e-8 at T' = 861, shrink like 1/T' (the head seeds dz / T') and shrink
  // further as tanh saturates: k_head_final picks a per-clip power-of-two loss scale every
  // iteration that puts the largest seeded dz at 0.5 (removed again where dP0 is consumed)
  static constexpr float GSCALE = 4096.0f;
};
// target magnitude of the seeded gradient for the per-clip power-of-two loss scale that
// k_head_final chooses every iteration (0 = no scaling: fp32 / TF32 / bf16 storage)
template <typename AT>
static float grad_target() { return ModeOf<AT>::GSCALE == 1.0f ? 0.0f : 0.5f; }

// spectra are stored for the whole (halo-extended) segment; the detector net runs on the own frames
static float* own_frames(aw_ctx* ctx, float* base, int nb) {
  return ctx->sh ? base + (size_t)ctx->sh->own_lo * nb : base;
}
// frame-sharded InstanceNorm statistics: local raw sums -> all-reduce -> (mean, rstd) / adjoint means
template <bool BWD>
static int sh_finalize(aw_ctx* ctx, const Dims& d, int C, float* stat, cudaStream_t st) {
  double* red = (double*)((uint8_t*)ctx->sh->comm.d_arena + AW_ARENA_RED);
  k_finalize<2><<<dim3((C + 31) / 32, 1), 256, 0, st>>>((float*)ctx->part.p, C, d.tiles, C, 1, nullptr, red);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  if (sh_allreduce(ctx, 2 * (int64_t)C, AW_COMM_F64, AW_COMM_SUM, st)) return 1;
  k_stat_from_sums<BWD><<<dim3((C + 255) / 256, 1), 256, 0, st>>>(red, C, d.Tp_clip, stat);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

template <typename AT>
static int net_forward(aw_ctx* ctx, const Dims& d, const Acc& acc, const SparseMel& sm,
                       cudaStream_t st, const unsigned long long* peak_scale = nullptr) {
  constexpr int B = ModeOf<AT>::B;
  const int tf = ctx->prec == AW_PREC_TF32;
  {
    dim3 g((d.T + AW_MEL_FRAMES - 1) / AW_MEL_FRAMES, d.n);
    prof_mark(ctx, st, "mel");
    k_mel<<<g, 128, AW_MEL_FRAMES * d.nb * 4, st>>>(own_frames(ctx, (float*)ctx->mag.p, d.nb), d.T, d.nb, sm,
                                                    (float*)ctx->M.p, acc.chan_part, peak_scale);
    ctx->launches++;
    AW_LAUNCH_CHECK();
    dim3 g2((d.Tp_pad + AW_P0_ROWS - 1) / AW_P0_ROWS, d.n);
    const double* cp = acc.chan_part;
    int cb = acc.mel_blocks;
    if (clip_sums(ctx, ctx->red_a, cp, cb, d.n, 2 * AW_NMEL, st)) return 1;   // channel sums over the WHOLE clip
    prof_mark(ctx, st, "mel_stats");
    k_mel_stats<<<d.n, 128, 0, st>>>(cp, cb, d.T_clip, (ChanStats*)ctx->cs.p, (float*)ctx->sigma.p);
    ctx->launches++;
    AW_LAUNCH_CHECK();
    prof_mark(ctx, st, "p0");
    k_p0<AT><<<g2, 128, 0, st>>>((float*)ctx->M.p, d.T, d.Tp, d.Tp_pad, (ChanStats*)ctx->cs.p,
                                 (float*)ctx->sigma.p, (AT*)ctx->act[0].p, tf);
    ctx->launches++;
    AW_LAUNCH_CHECK();
  }
  for (int l = 0; l < 4; ++l) {
    const int cin = kCp[l], cout = kCp[l + 1];
    EpiArgsT<AT> ep{};
    ep.out = (AT*)ctx->act[l + 1].p; ep.ldo = cout;
    ep.part = (float*)ctx->part.p; ep.ldp = cout; ep.act = nullptr;
    const CUtensorMap& mw = ModeOf<AT>::w(ctx, l);
    const void* w = ModeOf<AT>::wp(ctx, l);
    // layer 0 (K = 128): the GEMM (30 GFLOP at 256 clips) is cheaper than one round trip of its 235 MB
    // output, so it runs twice -- column sums only, then again with InstanceNorm + LeakyReLU applied in
    // the epilogue -- and the raw H1 never exists (exact fp32 mode keeps the one-pass form)
    const bool two_pass = l == 0 && ctx->prec != AW_PREC_FP32 && ctx->two_pass;
    if (two_pass) {
      if (launch_tc<AT, AT, 256, EPI_FWD_STATS>(ctx, ctx->tm_act[B][l], mw, d.rows, cout, cin, ep, st)) return 1;
    } else if (ctx->prec != AW_PREC_FP32 && pair_ok(ctx, d.rows, cout, cin, (int)sizeof(AT))) {
      if (launch_tc_pair<AT, AT, EPI_FWD>(ctx, ctx->tm_act[B][l], ModeOf<AT>::wP(ctx, l), d.rows, cout, cin, ep, st))
        return 1;
    } else if (gemm_layer<AT, EPI_FWD>(ctx, ctx->tm_act[B][l], ctx->act[l].p, mw, w, d.rows, cout, cin, ep, st))
      return 1;
    dim3 g((cout + 31) / 32, d.n);
    prof_mark(ctx, st, "finalize_fwd");
    if (ctx->sh) {
      if (sh_finalize<false>(ctx, d, cout, (float*)ctx->stat[l + 1].p, st)) return 1;
    } else {
      if (d.tiles <= 16)
        k_finalize_small<0><<<dim3((cout + 255) / 256, d.n), 256, 0, st>>>((float*)ctx->part.p, cout, d.tiles, cout,
                                                                           d.Tp, (float*)ctx->stat[l + 1].p);
      else
        k_finalize<0><<<g, 256, 0, st>>>((float*)ctx->part.p, cout, d.tiles, cout, d.Tp,
                                         (float*)ctx->stat[l + 1].p, nullptr);
      ctx->launches++;
      AW_LAUNCH_CHECK();
    }
    if (two_pass) {
      ep.stat = (float*)ctx->stat[l + 1].p; ep.tiles_per_clip = d.tiles; ep.Tp = d.Tp; ep.round_tf32 = tf && l < 3;
      if (launch_tc<AT, AT, 256, EPI_FWD_APPLY>(ctx, ctx->tm_act[B][l], mw, d.rows, cout, cin, ep, st)) return 1;
      continue;
    }
    prof_mark(ctx, st, "norm_act");
    {
      const int rl = 128 / std::min(128, cout / Vec16<AT>::N);       // row lanes per block (narrow layers)
      dim3 gn((d.Tp_pad + AW_NORM_ROWS * rl - 1) / (AW_NORM_ROWS * rl), (cout / Vec16<AT>::N + 127) / 128, d.n);
      k_norm_rows<AT, NORM_FWD><<<gn, 128, 0, st>>>((AT*)ctx->act[l + 1].p, nullptr, cout, d.Tp, d.Tp_pad,
                                                    (float*)ctx->stat[l + 1].p, nullptr, tf && l < 3);
    }
    ctx->launches++;
    AW_LAUNCH_CHECK();
  }
  return 0;
}

template <typename AT>
static int net_backward(aw_ctx* ctx, const Dims& d, const Acc& acc, const SparseMel& sm,
                        cudaStream_t st, bool euler_s2 = false) {
  constexpr int B = ModeOf<AT>::B;
  const int tf = ctx->prec == AW_PREC_TF32;
  AT* ga = (AT*)ctx->ga.p;
  AT* gb = (AT*)ctx->gb.p;
  struct Step { const CUtensorMap* ma; const AT* a; int l; AT* out; };
  // l = index of the weight matrix: dP_l = dH_{l+1} * W_l
  const Step steps[3] = {{&ctx->tm_dh4[B], (AT*)ctx->dh4.p, 3, ga},
                         {&ctx->tm_ga1024[B], ga, 2, gb},
                         {&ctx->tm_gb1024[B], gb, 1, ga}};
  for (int s = 0; s < 3; ++s) {
    const int l = steps[s].l, k = kCp[l + 1], n = kCp[l];
    EpiArgsT<AT> ep{};
    ep.out = steps[s].out; ep.ldo = n;
    ep.part = (float*)ctx->part.p; ep.ldp = n; ep.act = (AT*)ctx->act[l].p;
    const CUtensorMap& mw = ModeOf<AT>::wt(ctx, l);
    const void* w = ModeOf<AT>::wtp(ctx, l);
    // dP3 = dH4 W3 has K = 64: recomputing it is cheaper than writing dHhat3 (470 MB at 256 clips) and
    // reading it back for the InstanceNorm adjoint -- statistics pass, then a pass that applies the adjoint
    const bool two_pass = s == 0 && ctx->prec != AW_PREC_FP32 && ctx->two_pass;
    // 16-bit loops: that layer on the streaming kernel (activations through a TMA ring, no epilogue loads)
    const bool stream64 = two_pass && sizeof(AT) == 2 && ctx->bwd64_stream;
    Gemm64Args g64;
    memset(&g64, 0, sizeof(g64));
    g64.part = (float*)ctx->part.p; g64.ldp = n; g64.ldo = n; g64.tiles_per_clip = d.tiles; g64.Tp = d.Tp;
    g64.stat = (float*)ctx->stat[l].p; g64.bstat = (float*)ctx->bstat.p;
    if (stream64) {
      if constexpr (sizeof(AT) == 2) {
        if (launch_bwd64<AT, EPI_BWD_STATS>(ctx, *steps[s].ma, ModeOf<AT>::wtP(ctx, l), ctx->tm_act[B][l], ctx->tm_ga1024[B],
                                            d.rows, n, k, g64, st))
          return 1;
      }
    } else if (two_pass) {
      if (launch_tc<AT, AT, 256, EPI_BWD_STATS>(ctx, *steps[s].ma, mw, d.rows, n, k, ep, st)) return 1;
    } else if (ctx->prec != AW_PREC_FP32 && pair_ok(ctx, d.rows, n, k, (int)sizeof(AT))) {
      if (launch_tc_pair<AT, AT, EPI_BWD>(ctx, *steps[s].ma, ModeOf<AT>::wtP(ctx, l), d.rows, n, k, ep, st)) return 1;
    } else if (gemm_layer<AT, EPI_BWD>(ctx, *steps[s].ma, steps[s].a, mw, w, d.rows, n, k, ep, st)) return 1;
    dim3 g((n + 31) / 32, d.n);
    prof_mark(ctx, st, "finalize_bwd");
    if (ctx->sh) {
      if (sh_finalize<true>(ctx, d, n, (float*)ctx->bstat.p, st)) return 1;
    } else {
      if (d.tiles <= 16)
        k_finalize_small<1><<<dim3((n + 255) / 256, d.n), 256, 0, st>>>((float*)ctx->part.p, n, d.tiles, n, d.Tp,
                                                                        (float*)ctx->bstat.p);
      else
        k_finalize<1><<<g, 256, 0, st>>>((float*)ctx->part.p, n, d.tiles, n, d.Tp,
                                         (float*)ctx->bstat.p, nullptr);
      ctx->launches++;
      AW_LAUNCH_CHECK();
    }
    if (stream64) {
      if constexpr (sizeof(AT) == 2) {
        if (launch_bwd64<AT, EPI_BWD_APPLY>(ctx, *steps[s].ma, ModeOf<AT>::wtP(ctx, l), ctx->tm_act[B][l], ctx->tm_ga1024[B],
                                            d.rows, n, k, g64, st))
          return 1;
      }
      continue;
    }
    if (two_pass) {
      ep.stat = (float*)ctx->stat[l].p; ep.bstat = (float*)ctx->bstat.p;
      ep.tiles_per_clip = d.tiles; ep.Tp = d.Tp; ep.round_tf32 = tf;
      if (launch_tc<AT, AT, 256, EPI_BWD_APPLY>(ctx, *steps[s].ma, mw, d.rows, n, k, ep, st)) return 1;
      continue;
    }
    prof_mark(ctx, st, "in_bwd_apply");
    {
      const int rl = 128 / std::min(128, n / Vec16<AT>::N);
      dim3 gn((d.Tp_pad + AW_NORM_ROWS * rl - 1) / (AW_NORM_ROWS * rl), (n / Vec16<AT>::N + 127) / 128, d.n);
      k_norm_rows<AT, NORM_BWD><<<gn, 128, 0, st>>>(steps[s].out, (AT*)ctx->act[l].p, n, d.Tp, d.Tp_pad,
                                                    (float*)ctx->stat[l].p, (float*)ctx->bstat.p, tf);
    }
    ctx->launches++;
    AW_LAUNCH_CHECK();
  }
  {
    // dP0 = dH1 * W0 stays float32 (128 columns; feeds the fp32 front-end adjoints)
    EpiArgsT<float> ep;
    memset(&ep, 0, sizeof(ep));
    ep.out = (float*)ctx->dp0.p; ep.ldo = 128;
    ep.part = nullptr; ep.ldp = 0; ep.act = nullptr;
    if (B) {
      if (launch_tc<AT, float, 128, EPI_PLAIN>(ctx, ctx->tm_ga512[1], ModeOf<AT>::wt(ctx, 0), d.rows, 128, 512, ep, st))
        return 1;
    } else if (ctx->prec == AW_PREC_FP32) {
      if (launch_exact<EPI_PLAIN>(ctx, (const float*)ga, ctx->d_wt[0], d.rows, 128, 512, ep, st)) return 1;
    } else {
      if (launch_tc<float, float, 128, EPI_PLAIN>(ctx, ctx->tm_ga512[0], ctx->tm_wt[0], d.rows, 128, 512, ep, st))
        return 1;
    }
  }
  dim3 g1((2 * d.Tp + AW_P0B_FRAMES - 1) / AW_P0B_FRAMES, d.n);
  prof_mark(ctx, st, "p0_bwd_reduce");
  k_p0_bwd_reduce<<<g1, 128, 0, st>>>((float*)ctx->dp0.p, (float*)ctx->M.p, d.T, d.Tp, d.Tp_pad,
                                      (ChanStats*)ctx->cs.p, acc.bpart, (const float*)ctx->gsc.p);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  dim3 g2((d.T + AW_P0A_FRAMES - 1) / AW_P0A_FRAMES, d.n);
  const double* bp = acc.bpart;
  int bb = acc.p0b_blocks;
  if (clip_sums(ctx, ctx->red_b, bp, bb, d.n, 2 * AW_NMEL, st)) return 1;
  prof_mark(ctx, st, "p0_bwd_coef");
  k_p0_bwd_coef<<<d.n, 128, 0, st>>>(bp, bb, d.T_clip, (ChanStats*)ctx->cs.p, (float*)ctx->sigma.p,
                                     (P0BwdCoef*)ctx->p0coef.p, (P0BwdScal*)ctx->p0scal.p);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  prof_mark(ctx, st, "p0_bwd_apply");
  k_p0_bwd_apply<<<g2, 128, 0, st>>>((float*)ctx->dp0.p, (float*)ctx->M.p, d.T, d.Tp, d.Tp_pad,
                                     (ChanStats*)ctx->cs.p, (P0BwdCoef*)ctx->p0coef.p,
                                     (P0BwdScal*)ctx->p0scal.p, sm, d.nb, own_frames(ctx, (float*)ctx->dA.p, d.nb),
                                     euler_s2 ? (const float*)own_frames(ctx, (float*)ctx->mag.p, d.nb) : nullptr, acc.s2_part,
                                     (const float*)ctx->gsc.p);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

template <typename AT>
static int run_head(aw_ctx* ctx, const Dims& d, const float* pattern, float* values, float* losses,
                    int n_total, bool backward, cudaStream_t st) {
  HeadArgs<AT> h;
  h.P4 = (AT*)ctx->act[4].p; h.Tp = d.Tp; h.Tp_pad = d.Tp_pad;
  h.Tp_glob = d.Tp_clip;
  h.stat4 = (float*)ctx->stat[4].p;
  h.pattern = pattern; h.values = values; h.losses = losses;
  h.best = (float*)ctx->best.p; h.improved = (int*)ctx->improved.p;
  h.dH4 = backward ? (AT*)ctx->dh4.p : nullptr;
  h.it_ptr = (int*)ctx->itc.p; h.n_clips = n_total;
  h.round_tf32 = ctx->prec == AW_PREC_TF32;
  h.gscale = grad_target<AT>();
  h.gsc = (float*)ctx->gsc.p;
  h.hpart = (double*)ctx->hpart.p;
  h.hcoef = (float*)ctx->hcoef.p;
  prof_mark(ctx, st, "head");
  k_head_partial<AT><<<dim3(d.tiles, d.n), 256, 0, st>>>(h);
  const double* hp = h.hpart;
  int hb = d.tiles;
  // k_head_final takes any number of tile partials: whole clips pass them on ungrouped
  if (ctx->sh && clip_sums(ctx, ctx->red_a, hp, hb, d.n, 64 * 3, st)) return 1;
  HeadArgs<AT> hf = h;
  hf.hpart = const_cast<double*>(hp);
  k_head_final<AT><<<d.n, 64, 0, st>>>(hf, hb);
  ctx->launches += 2;
  if (backward && pattern) {
    k_head_seed<AT><<<dim3(d.tiles, d.n), 256, 0, st>>>(h);
    ctx->launches++;
  }
  AW_LAUNCH_CHECK();
  return 0;
}

static AnaArgs ana_base(aw_ctx* ctx, const Dims& d) {
  AnaArgs a;
  memset(&a, 0, sizeof(a));
  a.T = d.T; a.bin0 = d.bin0; a.nbins = d.nb;
  a.window = ctx->d_window; a.twiddle = ctx->d_twiddle; a.env256 = ctx->d_env256;
  a.tol_ratio = (float)pow(10.0, -(double)ctx->tol_db / 20.0);
  return a;
}
static SynArgs syn_base(aw_ctx* ctx, const Dims& d) {
  SynArgs s;
  memset(&s, 0, sizeof(s));
  s.T = d.T; s.L = d.L; s.bin0 = d.bin0; s.nbins = d.nb;
  s.window = ctx->d_window; s.twiddle = ctx->d_twiddle; s.env256 = ctx->d_env256;
  return s;
}
template <int MODE, int K2LO, int K2HI>
static int launch_ana_k(aw_ctx* ctx, const Dims& d, const AnaArgs& a, cudaStream_t st) {
  if (raise_smem_limit(ctx, (const void*)k_analysis<MODE, K2LO, K2HI>, AW_ANA_SMEM)) return 1;
  dim3 g((d.T + AW_ANA_FRAMES - 1) / AW_ANA_FRAMES, d.n);
  prof_mark(ctx, st, MODE == ANA_MAG ? "analysis_mag" : "analysis_init");
  k_analysis<MODE, K2LO, K2HI><<<g, 128, AW_ANA_SMEM, st>>>(a);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}
// the band's 32-bin groups select a compile-time specialisation:
// 44.1 kHz (bins 12..92) -> groups 0..2, 16 kHz (bins 32..256) -> groups 1..8, else generic
template <int MODE>
static int launch_ana(aw_ctx* ctx, const Dims& d, const AnaArgs& a, cudaStream_t st) {
  const int lo = d.bin0 >> 5, hi = (d.bin0 + d.nb - 1) >> 5;
  if (hi <= 2) return launch_ana_k<MODE, 0, 2>(ctx, d, a, st);
  if (lo >= 1 && hi <= 8) return launch_ana_k<MODE, 1, 8>(ctx, d, a, st);
  return launch_ana_k<MODE, 0, 15>(ctx, d, a, st);
}
template <int MODE, int K2LO, int K2HI>
static int launch_syn_k(aw_ctx* ctx, const Dims& d, const SynArgs& s, cudaStream_t st) {
  if (raise_smem_limit(ctx, (const void*)k_synthesis<MODE, K2LO, K2HI>, AW_SYN_SMEM)) return 1;
  dim3 g((d.T + 3 + AW_SYN_HOPS - 1) / AW_SYN_HOPS, d.n);
  prof_mark(ctx, st, MODE == SYN_OOB ? "synthesis_oob" : "synthesis_wave");
  k_synthesis<MODE, K2LO, K2HI><<<g, 128, AW_SYN_SMEM, st>>>(s);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}
template <int MODE>
static int launch_syn(aw_ctx* ctx, const Dims& d, const SynArgs& s, cudaStream_t st) {
  const int lo = d.bin0 >> 5, hi = (d.bin0 + d.nb - 1) >> 5;
  if (hi <= 2) return launch_syn_k<MODE, 0, 2>(ctx, d, s, st);
  if (lo >= 1 && hi <= 8) return launch_syn_k<MODE, 1, 8>(ctx, d, s, st);
  return launch_syn_k<MODE, 0, 15>(ctx, d, s, st);
}
template <int MODE, int K2LO, int K2HI>
static int launch_spec_k(aw_ctx* ctx, const Dims& d, SpecArgs& a, cudaStream_t st) {
  if (raise_smem_limit(ctx, (const void*)k_spec<MODE, K2LO, K2HI>, AW_SP_SMEM)) return 1;
  a.n_clips = d.n; a.T = d.T; a.L = d.L; a.bin0 = d.bin0; a.nbins = d.nb;
  a.tiles = (d.T + AW_SP_FA - 1) / AW_SP_FA;
  a.window = ctx->d_window; a.twiddle = ctx->d_twiddle; a.env256 = ctx->d_env256;
  const int items = a.edge_mode ? a.n_clips * 2 : a.n_clips * a.tiles;
  const int grid = std::min(items, 2 * ctx->num_sms);
  prof_mark(ctx, st, a.edge_mode ? (MODE == SPEC_FWD ? "spec_edge_fwd" : "spec_edge_bwd") : (MODE == SPEC_FWD ? "spec_fwd" : "spec_bwd"));
  k_spec<MODE, K2LO, K2HI><<<grid, 32 * AW_SP_WARPS, AW_SP_SMEM, st>>>(a);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}
template <int MODE>
static int launch_spec(aw_ctx* ctx, const Dims& d, SpecArgs& a, cudaStream_t st) {
  const int lo = d.bin0 >> 5, hi = (d.bin0 + d.nb - 1) >> 5;
  if (hi <= 2) return launch_spec_k<MODE, 0, 2>(ctx, d, a, st);
  if (lo >= 1 && hi <= 8) return launch_spec_k<MODE, 1, 8>(ctx, d, a, st);
  return launch_spec_k<MODE, 0, 15>(ctx, d, a, st);
}
__global__ void k_fill_int(int* p, int v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// smax != null: also the signed max of every clip (order-encoded int, see k_peak)
static int launch_peak(aw_ctx* ctx, const float* x, int64_t stride, int n, int n_clips,
                       unsigned long long* peak, cudaStream_t st, int* smax = nullptr) {
  AW_CUDA(cudaMemsetAsync(peak, 0, (size_t)n_clips * 8, st));
  if (smax) {
    k_fill_int<<<(n_clips + 255) / 256, 256, 0, st>>>(smax, INT_MIN, n_clips);
    ctx->launches++;
  }
  dim3 g(std::min((n + 4095) / 4096, std::max(64, 8192 / n_clips)), n_clips);
  prof_mark(ctx, st, "peak");
  k_peak<<<g, 256, 0, st>>>(x, stride, n, peak, smax);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}
static int begin_pass(aw_ctx* ctx, int n, int* it, cudaStream_t st, unsigned* dmax = nullptr) {
  prof_mark(ctx, st, "iter_begin");
  k_iter_begin<<<(n + 255) / 256, 256, 0, st>>>((unsigned long long*)ctx->accum.p, n, it, dmax);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

// f(AT()) with the activation storage type of the context's precision
template <typename F>
static int with_act_type(aw_ctx* ctx, F&& f) {
  if (ctx->prec == AW_PREC_BF16) return f(__nv_bfloat16());
  if (ctx->prec == AW_PREC_FP16) return f(__half());
  return f(float());
}

// ---------------------------------------------------------------------------
// One detector pass over ds.n clips x (or over one shard's segment; see ensure_net_ws for ds / dn).
static int detect_pass(aw_ctx* ctx, const Dims& ds, const Dims& dn, const float* x, int64_t stride, float* d_values,
                       cudaStream_t st) {
  if (ensure_net_ws(ctx, ds, dn, false)) return 1;
  SparseMel sm;
  if (get_mel(ctx, ds.bin0, ds.nb, &sm)) return 1;
  const Acc acc = acc_view(ctx, dn);
  unsigned long long* peak = (unsigned long long*)ctx->peakx.p;
  if (begin_pass(ctx, ds.n, nullptr, st)) return 1;
  if (launch_peak(ctx, x, stride, ds.N, ds.n, peak, st)) return 1;
  if (sync_peak(ctx, peak, st)) return 1;        // waveform.py:19 over the whole clip
  AnaArgs a = ana_base(ctx, ds);
  a.sig = x; a.sig_stride = stride; a.len = ds.N;
  a.peak = peak;
  a.mag = (float*)ctx->mag.p;
  if (launch_ana<ANA_MAG>(ctx, ds, a, st)) return 1;
  return with_act_type(ctx, [&](auto tag) -> int {
    using AT = decltype(tag);
    if (net_forward<AT>(ctx, dn, acc, sm, st)) return 1;
    return run_head<AT>(ctx, dn, nullptr, d_values, nullptr, dn.n, false, st);
  });
}

// flags[0] = number of clips with min_i |v_i - thr| < margin, flags[1 + clip] = 1 for those clips
__global__ void __launch_bounds__(128) k_flag_low_margin(const float* __restrict__ values, float thr, float margin,
                                                         int n_clips, int* __restrict__ flags) {
  const int clip = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (clip >= n_clips) return;
  const float dist = lane < AW_NBITS ? fabsf(values[(long long)clip * AW_NBITS + lane] - thr) : INFINITY;
  const unsigned m = __ballot_sync(0xffffffffu, !(dist >= margin));      // NaN counts as low margin
  if (lane == 0) {
    flags[1 + clip] = m != 0;
    if (m) atomicAdd(flags, 1);
  }
}

// The tensor-core pass (TF32 / 16-bit operands) moves a detector output by up to ~2e-4, so a bit
// whose |v - threshold| is below `exact_margin` (default 1e-3) could decode differently from the
// reference's fp32 arithmetic (utils/watermark/decoder.py:51,63 is a strict '>').  Those clips --
// none on watermarked audio, a few on un-watermarked or heavily attacked audio -- are evaluated
// again through the exact CUDA-core GEMMs (float64 accumulation, <= 7e-7 from the reference), so
// the decoded bits are the reference's.  Costs one 4-byte D2H copy + stream synchronisation per call.
extern "C" int aw_detect_batch(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples,
                               int64_t stride, int sample_rate, float* d_values, void* stream) {
  AW_REQUIRE(ctx && d_audio && d_values, "aw_detect_batch: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  AW_CUDA(cudaSetDevice(ctx->device));
  AW_ENTRY("aw_detect_batch");
  nvtxRangePushA("aw_detect_batch");
  struct Pop { ~Pop() { nvtxRangePop(); } } pop_;
  Dims d;
  if (make_dims(ctx, n_clips, n_samples, sample_rate, &d)) return 1;
  if (detect_pass(ctx, d, d, d_audio, stride, d_values, st)) return 1;
  ctx->stat_detect_clips += n_clips;
  if (ctx->prec == AW_PREC_FP32 || ctx->exact_margin <= 0.0) {
    prof_mark(ctx, st, nullptr);
    return 0;
  }
  if (ensure(ctx->lowm, (size_t)(1 + n_clips) * 4)) return 1;
  if (ctx->h_lowm_cap < (size_t)(1 + n_clips)) {
    if (ctx->h_lowm) AW_CUDA(cudaFreeHost(ctx->h_lowm));
    ctx->h_lowm = nullptr;
    AW_CUDA(cudaMallocHost((void**)&ctx->h_lowm, (size_t)(1 + n_clips) * 4));
    ctx->h_lowm_cap = (size_t)(1 + n_clips);
  }
  int* flags = (int*)ctx->lowm.p;
  AW_CUDA(cudaMemsetAsync(flags, 0, 4, st));
  prof_mark(ctx, st, "flag_low_margin");
  k_flag_low_margin<<<(n_clips + 3) / 4, 128, 0, st>>>(d_values, ctx->threshold, (float)ctx->exact_margin, n_clips, flags);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  prof_mark(ctx, st, nullptr);
  AW_CUDA(cudaMemcpyAsync(ctx->h_lowm, flags, 4, cudaMemcpyDeviceToHost, st));
  AW_CUDA(cudaStreamSynchronize(st));
  const int n_low = ctx->h_lowm[0];
  if (n_low == 0) return 0;
  AW_CUDA(cudaMemcpyAsync(ctx->h_lowm + 1, flags + 1, (size_t)n_clips * 4, cudaMemcpyDeviceToHost, st));
  AW_CUDA(cudaStreamSynchronize(st));
  nvtxRangePushA("exact_reevaluation");
  const int prev = ctx->prec;
  ctx->prec = AW_PREC_FP32;
  Dims d1 = d;
  d1.n = 1;
  d1.rows = d1.Tp_pad;
  int rc = 0;
  for (int i = 0; i < n_clips && !rc; ++i)
    if (ctx->h_lowm[1 + i])
      rc = detect_pass(ctx, d1, d1, d_audio + (size_t)i * stride, stride, d_values + (size_t)i * AW_NBITS, st);
  ctx->prec = prev;
  nvtxRangePop();
  prof_mark(ctx, st, nullptr);
  ctx->stat_reeval_clips += n_low;
  return rc;
}

__global__ void k_to_bf16(const float* in, __nv_bfloat16* out, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16_rn(in[i]);
}
__global__ void k_pattern_to_float(const int32_t* p, float* o, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = (float)p[i];
}
__global__ void k_fill(float* p, float v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void k_set_int(int* p, int v) { *p = v; }

// torch/optim/nadam.py scalars, Python-float arithmetic with the float32 mu_product
static void nadam_table(int iters, std::vector<NadamStep>& out) {
  out.resize(iters);
  const double lr = 0.1, beta1 = 0.9, beta2 = 0.999, decay = 4e-3;
  float mu_product = 1.0f;
  for (int step = 1; step <= iters; ++step) {
    const double bc2 = 1.0 - pow(beta2, (double)step);
    const double mu = beta1 * (1.0 - 0.5 * pow(0.96, step * decay));
    const double mu_next = beta1 * (1.0 - 0.5 * pow(0.96, (step + 1) * decay));
    mu_product = mu_product * (float)mu;
    const double mp = (double)mu_product;
    NadamStep s;
    s.a_g = (float)(-lr * (1.0 - mu) / (1.0 - mp));
    s.a_m = (float)((-lr * mu_next) / (1.0 - mp * mu_next));
    s.inv_bc2 = 1.0f / (float)bc2;
    s.pad = 0.f;
    out[step - 1] = s;
  }
}


// ---------------------------------------------------------------------------
// tensor-core spectral path of the fp16 embed loop (spectc.cuh)
// ---------------------------------------------------------------------------
// Large batches only: the path adds five launches per iteration (peak, spectrum, adjoint, two edge passes, frame
// rows, update instead of two fused kernels), which costs more than it saves while an iteration is launch-latency
// bound -- a single clip (the service API's shape) stays on the fused FFT kernels.
static bool tc_eligible(aw_ctx* ctx, const Dims& d) {
  return ctx->tc_spec && ctx->prec == AW_PREC_FP16 && 2 * d.nb <= AW_TC_P && d.T >= 128 && !ctx->sh &&
         (long long)d.n * d.T >= (long long)ctx->tc_min_frames;
}
static long long tc_rows128(const Dims& d) { return (((long long)d.n * (d.T + 6) + 127) / 128) * 128; }

static int tc_prepare_mats(aw_ctx* ctx, const Dims& d, const float* h_window) {
  aw_ctx::TcMats& m = ctx->tcm;
  if (m.bin0 == d.bin0 && m.nb == d.nb) return 0;
  SpecTcMats h;
  spectc_build(h_window, d.bin0, d.nb, h);
  cudaFree(m.peakB); cudaFree(m.compB); cudaFree(m.compBT); cudaFree(m.fix);
  m.peakB = m.compB = m.compBT = nullptr; m.fix = nullptr;
  AW_CUDA(cudaMalloc(&m.peakB, h.peakB.size() * 2));
  AW_CUDA(cudaMalloc(&m.compB, h.compB.size() * 2));
  AW_CUDA(cudaMalloc(&m.compBT, h.compBT.size() * 2));
  AW_CUDA(cudaMalloc(&m.fix, h.fix.size() * 4));
  AW_CUDA(cudaMemcpy(m.peakB, h.peakB.data(), h.peakB.size() * 2, cudaMemcpyHostToDevice));
  AW_CUDA(cudaMemcpy(m.compB, h.compB.data(), h.compB.size() * 2, cudaMemcpyHostToDevice));
  AW_CUDA(cudaMemcpy(m.compBT, h.compBT.data(), h.compBT.size() * 2, cudaMemcpyHostToDevice));
  AW_CUDA(cudaMemcpy(m.fix, h.fix.data(), h.fix.size() * 4, cudaMemcpyHostToDevice));
  if (make_map(ctx, &m.tm_peakB, m.peakB, 256, 4 * AW_TC_P, 256, true)) return 1;
  if (make_map(ctx, &m.tm_compB, m.compB, AW_TC_P, 7 * AW_TC_P, AW_TC_P, true)) return 1;
  if (make_map(ctx, &m.tm_compBT, m.compBT, AW_TC_P, 7 * AW_TC_P, AW_TC_P, true)) return 1;
  m.bin0 = d.bin0; m.nb = d.nb;
  return 0;
}

// buffers, Toeplitz maps, the constant out-of-band spectrum and the first frame rows of a wave
static int tc_setup_wave(aw_ctx* ctx, const Dims& d, cudaStream_t st) {
  const long long rows = (long long)d.n * (d.T + 6), r128 = tc_rows128(d);
  const size_t frame_bytes = (size_t)(r128 + 8) * AW_TC_P * 2;          // + 8 rows: the Toeplitz reach of the last rows
  if (ensure(ctx->tc_X, frame_bytes) || ensure(ctx->tc_dS, frame_bytes) ||
      ensure(ctx->tc_soob, (size_t)d.n * d.T * d.nb * 8) || ensure(ctx->tc_dX, (size_t)r128 * AW_TC_P * 4) ||
      ensure(ctx->tc_gedge, (size_t)d.n * 12 * d.nb * 4) || ensure(ctx->tc_dmax, (size_t)d.n * 8) ||
      ensure(ctx->tc_ones, (size_t)d.n * 8))
    return 1;
  if (ctx->tc_map_x != ctx->tc_X.p || ctx->tc_map_ds != ctx->tc_dS.p || ctx->tc_map_rows != rows) {
    if (make_map(ctx, &ctx->tm_tcX, ctx->tc_X.p, r128 + 8, AW_TC_P, 128, true)) return 1;
    if (make_map(ctx, &ctx->tm_tcdS, ctx->tc_dS.p, r128 + 8, AW_TC_P, 128, true)) return 1;
    ctx->tc_map_x = ctx->tc_X.p; ctx->tc_map_ds = ctx->tc_dS.p; ctx->tc_map_rows = rows;
  }
  AW_CUDA(cudaMemsetAsync(ctx->tc_X.p, 0, frame_bytes, st));
  AW_CUDA(cudaMemsetAsync(ctx->tc_dS.p, 0, frame_bytes, st));
  AW_CUDA(cudaMemsetAsync(ctx->tc_gedge.p, 0, (size_t)d.n * 12 * d.nb * 4, st));
  AW_CUDA(cudaMemsetAsync(ctx->tc_dmax.p, 0, (size_t)d.n * 8, st));
  // S_oob = STFT(y_oob) restricted to the band, un-normalised (peak word 1.0: x / (1 + 1e-8) == x in fp32)
  k_fill_u64<<<(d.n + 255) / 256, 256, 0, st>>>((unsigned long long*)ctx->tc_ones.p, (unsigned long long)0x3f800000u << 32, d.n);
  ctx->launches++;
  AnaArgs a = ana_base(ctx, d);
  a.sig = (const float*)ctx->yoob.p; a.sig_stride = d.L; a.len = d.L;
  a.peak = (unsigned long long*)ctx->tc_ones.p;
  a.ph = (float2*)ctx->tc_soob.p;
  if (launch_ana<ANA_CPLX>(ctx, d, a, st)) return 1;
  prof_mark(ctx, st, "tc_xprep");
  k_tc_xprep<<<dim3((d.T + AW_TC_FR - 1) / AW_TC_FR, d.n), 256, 0, st>>>((const float*)ctx->c.p, (const float2*)ctx->ph_u.p, d.T, d.nb,
                                              (__half*)ctx->tc_X.p);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

static EpiArgsT<float> tc_epi(const Dims& d) {
  EpiArgsT<float> ep{};
  ep.toep_P = AW_TC_P;
  ep.rpc = d.T + 6;
  ep.total_rows = d.n * (d.T + 6);
  ep.T = d.T; ep.L = d.L; ep.nb = d.nb;
  return ep;
}

// c u (frame rows) -> max |y| -> |S|, S/|S| ; then the six edge frames per clip exactly
static int tc_forward(aw_ctx* ctx, const Dims& d, const Acc& acc, cudaStream_t st) {
  const int r128 = (int)tc_rows128(d);
  EpiArgsT<float> ep = tc_epi(d);
  ep.aux = (const float*)ctx->yoob.p; ep.fix = ctx->tcm.fix; ep.fix0 = 1.0f / 1024.0f; ep.peak = acc.peak_y;
  if (launch_tc<__half, float, 256, EPI_PEAK>(ctx, ctx->tm_tcX, ctx->tcm.tm_peakB, r128, 256, 4 * AW_TC_P, ep, st)) return 1;
  EpiArgsT<float> es = tc_epi(d);
  es.aux = (const float*)ctx->tc_soob.p; es.mag = (float*)ctx->mag.p; es.qph = (float2*)ctx->ph_q.p;
  if (launch_tc<__half, float, AW_TC_P, EPI_SPEC>(ctx, ctx->tm_tcX, ctx->tcm.tm_compB, r128, AW_TC_P, 7 * AW_TC_P, es, st)) return 1;
  SpecArgs f;
  memset(&f, 0, sizeof(f));
  f.amp = (float*)ctx->c.p; f.ph = (float2*)ctx->ph_u.p;
  f.z_oob = (float*)ctx->zoob.p; f.peak_y = acc.peak_y;
  f.mag = (float*)ctx->mag.p; f.q = (float2*)ctx->ph_q.p;
  f.edge_mode = 1;
  return launch_spec<SPEC_FWD>(ctx, d, f, st);
}

// dA q (frame rows, edge rows zeroed) -> K^T -> + exact edge adjoint + peak sub-gradient -> NAdam
static int tc_backward(aw_ctx* ctx, const Dims& d, int* itc, cudaStream_t st, int* nonfinite, bool first) {
  const int r128 = (int)tc_rows128(d);
  if (first) {            // the first iteration has no predecessor to take the scale from
    prof_mark(ctx, st, "tc_absmax");
    k_tc_absmax<<<dim3(32, d.n), 256, 0, st>>>((const float*)ctx->dA.p, (long long)d.T * d.nb, (unsigned*)ctx->tc_dmax.p);
    ctx->launches++;
  }
  prof_mark(ctx, st, "tc_dsprep");
  k_tc_dsprep<<<dim3((d.T + AW_TC_FR - 1) / AW_TC_FR, d.n), 256, 0, st>>>((const float*)ctx->dA.p, (const float2*)ctx->ph_q.p, d.T, d.nb,
                                                                          (unsigned*)ctx->tc_dmax.p, itc, d.n, (__half*)ctx->tc_dS.p);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  EpiArgsT<float> ep = tc_epi(d);
  ep.out = (float*)ctx->tc_dX.p; ep.ldo = AW_TC_P;
  if (launch_tc<__half, float, AW_TC_P, EPI_PLAIN>(ctx, ctx->tm_tcdS, ctx->tcm.tm_compBT, r128, AW_TC_P, 7 * AW_TC_P, ep, st)) return 1;
  SpecArgs b;
  memset(&b, 0, sizeof(b));
  b.amp = (float*)ctx->dA.p; b.ph = (float2*)ctx->ph_q.p;
  b.scal = (ClipScal*)ctx->scal.p; b.u = (float2*)ctx->ph_u.p;
  b.c = (float*)ctx->c.p; b.m = (float*)ctx->m.p; b.v = (float*)ctx->v.p;
  b.cbest = (float*)ctx->cbest.p; b.c0 = (float*)ctx->c0.p;
  b.improved = (int*)ctx->improved.p; b.steps = (NadamStep*)ctx->steps.p; b.it_ptr = itc;
  b.tol_ratio = (float)pow(10.0, -(double)ctx->tol_db / 20.0);
  b.edge_mode = 1; b.g_edge = (float*)ctx->tc_gedge.p;
  if (launch_spec<SPEC_BWD>(ctx, d, b, st)) return 1;
  TcUpdateArgs u{};
  u.T = d.T; u.nb = d.nb; u.rpc = d.T + 6;
  u.dX = (const float*)ctx->tc_dX.p; u.dmax = (const unsigned*)ctx->tc_dmax.p; u.n_clips = d.n;
  u.scal = (const ClipScal*)ctx->scal.p; u.g_edge = (const float*)ctx->tc_gedge.p;
  u.u = (const float2*)ctx->ph_u.p;
  u.c = (float*)ctx->c.p; u.m = (float*)ctx->m.p; u.v = (float*)ctx->v.p; u.cbest = (float*)ctx->cbest.p;
  u.c0 = (const float*)ctx->c0.p; u.improved = (const int*)ctx->improved.p;
  u.steps = (const NadamStep*)ctx->steps.p; u.it_ptr = itc;
  u.tol_ratio = b.tol_ratio;
  u.window = ctx->d_window; u.env256 = ctx->d_env256; u.bin0 = d.bin0;
  u.X = (__half*)ctx->tc_X.p;
  u.nonfinite = nonfinite;
  prof_mark(ctx, st, "tc_update");
  k_tc_update<<<dim3((d.T + AW_TC_FR - 1) / AW_TC_FR, d.n), 256, 0, st>>>(u);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

// Workspace of an embed call (see ensure_net_ws for ds / dn), the NAdam step table and n_flags cleared
// non-finite flags.
static int embed_setup(aw_ctx* ctx, const Dims& ds, const Dims& dn, int n_flags, int iters, cudaStream_t st) {
  if (ensure_net_ws(ctx, ds, dn, true)) return 1;
  const size_t sp = (size_t)ds.n * ds.T * ds.nb;
  if (ensure(ctx->ph_u, sp * 8) || ensure(ctx->ph_q, sp * 8) || ensure(ctx->c0, sp * 4) ||
      ensure(ctx->c, sp * 4) || ensure(ctx->m, sp * 4) || ensure(ctx->v, sp * 4) ||
      ensure(ctx->cbest, sp * 4) || ensure(ctx->dA, sp * 4) ||
      ensure(ctx->yoob, (size_t)ds.n * ds.L * 4) || ensure(ctx->y, (size_t)ds.n * ds.L * 4) ||
      ensure(ctx->zoob, (size_t)ds.n * ds.L * 4) ||
      ensure(ctx->pattern, (size_t)ds.n * AW_NBITS * 4) || ensure(ctx->scal, (size_t)ds.n * sizeof(ClipScal)) ||
      ensure(ctx->nonfinite, (size_t)n_flags * 4) || ensure(ctx->smax, (size_t)ds.n * 4) ||
      ensure(ctx->steps, (size_t)(iters > 0 ? iters : 1) * sizeof(NadamStep)))
    return 1;
  std::vector<NadamStep> tab;
  nadam_table(iters, tab);
  if (iters > 0)
    AW_CUDA(cudaMemcpyAsync(ctx->steps.p, tab.data(), tab.size() * sizeof(NadamStep),
                            cudaMemcpyHostToDevice, st));
  AW_CUDA(cudaMemsetAsync(ctx->nonfinite.p, 0, (size_t)n_flags * 4, st));
  ctx->last_embed_clips = n_flags;
  AW_CUDA(cudaStreamSynchronize(st));   // `tab` is pageable host memory
  return 0;
}

// What one embed wave reads and writes, offset to the wave's first clip.
struct WaveIO {
  const float* x; int64_t stride;
  const int32_t* pattern;                 // [n][AW_NBITS]
  const float* scale; bool signed_max;    // output scale: per clip, the input's signed max (AW_SCALE_SIGNED_MAX) or none
  float* out; int64_t out_stride;
  // samples [pk_lo, pk_hi) compete for the peak and are written out (pk_hi = 0: all); the peak word packs
  // local index + idx_base (frame-sharded mode: a segment's own samples, global indices)
  int pk_lo, pk_hi, idx_base;
  float* best_loss;                       // [n] or null
  float* losses; int n_total;             // [iters][n_total] or null
  int* nonfinite;                         // [n]
};

// One embed wave: init, the optimisation loop and the final synthesis of ds.n clips, or of one shard's
// segment (see ensure_net_ws for ds / dn).
static int embed_wave(aw_ctx* ctx, const Dims& ds, const Dims& dn, const WaveIO& w, int iters, bool use_graph,
                      cudaStream_t st) {
  SparseMel sm;
  if (get_mel(ctx, ds.bin0, ds.nb, &sm)) return 1;
  const Acc acc = acc_view(ctx, dn);           // peak word at the base; partial-sum arrays of the net's frames
  unsigned long long* peakx = (unsigned long long*)ctx->peakx.p;
  int* itc = (int*)ctx->itc.p;

  k_set_int<<<1, 1, 0, st>>>(itc, -1);
  k_fill<<<(ds.n + 255) / 256, 256, 0, st>>>((float*)ctx->best.p, INFINITY, ds.n);
  k_pattern_to_float<<<(ds.n * AW_NBITS + 255) / 256, 256, 0, st>>>(w.pattern, (float*)ctx->pattern.p,
                                                                      ds.n * AW_NBITS);
  ctx->launches += 3;
  AW_LAUNCH_CHECK();
  if (launch_peak(ctx, w.x, w.stride, ds.N, ds.n, peakx, st, w.signed_max ? (int*)ctx->smax.p : nullptr)) return 1;
  if (sync_peak(ctx, peakx, st)) return 1;

  // ---- pre-STFT, bounds, constant out-of-band waveform (multibit_embedder.py:143-160)
  nvtxRangePushA("embed:init_stft_bounds_oob");
  AnaArgs a0 = ana_base(ctx, ds);
  a0.sig = w.x; a0.sig_stride = w.stride; a0.len = ds.N;
  a0.peak = peakx;
  a0.mag = (float*)ctx->c0.p; a0.ph = (float2*)ctx->ph_u.p;
  a0.c = (float*)ctx->c.p; a0.m = (float*)ctx->m.p; a0.v = (float*)ctx->v.p;
  a0.cbest = (float*)ctx->cbest.p;
  if (launch_ana<ANA_INIT>(ctx, ds, a0, st)) return 1;
  SynArgs s0 = syn_base(ctx, ds);
  s0.amp = (float*)ctx->c0.p; s0.ph = (float2*)ctx->ph_u.p; s0.scale = 1.0f / AW_NFFT;
  s0.x = w.x; s0.x_stride = w.stride; s0.peak_x = peakx;
  s0.y_oob = (float*)ctx->yoob.p;
  s0.z_oob = (float*)ctx->zoob.p;
  if (launch_syn<SYN_OOB>(ctx, ds, s0, st)) return 1;
  // fp16 loop at 44.1 / 48 kHz: the loop's band-limited transforms run on the tensor cores (spectc.cuh)
  const bool tc = tc_eligible(ctx, ds);
  if (tc) {
    if (tc_prepare_mats(ctx, ds, ctx->h_window.data())) return 1;
    if (tc_setup_wave(ctx, ds, st)) return 1;
  }
  ctx->tc_active = tc;
  struct TcOff { aw_ctx* c; ~TcOff() { c->tc_active = false; } } tc_off_{ctx};
  nvtxRangePop();

  // ---- optimisation loop (multibit_embedder.py:95-122)
  nvtxRangePushA("embed:nadam_loop");
  auto iteration = [&](bool first) -> int {
    // fused spectral passes (spec.cuh): y and dpad never leave shared memory
    if (begin_pass(ctx, ds.n, itc, st)) return 1;
    if (tc) {
      if (tc_forward(ctx, ds, acc, st)) return 1;
    } else {
      SpecArgs f;
      memset(&f, 0, sizeof(f));
      f.amp = (float*)ctx->c.p; f.ph = (float2*)ctx->ph_u.p;
      f.z_oob = (float*)ctx->zoob.p; f.peak_y = acc.peak_y;
      f.mag = (float*)ctx->mag.p; f.q = (float2*)ctx->ph_q.p;
      f.pk_lo = w.pk_lo; f.pk_hi = w.pk_hi; f.idx_base = w.idx_base;
      if (launch_spec<SPEC_FWD>(ctx, ds, f, st)) return 1;
    }
    if (sync_peak(ctx, acc.peak_y, st)) return 1;                      // max |y| over the whole clip
    if (with_act_type(ctx, [&](auto tag) -> int {
          using AT = decltype(tag);
          if (net_forward<AT>(ctx, dn, acc, sm, st, acc.peak_y)) return 1;
          if (run_head<AT>(ctx, dn, (float*)ctx->pattern.p, (float*)ctx->values.p, w.losses, w.n_total, true, st))
            return 1;
          return net_backward<AT>(ctx, dn, acc, sm, st, true);
        }))
      return 1;
    const double* sp2 = acc.s2_part;
    int sb2 = p0a_blocks(dn);
    if (clip_sums(ctx, ctx->red_c, sp2, sb2, dn.n, 1, st)) return 1;                       // Euler sum over the clip
    if (sb2 > 512 && reduce_if_long(ctx, ctx->red_a, sp2, sb2, dn.n, 1, st)) return 1;   // 1 h: 38 760 -> 606 -> 10
    prof_mark(ctx, st, "clip_scalars");
    k_clip_scalars<<<(dn.n + 127) / 128, 128, 0, st>>>(acc.peak_y, sp2, sb2, dn.n, (ClipScal*)ctx->scal.p, w.idx_base,
                                                       tc ? (unsigned*)ctx->tc_dmax.p : nullptr, itc);
    ctx->launches++;
    AW_LAUNCH_CHECK();
    if (sync_halo(ctx, (float*)ctx->dA.p, ds.nb, st)) return 1;       // spectral gradient of the halo frames
    if (tc) return tc_backward(ctx, ds, itc, st, w.nonfinite, first);
    SpecArgs b;
    memset(&b, 0, sizeof(b));
    b.amp = (float*)ctx->dA.p; b.ph = (float2*)ctx->ph_q.p;
    b.scal = (ClipScal*)ctx->scal.p; b.u = (float2*)ctx->ph_u.p;
    b.c = (float*)ctx->c.p; b.m = (float*)ctx->m.p; b.v = (float*)ctx->v.p;
    b.cbest = (float*)ctx->cbest.p; b.c0 = (float*)ctx->c0.p;
    b.improved = (int*)ctx->improved.p; b.steps = (NadamStep*)ctx->steps.p; b.it_ptr = itc;
    b.nonfinite = w.nonfinite;
    b.tol_ratio = (float)pow(10.0, -(double)ctx->tol_db / 20.0);
    if (launch_spec<SPEC_BWD>(ctx, ds, b, st)) return 1;
    return sync_halo(ctx, (float*)ctx->c.p, ds.nb, st);              // updated coefficients of the halo frames
  };
  if (use_graph) {
    // iteration 0 runs eagerly (function attributes, scratch sizes), iteration 1 is captured
    // without executing, and the graph is replayed for iterations 1 .. iters-1; the iteration
    // index and all per-clip state live on the device, so every replay is identical work
    const int64_t l0 = ctx->launches;
    if (iteration(true)) return 1;
    const int64_t per_iter = ctx->launches - l0 - (tc ? 1 : 0);
    AW_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
    const int rc = iteration(false);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc || ce != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      return rc ? 1 : set_error("aw_embed_batch: stream capture failed: %s", cudaGetErrorString(ce));
    }
    cudaGraphExec_t exec = nullptr;
    if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
      cudaGraphDestroy(graph);
      return set_error("aw_embed_batch: cudaGraphInstantiate failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    for (int it = 1; it < iters; ++it) {
      if (cudaGraphLaunch(exec, st) != cudaSuccess) {
        cudaGraphExecDestroy(exec);
        cudaGraphDestroy(graph);
        return set_error("aw_embed_batch: cudaGraphLaunch failed: %s", cudaGetErrorString(cudaGetLastError()));
      }
    }
    ctx->launches += per_iter * (iters - 2);      // the captured pass was counted once already
    cudaGraphExecDestroy(exec);
    cudaGraphDestroy(graph);
  } else {
    for (int it = 0; it < iters; ++it)
      if (iteration(it == 0)) return 1;
  }
  nvtxRangePop();
  // ---- final synthesis from the best coefficients (multibit_embedder.py:173-192), peak over the whole clip
  nvtxRangePushA("embed:final_synthesis");
  if (sync_halo(ctx, (float*)ctx->cbest.p, ds.nb, st)) return 1;
  if (begin_pass(ctx, ds.n, nullptr, st)) return 1;
  SynArgs sf = syn_base(ctx, ds);
  sf.amp = (float*)ctx->cbest.p; sf.ph = (float2*)ctx->ph_u.p; sf.scale = 1.0f / AW_NFFT;
  sf.y_oob = (float*)ctx->yoob.p; sf.y = (float*)ctx->y.p; sf.peak_y = acc.peak_y;
  sf.pk_lo = w.pk_lo; sf.pk_hi = w.pk_hi;
  if (launch_syn<SYN_WAVE>(ctx, ds, sf, st)) return 1;
  if (sync_peak(ctx, acc.peak_y, st)) return 1;
  const int len = (w.pk_hi > 0 ? w.pk_hi : ds.L) - w.pk_lo;
  dim3 g(std::min((len + 4095) / 4096, std::max(64, 8192 / ds.n)), ds.n);
  prof_mark(ctx, st, "final_normalize");
  k_final_normalize<<<g, 256, 0, st>>>((float*)ctx->y.p + w.pk_lo, len, acc.peak_y, w.scale,
                                       w.signed_max ? (const int*)ctx->smax.p : nullptr, w.out, w.out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  if (w.best_loss)
    AW_CUDA(cudaMemcpyAsync(w.best_loss, ctx->best.p, (size_t)ds.n * 4, cudaMemcpyDeviceToDevice, st));
  ctx->last_n = ds.n; ctx->last_T = ds.T; ctx->last_nb = ds.nb;
  nvtxRangePop();
  return 0;
}

extern "C" int aw_embed_batch(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples,
                              int64_t stride, int sample_rate, const int32_t* d_pattern, int iters,
                              const float* d_scale, int scale_mode, float* d_out, int64_t out_stride,
                              float* d_best_loss, float* d_losses, int wave_clips, void* stream) {
  AW_REQUIRE(ctx && d_audio && d_pattern && d_out, "aw_embed_batch: null argument");
  AW_REQUIRE(iters >= 0, "aw_embed_batch: iters < 0");
  AW_REQUIRE(scale_mode == AW_SCALE_NONE || scale_mode == AW_SCALE_SIGNED_MAX, "aw_embed_batch: bad scale_mode %d", scale_mode);
  AW_REQUIRE(!(d_scale && scale_mode != AW_SCALE_NONE), "aw_embed_batch: d_scale and scale_mode are exclusive");
  cudaStream_t user_stream = (cudaStream_t)stream, st = user_stream;
  AW_CUDA(cudaSetDevice(ctx->device));
  AW_ENTRY("aw_embed_batch");
  nvtxRangePushA("aw_embed_batch");
  struct Pop { ~Pop() { nvtxRangePop(); } } pop_;
  // Graph replay needs a capturable stream (the caller's may be the legacy default stream): the
  // whole call runs on the context's stream, ordered after / before the caller's by two events.
  const bool use_graph = ctx->graphs && !ctx->prof_on && iters >= 4;
  if (use_graph) {
    AW_CUDA(cudaEventRecord(ctx->ev_in, user_stream));
    AW_CUDA(cudaStreamWaitEvent(ctx->gstream, ctx->ev_in, 0));
    st = ctx->gstream;
  }
  if (wave_clips <= 0 || wave_clips > n_clips) {
    // default: the whole batch in one wave, unless its workspace would not fit in device memory
    // (then the largest wave that fits in 85 % of what is free plus what this context already holds)
    wave_clips = n_clips;
    Dims d1;
    if (make_dims(ctx, 1, n_samples, sample_rate, &d1)) return 1;
    const double per_clip = (double)d1.T * d1.nb * (7 * 4 + 2 * 8) + 3.0 * d1.L * 4 + (double)d1.T * AW_NMEL * 4 +
                            (double)d1.Tp_pad * ((128 + 512 + 1024 + 1024 + 64) * 4 + 2 * 1024 * 4 + 64 * 4 + 128 * 4) +
                            (double)d1.tiles * (1024 * 8 + 64 * 24) + 64 * 1024;
    size_t free_b = 0, total_b = 0;
    AW_CUDA(cudaMemGetInfo(&free_b, &total_b));
    double held = 0.0;
    for (Buf* b : all_bufs(ctx)) held += (double)b->cap;
    const double budget = 0.85 * ((double)free_b + held);
    if (per_clip * n_clips > budget) {
      wave_clips = (int)std::max(1.0, floor(budget / per_clip));
      AW_REQUIRE(per_clip <= budget, "aw_embed_batch: one %d-sample clip needs %.1f GB of workspace, %.1f GB available",
                 n_samples, per_clip / 1e9, budget / 1e9);
    }
  }
  Dims d;
  if (make_dims(ctx, wave_clips, n_samples, sample_rate, &d)) return 1;
  AW_REQUIRE(out_stride >= d.L, "aw_embed_batch: out_stride %lld < %d", (long long)out_stride, d.L);
  if (embed_setup(ctx, d, d, n_clips, iters, st)) return 1;

  for (int w0 = 0; w0 < n_clips; w0 += wave_clips) {
    Dims dw = d;
    dw.n = std::min(wave_clips, n_clips - w0);
    dw.rows = dw.n * dw.Tp_pad;
    // tensor maps are encoded for d.rows; a smaller last wave only uses a prefix of rows
    WaveIO w{};
    w.x = d_audio + (size_t)w0 * stride; w.stride = stride;
    w.pattern = d_pattern + (size_t)w0 * AW_NBITS;
    w.scale = d_scale ? d_scale + w0 : nullptr; w.signed_max = scale_mode == AW_SCALE_SIGNED_MAX;
    w.out = d_out + (size_t)w0 * out_stride; w.out_stride = out_stride;
    w.best_loss = d_best_loss ? d_best_loss + w0 : nullptr;
    w.losses = d_losses ? d_losses + w0 : nullptr; w.n_total = n_clips;
    w.nonfinite = (int*)ctx->nonfinite.p + w0;
    if (embed_wave(ctx, dw, dw, w, iters, use_graph, st)) return 1;
  }
  prof_mark(ctx, st, nullptr);
  if (use_graph) {
    AW_CUDA(cudaEventRecord(ctx->ev_out, st));
    AW_CUDA(cudaStreamWaitEvent(user_stream, ctx->ev_out, 0));
  }
  return 0;
}


// ---------------------------------------------------------------------------
// frame-sharded long-form mode (SURVEY 8f-1, BASELINE configs[4]): ONE long clip, frames split over
// the ranks of a box.  Every statistic the reference takes is whole-clip (utils/audio/waveform.py:19,
// detection/modules/globalStandardize.py:17-19, multibit_detector_net.py:50,126, modules/BRH.py:18),
// so a rank processes a halo-extended SEGMENT of the clip as if it were a clip of its own -- the
// pseudo-edges only contaminate halo frames, which are never used -- while (a) every per-clip sum /
// max is reduced over the ranks between the kernel that produces its partials and the kernel that
// consumes it, and (b) the halo frames of the optimisation variables and of the spectral gradient are
// refreshed from their owners every iteration.  Results equal the single-GPU run up to the summation
// order of the float64 statistics.  The segment runs through detect_pass / embed_wave; the hooks
// sync_peak, sync_halo and clip_sums are where it differs from a batch of one clip.
// ---------------------------------------------------------------------------
static int shard_begin(aw_ctx* ctx, aw_ctx::Shard* sh, const aw_comm* comm, int seg_samples, int seg_first_frame,
                       int own_lo, int own_hi, int total_frames, int sample_rate, Dims* ds, Dims* dn) {
  AW_REQUIRE(comm && comm->allreduce && comm->allgather && comm->d_arena, "sharded mode: incomplete aw_comm");
  AW_REQUIRE(comm->world >= 1 && comm->rank >= 0 && comm->rank < comm->world, "sharded mode: bad rank %d / %d",
             comm->rank, comm->world);
  AW_REQUIRE(comm->arena_bytes >= AW_ARENA_RECV + (int64_t)comm->world * (32 << 10),
             "sharded mode: arena must hold %d bytes", AW_ARENA_RECV + comm->world * (32 << 10));
  if (make_dims(ctx, 1, seg_samples, sample_rate, ds)) return 1;
  AW_REQUIRE(own_lo >= 0 && own_hi <= ds->T && own_hi - own_lo >= 2 * AW_HALO,
             "sharded mode: own frames [%d,%d) of a %d-frame segment (need >= %d)", own_lo, own_hi, ds->T, 2 * AW_HALO);
  const bool first = comm->rank == 0, last = comm->rank == comm->world - 1;
  AW_REQUIRE(first ? (own_lo == 0 && seg_first_frame == 0) : own_lo == AW_HALO, "sharded mode: left halo must be %d frames", AW_HALO);
  AW_REQUIRE(last ? own_hi == ds->T : own_hi == ds->T - AW_HALO, "sharded mode: right halo must be %d frames", AW_HALO);
  AW_REQUIRE(((seg_first_frame + own_lo) & 1) == 0 && (last || ((own_hi - own_lo) & 1) == 0),
             "sharded mode: shard boundaries must fall on even frames (AvgPool1d(2,2) pairs)");
  AW_REQUIRE(last ? seg_first_frame + ds->T == total_frames : seg_first_frame + ds->T < total_frames + AW_HALO,
             "sharded mode: segment does not fit the clip");
  sh->comm = *comm;
  sh->e0 = seg_first_frame;
  sh->own_lo = own_lo;
  sh->own_hi = own_hi;
  *dn = *ds;
  set_frames(dn, own_hi - own_lo);
  dn->T_clip = total_frames;
  dn->Tp_clip = total_frames / 2;
  return 0;
}

extern "C" int aw_detect_sharded(aw_ctx* ctx, const float* d_segment, int seg_samples, int seg_first_frame,
                                 int own_lo, int own_hi, int total_frames, int sample_rate, const aw_comm* comm,
                                 float* d_values, void* stream) {
  AW_REQUIRE(ctx && d_segment && d_values, "aw_detect_sharded: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  AW_CUDA(cudaSetDevice(ctx->device));
  aw_ctx::Shard sh;
  Dims ds, dn;
  if (shard_begin(ctx, &sh, comm, seg_samples, seg_first_frame, own_lo, own_hi, total_frames, sample_rate, &ds, &dn)) return 1;
  ctx->sh = &sh;
  struct Clear { aw_ctx* c; ~Clear() { c->sh = nullptr; } } clear_{ctx};
  nvtxRangePushA("aw_detect_sharded");
  struct Pop { ~Pop() { nvtxRangePop(); } } pop_;
  const int rc = detect_pass(ctx, ds, dn, d_segment, seg_samples, d_values, st);
  prof_mark(ctx, st, nullptr);
  return rc;
}

extern "C" int aw_embed_sharded(aw_ctx* ctx, const float* d_segment, int seg_samples, int seg_first_frame,
                                int own_lo, int own_hi, int total_frames, int sample_rate,
                                const int32_t* d_pattern, int iters, const aw_comm* comm, float* d_out_own,
                                int64_t out_capacity, float* d_best_loss, float* d_losses, int64_t* comm_counts,
                                void* stream) {
  AW_REQUIRE(ctx && d_segment && d_pattern && d_out_own, "aw_embed_sharded: null argument");
  AW_REQUIRE(iters >= 0, "aw_embed_sharded: iters < 0");
  cudaStream_t st = (cudaStream_t)stream;
  AW_CUDA(cudaSetDevice(ctx->device));
  aw_ctx::Shard sh;
  Dims ds, dn;
  if (shard_begin(ctx, &sh, comm, seg_samples, seg_first_frame, own_lo, own_hi, total_frames, sample_rate, &ds, &dn)) return 1;
  // own output samples: global [256 f0, 256 f1) cut at the clip's length 256 (T - 1)
  const int out_lo = AW_HOP * own_lo, out_hi = std::min(AW_HOP * own_hi, ds.L);
  AW_REQUIRE(out_capacity >= out_hi - out_lo, "aw_embed_sharded: output capacity %lld < %d", (long long)out_capacity, out_hi - out_lo);
  if (embed_setup(ctx, ds, dn, 1, iters, st)) return 1;
  AW_CUDA(cudaMemsetAsync(ctx->dA.p, 0, (size_t)ds.T * ds.nb * 4, st));
  ctx->sh = &sh;
  struct Clear { aw_ctx* c; ~Clear() { c->sh = nullptr; } } clear_{ctx};
  nvtxRangePushA("aw_embed_sharded");
  struct Pop { ~Pop() { nvtxRangePop(); } } pop_;
  WaveIO w{};
  w.x = d_segment; w.stride = seg_samples;
  w.pattern = d_pattern;
  w.out = d_out_own; w.out_stride = out_capacity;
  w.pk_lo = out_lo; w.pk_hi = out_hi;
  w.idx_base = AW_HOP * seg_first_frame;     // global index of the segment's sample 0
  w.best_loss = d_best_loss;
  w.losses = d_losses; w.n_total = 1;
  w.nonfinite = (int*)ctx->nonfinite.p;
  // the collectives are host callbacks: no graph replay
  if (embed_wave(ctx, ds, dn, w, iters, false, st)) return 1;
  if (comm_counts) { comm_counts[0] = sh.n_allreduce; comm_counts[1] = sh.n_allgather; }
  prof_mark(ctx, st, nullptr);
  return 0;
}

extern "C" int aw_embed_state(aw_ctx* ctx, int which, float* d_dst, int64_t capacity, void* stream) {
  AW_REQUIRE(ctx && d_dst, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  const size_t cnt = (size_t)ctx->last_n * ctx->last_T * ctx->last_nb;
  AW_REQUIRE(cnt > 0, "aw_embed_state: no embed has run");
  if (which >= 10) {
    // debug views of the last iteration's intermediates (float32 words)
    const size_t L = (size_t)AW_HOP * (ctx->last_T - 1), n = ctx->last_n;
    const void* p = nullptr;
    size_t words = 0;
    switch (which) {
      case 10: p = ctx->y.p; words = n * L; break;                // final synthesis only
      case 12: p = ctx->accum.p; words = n * 2; break;            // packed peak (u64 per clip)
      case 13: p = ctx->dA.p; words = cnt; break;
      case 14: p = ctx->mag.p; words = cnt; break;
      case 15: p = ctx->yoob.p; words = n * L; break;
      case 16: p = ctx->ph_q.p; words = cnt * 2; break;
      case 17: p = ctx->M.p; words = n * ctx->last_T * AW_NMEL; break;
      case 18: p = ctx->dp0.p; words = (size_t)ctx->ws_rows * 128; break;
      default: return set_error("aw_embed_state: bad selector");
    }
    AW_REQUIRE((int64_t)words <= capacity, "aw_embed_state: capacity %lld < %zu", (long long)capacity, words);
    AW_CUDA(cudaMemcpyAsync(d_dst, p, words * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
  }
  AW_REQUIRE((int64_t)cnt <= capacity, "aw_embed_state: capacity %lld < %zu", (long long)capacity, cnt);
  Buf* src[5] = {&ctx->c, &ctx->cbest, &ctx->c0, &ctx->m, &ctx->v};
  AW_REQUIRE(which >= 0 && which < 5, "aw_embed_state: bad selector");
  AW_CUDA(cudaMemcpyAsync(d_dst, src[which]->p, cnt * 4, cudaMemcpyDeviceToDevice,
                          (cudaStream_t)stream));
  return 0;
}

extern "C" int aw_decide_and_count(aw_ctx* ctx, const float* d_values, const int32_t* d_ref_bits,
                                   int n_clips, int32_t* d_bits_out, int32_t* d_err_per_clip,
                                   uint64_t* d_counters, void* stream) {
  AW_REQUIRE(ctx && d_values, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "decide_count");
  k_decide_count<<<(n_clips + 3) / 4, 128, 0, (cudaStream_t)stream>>>(
      d_values, d_ref_bits, ctx->threshold, n_clips, d_bits_out, d_err_per_clip,
      (unsigned long long*)d_counters);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_snr_batch(aw_ctx* ctx, const float* d_out, int64_t out_stride,
                            const float* d_target, int64_t tgt_stride, int n_clips, int n,
                            double* d_snr, double* d_snr_sum, void* stream) {
  AW_REQUIRE(ctx && d_out && d_target && d_snr, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (ensure(ctx->bstat, (size_t)std::max(n_clips, 1) * 16)) return 1;
  AW_CUDA(cudaMemsetAsync(ctx->bstat.p, 0, (size_t)n_clips * 16, st));
  dim3 g(std::min((n + 2047) / 2048, 64), n_clips);
  k_snr_partial<<<g, 256, 0, st>>>(d_out, out_stride, d_target, tgt_stride, n, (double*)ctx->bstat.p);
  k_snr_final<<<(n_clips + 127) / 128, 128, 0, st>>>((double*)ctx->bstat.p, n_clips, d_snr, d_snr_sum);
  ctx->launches += 2;
  AW_LAUNCH_CHECK();
  return 0;
}

// STOI of n_clips (clean, processed) pairs at 10 kHz (metrics/audio.py:43-64 through pystoi; stoi.cuh)
extern "C" int aw_stoi_batch(aw_ctx* ctx, const float* d_clean, int64_t clean_stride, const float* d_proc,
                             int64_t proc_stride, int n_clips, int n, double* d_stoi, double* d_sum,
                             double keep_above, void* stream) {
  AW_REQUIRE(ctx && d_clean && d_proc && d_stoi, "null argument");
  AW_REQUIRE(n_clips >= 1 && n >= 1, "bad argument");
  if (ctx) cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  StoiArgs a;
  memset(&a, 0, sizeof(a));
  a.x = d_clean; a.y = d_proc; a.sx = clean_stride; a.sy = proc_stride; a.n = n;
  a.F0 = n >= AW_STOI_FRAME ? (n - AW_STOI_FRAME) / AW_STOI_HOP + 1 : 0;
  a.out = d_stoi; a.out_sum = d_sum; a.keep_above = keep_above;
  const int F0 = std::max(a.F0, 1);
  a.seg_blocks = (F0 + AW_STOI_SEGS_PER_BLOCK - 1) / AW_STOI_SEGS_PER_BLOCK;
  // workspace: energy f64[F0] | part f64[seg_blocks] | emax u64 | tob f32[2][F0][16] | src i32[F0] | kept i32
  const size_t per_clip = (size_t)F0 * 8 + (size_t)a.seg_blocks * 8 + 8 + (size_t)F0 * 2 * 16 * 4 + (size_t)F0 * 4 + 8;
  if (ensure(ctx->stoi_ws, per_clip * n_clips)) return 1;
  uint8_t* w = (uint8_t*)ctx->stoi_ws.p;
  a.energy = (double*)w; w += (size_t)n_clips * F0 * 8;
  a.part = (double*)w; w += (size_t)n_clips * a.seg_blocks * 8;
  a.emax = (unsigned long long*)w; w += (size_t)n_clips * 8;
  a.tob = (float*)w; w += (size_t)n_clips * F0 * 2 * 16 * 4;
  a.src = (int*)w; w += (size_t)n_clips * F0 * 4;
  a.kept = (int*)w;
  if (!ctx->stoi_edges_set) {
    // pystoi thirdoct(10000, 512, 15, 150): band i spans the bins nearest to 150 * 2^((2i -+ 1) / 6) Hz
    int edge[AW_STOI_BANDS + 1];
    for (int i = 0; i <= AW_STOI_BANDS; ++i) {
      const double fr = 150.0 * pow(2.0, (2.0 * i - 1.0) / 6.0);
      int best = 0;
      double bd = 1e300;
      for (int k = 0; k <= AW_STOI_NFFT / 2; ++k) {
        const double f = 10000.0 * k / AW_STOI_NFFT, d = (f - fr) * (f - fr);
        if (d < bd) { bd = d; best = k; }
      }
      edge[i] = best;
    }
    AW_REQUIRE(edge[0] == AW_STOI_BIN0 && edge[AW_STOI_BANDS] == AW_STOI_BIN0 + AW_STOI_NBIN, "STOI band table");
    AW_CUDA(cudaMemcpyToSymbol(c_stoi_edge, edge, sizeof(edge)));
    ctx->stoi_edges_set = true;
  }
  AW_CUDA(cudaMemsetAsync(a.emax, 0, (size_t)n_clips * 8, st));
  AW_CUDA(cudaMemsetAsync(a.kept, 0, (size_t)n_clips * 4, st));
  if (a.F0 > 0) {
    prof_mark(ctx, st, "stoi");
    k_stoi_energy<<<dim3((a.F0 + 7) / 8, n_clips), 256, 0, st>>>(a);
    k_stoi_scan<<<n_clips, 256, 0, st>>>(a);
    if (a.F0 > 1) k_stoi_tob<<<dim3(a.F0 - 1, n_clips), 256, 0, st>>>(a);
    k_stoi_corr<<<dim3(a.seg_blocks, n_clips), 128, 0, st>>>(a);
    ctx->launches += 4;
  }
  k_stoi_final<<<(n_clips + 127) / 128, 128, 0, st>>>(a, n_clips);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------
// stage-level entry points
// ---------------------------------------------------------------------------
extern "C" int aw_stft_band(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples,
                            int64_t stride, int sample_rate, int normalize, float* d_mag,
                            float* d_phasor, void* stream) {
  AW_REQUIRE(ctx && d_audio && d_mag, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  if (make_dims(ctx, n_clips, n_samples, sample_rate, &d)) return 1;
  if (ensure(ctx->peakx, (size_t)n_clips * 8)) return 1;
  if (normalize) {
    if (launch_peak(ctx, d_audio, stride, n_samples, n_clips, (unsigned long long*)ctx->peakx.p, st)) return 1;
  } else {
    // peak = 1 - 1e-8 is not representable; use a packed peak of exactly 1.0 and accept the
    // 1e-8 relative bias (documented: normalize=0 is only approximately un-normalised)
    std::vector<unsigned long long> one(n_clips, ((unsigned long long)0x3f800000u << 32));
    AW_CUDA(cudaMemcpyAsync(ctx->peakx.p, one.data(), (size_t)n_clips * 8, cudaMemcpyHostToDevice, st));
    AW_CUDA(cudaStreamSynchronize(st));
  }
  AnaArgs a = ana_base(ctx, d);
  a.sig = d_audio; a.sig_stride = stride; a.len = n_samples;
  a.peak = (unsigned long long*)ctx->peakx.p;
  a.mag = d_mag; a.ph = (float2*)d_phasor;
  if (d_phasor) {
    // ANA_LOOP writes mag + phasor but divides twice; use INIT semantics without state:
    // route state writes to scratch buffers
    const size_t sp = (size_t)n_clips * d.T * d.nb;
    if (ensure(ctx->c, sp * 4) || ensure(ctx->m, sp * 4) || ensure(ctx->v, sp * 4) || ensure(ctx->cbest, sp * 4)) return 1;
    a.c = (float*)ctx->c.p; a.m = (float*)ctx->m.p; a.v = (float*)ctx->v.p; a.cbest = (float*)ctx->cbest.p;
    return launch_ana<ANA_INIT>(ctx, d, a, st);
  }
  return launch_ana<ANA_MAG>(ctx, d, a, st);
}

extern "C" int aw_istft_band(aw_ctx* ctx, const float* d_mag, const float* d_phasor, int n_clips,
                             int n_frames, int sample_rate, float* d_wave, void* stream) {
  AW_REQUIRE(ctx && d_mag && d_phasor && d_wave, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  if (make_dims(ctx, n_clips, AW_HOP * (n_frames - 1) + 1, sample_rate, &d)) return 1;
  AW_REQUIRE(d.T == n_frames, "internal: frame count");
  if (ensure(ctx->accum, acc_doubles(d) * 8)) return 1;
  if (ensure(ctx->yoob, (size_t)n_clips * d.L * 4)) return 1;
  AW_CUDA(cudaMemsetAsync(ctx->yoob.p, 0, (size_t)n_clips * d.L * 4, st));
  const Acc acc = acc_view(ctx, d);
  if (begin_pass(ctx, n_clips, nullptr, st)) return 1;
  SynArgs s = syn_base(ctx, d);
  s.amp = d_mag; s.ph = (const float2*)d_phasor; s.scale = 1.0f / AW_NFFT;
  s.y_oob = (float*)ctx->yoob.p; s.y = d_wave; s.peak_y = acc.peak_y;
  return launch_syn<SYN_WAVE>(ctx, d, s, st);
}

// full-band STFT / phase vocoder / iSTFT (time-stretch and pitch-shift attacks): no band, no peak, no
// synchronisation and nothing staged on the host
extern "C" int aw_stft_full(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples, int64_t stride,
                            float* d_spec, void* stream) {
  AW_REQUIRE(ctx && d_audio && d_spec, "null argument");
  AW_REQUIRE(n_clips >= 1 && n_clips <= 65535, "aw_stft_full: n_clips must be in [1, 65535] (got %d)", n_clips);
  AW_REQUIRE(n_samples > AW_NFFT, "aw_stft_full: clips must be longer than 1024 samples (got %d)", n_samples);
  AW_REQUIRE(stride >= n_samples, "aw_stft_full: stride must be >= n_samples");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  AnaArgs a;
  memset(&a, 0, sizeof(a));
  a.sig = d_audio; a.sig_stride = stride; a.len = n_samples;
  a.T = 1 + n_samples / AW_HOP; a.bin0 = 0; a.nbins = AW_NBINS_FULL;
  a.window = ctx->d_window; a.twiddle = ctx->d_twiddle; a.env256 = ctx->d_env256;
  a.ph = (float2*)d_spec;
  if (raise_smem_limit(ctx, (const void*)k_analysis<ANA_FULL, 0, 16>, AW_ANA_SMEM)) return 1;
  dim3 g((a.T + AW_ANA_FRAMES - 1) / AW_ANA_FRAMES, n_clips);
  prof_mark(ctx, st, "stft_full");
  k_analysis<ANA_FULL, 0, 16><<<g, 128, AW_ANA_SMEM, st>>>(a);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_phase_vocoder(aw_ctx* ctx, const float* d_spec, int n_clips, int n_frames, double rate,
                                int n_frames_out, float* d_out, void* stream) {
  AW_REQUIRE(ctx && d_spec && d_out, "null argument");
  AW_REQUIRE(std::isfinite(rate) && rate >= 0.25 && rate <= 4.0,
             "aw_phase_vocoder: rate must be finite and in [0.25, 4] (got %g)", rate);
  AW_REQUIRE(n_clips >= 1 && n_frames >= 1, "aw_phase_vocoder: n_clips and n_frames must be >= 1");
  const double want = ceil((double)n_frames / rate);        // len(np.arange(0, n_frames, rate))
  AW_REQUIRE((double)n_frames_out == want, "aw_phase_vocoder: n_frames_out must be ceil(n_frames / rate) = %.0f (got %d)",
             want, n_frames_out);
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  const long long threads = (long long)n_clips * AW_NBINS_FULL;
  prof_mark(ctx, st, "phase_vocoder");
  k_phase_vocoder<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>((const float2*)d_spec, n_clips, n_frames, rate,
                                                                      n_frames_out, (float2*)d_out);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_istft_full(aw_ctx* ctx, const float* d_spec, int n_clips, int n_frames, int n_out,
                             float* d_wave, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_spec && d_wave, "null argument");
  AW_REQUIRE(n_clips >= 1 && n_clips <= 65535, "aw_istft_full: n_clips must be in [1, 65535] (got %d)", n_clips);
  AW_REQUIRE(n_frames >= 1, "aw_istft_full: n_frames must be >= 1 (got %d)", n_frames);
  AW_REQUIRE(n_out >= 1, "aw_istft_full: n_out must be >= 1 (got %d)", n_out);
  AW_REQUIRE(out_stride >= n_out, "aw_istft_full: out_stride must be >= n_out");
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  // samples past 256 (n_frames - 1) + 512 lie outside every frame: torch.istft pads them with zeros
  const int n_ola = std::min(n_out, AW_HOP * (n_frames - 1) + AW_HALF);
  SynArgs s;
  memset(&s, 0, sizeof(s));
  s.ph = (const float2*)d_spec; s.T = n_frames; s.L = n_out; s.bin0 = 0; s.nbins = AW_NBINS_FULL;
  s.scale = 1.0f / AW_NFFT;
  s.window = ctx->d_window; s.twiddle = ctx->d_twiddle; s.env256 = ctx->d_env256;
  s.y = d_wave; s.x_stride = out_stride;
  // (the bin-group template arguments select the band loader, which this mode does not use)
  if (raise_smem_limit(ctx, (const void*)k_synthesis<SYN_FULL, 0, 15>, AW_SYN_SMEM)) return 1;
  const int hops = (AW_HALF + n_ola + AW_HOP - 1) / AW_HOP;   // padded-axis hops holding the output samples
  dim3 g((hops + AW_SYN_HOPS - 1) / AW_SYN_HOPS, n_clips);
  prof_mark(ctx, st, "istft_full");
  k_synthesis<SYN_FULL, 0, 15><<<g, 128, AW_SYN_SMEM, st>>>(s);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  if (n_out > n_ola)
    AW_CUDA(cudaMemset2DAsync(d_wave + n_ola, (size_t)out_stride * 4, 0, (size_t)(n_out - n_ola) * 4, n_clips, st));
  return 0;
}

extern "C" int aw_gemm(aw_ctx* ctx, const float* d_a, const float* d_b, float* d_d, int rows, int n,
                       int k, int prec, void* stream) {
  AW_REQUIRE(ctx && d_a && d_b && d_d, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  AW_REQUIRE(rows % 128 == 0 && k % 32 == 0 && n % 64 == 0, "aw_gemm: unsupported shape");
  AW_REQUIRE(n % bn_for(n) == 0, "aw_gemm: n must be a multiple of its tile (%d)", bn_for(n));
  cudaStream_t st = (cudaStream_t)stream;
  EpiArgsT<float> ep;
  memset(&ep, 0, sizeof(ep));
  ep.out = d_d; ep.ldo = n; ep.part = nullptr; ep.ldp = 0; ep.act = nullptr;
  if (prec == AW_PREC_FP32) return launch_exact<EPI_PLAIN>(ctx, d_a, d_b, rows, n, k, ep, st);
  CUtensorMap ma, mb;
  if (prec == AW_PREC_BF16) {
    AW_REQUIRE(k % 64 == 0, "aw_gemm: bf16 needs k %% 64 == 0");
    if (ensure(ctx->cvt_a, (size_t)rows * k * 2) || ensure(ctx->cvt_b, (size_t)n * k * 2)) return 1;
    k_to_bf16<<<256, 256, 0, st>>>(d_a, (__nv_bfloat16*)ctx->cvt_a.p, (size_t)rows * k);
    k_to_bf16<<<256, 256, 0, st>>>(d_b, (__nv_bfloat16*)ctx->cvt_b.p, (size_t)n * k);
    ctx->launches += 2;
    if (make_map(ctx, &ma, ctx->cvt_a.p, rows, k, 128, true)) return 1;
    if (make_map(ctx, &mb, ctx->cvt_b.p, n, k, bn_for(n), true)) return 1;
    return launch_tc_bn<__nv_bfloat16, float, EPI_PLAIN>(ctx, ma, mb, rows, n, k, ep, st);
  }
  if (make_map(ctx, &ma, d_a, rows, k, 128, false)) return 1;
  if (make_map(ctx, &mb, d_b, n, k, bn_for(n), false)) return 1;
  return launch_tc_bn<float, float, EPI_PLAIN>(ctx, ma, mb, rows, n, k, ep, st);
}

// ---------------------------------------------------------------------------
// attacks
// ---------------------------------------------------------------------------
// streaming passes: 4 samples per thread and access, enough CTAs to cover the 148 SMs several times
static dim3 ew_grid(int n, int n_clips) { return dim3(std::min((n + 4095) / 4096, std::max(8, 4096 / n_clips)), n_clips); }

extern "C" int aw_attack_pcm(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                             int bits, float* d_out, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  float S, lo, hi;
  switch (bits) {
    case 8: S = 127.f; lo = -128.f; hi = 127.f; break;
    case 12: S = 4095.f; lo = -4096.f; hi = 4095.f; break;
    case 16: S = 32767.f; lo = -32768.f; hi = 32767.f; break;
    case 24: S = 8388607.f; lo = -8388608.f; hi = 8388607.f; break;
    default: return set_error("Unsupported PCM bit depth: %d", bits);
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (ensure(ctx->peakx, (size_t)n_clips * 8)) return 1;
  if (launch_peak(ctx, d_in, in_stride, n, n_clips, (unsigned long long*)ctx->peakx.p, st)) return 1;
  prof_mark(ctx, (cudaStream_t)stream, "attack_pcm");
  k_attack_pcm<<<ew_grid(n, n_clips), 256, 0, st>>>(d_in, in_stride, n,
                                                    (unsigned long long*)ctx->peakx.p, S, lo, hi,
                                                    d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_decimate_interp(aw_ctx* ctx, const float* d_in, int n_clips, int n,
                                         int64_t in_stride, int factor, float* d_out,
                                         int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && factor >= 2, "bad argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "attack_decim_interp");
  k_attack_decim_interp<<<ew_grid(n, n_clips), 256, 0, (cudaStream_t)stream>>>(
      d_in, in_stride, n, factor, d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_upfirdn(aw_ctx* ctx, const float* d_in, int n_clips, int n_in,
                                 int64_t in_stride, const float* d_h_tf, int taps_per_phase, int up,
                                 int down, int first_out, int n_out, float* d_out,
                                 int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && d_h_tf, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "attack_upfirdn");
  if (up == 1 && down == 1 && taps_per_phase >= 1 && taps_per_phase <= AW_FIR_MAXTAPS) {   // FIR filters: register-tiled
    const int tiles = (n_out + AW_FIR_TILE - 1) / AW_FIR_TILE;
    k_fir_tiled<<<dim3((unsigned)std::max(1, std::min(tiles, 65535)), n_clips), 256, 0, (cudaStream_t)stream>>>(
        d_in, in_stride, n_in, d_h_tf, taps_per_phase, first_out, n_out, d_out, out_stride);
    ctx->launches++;
    AW_LAUNCH_CHECK();
    return 0;
  }
  k_upfirdn<<<ew_grid(n_out, n_clips), 256, 0, (cudaStream_t)stream>>>(
      d_in, in_stride, n_in, d_h_tf, taps_per_phase, up, down, first_out, n_out, d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

static int fill_iir(IirArgs& a, const double* b, const double* av, const double* zi, int order) {
  AW_REQUIRE(order >= 1 && order <= AW_IIR_MAXORD, "IIR order %d unsupported (max %d)", order,
             AW_IIR_MAXORD);
  memset(&a, 0, sizeof(a));
  for (int i = 0; i <= order; ++i) { a.b[i] = b[i] / av[0]; a.a[i] = av[i] / av[0]; }
  if (zi) for (int i = 0; i < order; ++i) a.zi[i] = zi[i];
  a.order = order;
  return 0;
}

#define AW_IIR_CHUNK 2048
// warm > 0: chunk-parallel scan with `warm` look-back samples; warm <= 0: sequential
// (one thread per clip), bit-identical to scipy's recurrence.
static void iir_plan(IirArgs& ia, int n, int n_clips, int warm, dim3* grid) {
  ia.n = n; ia.n_clips = n_clips;
  if (warm > 0) {
    ia.chunk = std::max(AW_IIR_CHUNK, (warm / 2 + 255) / 256 * 256);
    ia.warm = warm;
  } else {
    ia.chunk = n;
    ia.warm = 0;
  }
  ia.n_chunks = (n + ia.chunk - 1) / ia.chunk;
  const long long items = (long long)n_clips * ia.n_chunks;
  *grid = dim3((unsigned)((items + 127) / 128));
}

extern "C" int aw_attack_lfilter(aw_ctx* ctx, const float* d_in, int n_clips, int n,
                                 int64_t in_stride, const double* b, const double* a, int order,
                                 int warm, float* d_out, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && b && a, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  IirArgs ia;
  if (fill_iir(ia, b, a, nullptr, order)) return 1;
  dim3 g;
  iir_plan(ia, n, n_clips, warm, &g);
  ia.x32 = d_in; ia.sx32 = in_stride; ia.n_x = n;
  ia.o32 = d_out; ia.so32 = out_stride;
  prof_mark(ctx, (cudaStream_t)stream, "attack_lfilter");
  if (warm <= 0)
    k_iir_seq8<IIR_SRC_F32, IIR_DST_F32><<<(n_clips + 3) / 4, 32, 0, (cudaStream_t)stream>>>(ia);
  else
    k_iir<IIR_SRC_F32, IIR_DST_F32><<<g, 128, 0, (cudaStream_t)stream>>>(ia);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_filtfilt(aw_ctx* ctx, const float* d_in, int n_clips, int n,
                                  int64_t in_stride, const double* b, const double* a,
                                  const double* zi, int order, int warm, float* d_out,
                                  int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && b && a && zi, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  const int pad = 3 * (order + 1);
  AW_REQUIRE(n > pad, "The length of the input vector x must be greater than padlen, which is %d.", pad);
  cudaStream_t st = (cudaStream_t)stream;
  const int next = n + 2 * pad;
  // two float64 scratch rows per clip, parked in the (otherwise idle) gradient buffers
  if (ensure(ctx->ga, (size_t)n_clips * next * 8)) return 1;
  ctx->ws_rows = 0;   // tensor maps over ga are stale now
  IirArgs ia;
  if (fill_iir(ia, b, a, zi, order)) return 1;
  dim3 g;
  iir_plan(ia, next, n_clips, warm, &g);
  ia.padlen = pad; ia.use_zi = 1;
  ia.x32 = d_in; ia.sx32 = in_stride; ia.n_x = n;
  ia.o64 = (double*)ctx->ga.p; ia.so64 = next;
  prof_mark(ctx, (cudaStream_t)stream, "attack_filtfilt_fwd");
  if (warm <= 0)
    k_iir_seq8<IIR_SRC_ODDEXT, IIR_DST_F64><<<(n_clips + 3) / 4, 32, 0, st>>>(ia);
  else
    k_iir<IIR_SRC_ODDEXT, IIR_DST_F64><<<g, 128, 0, st>>>(ia);
  IirArgs ib = ia;
  ib.x64 = (double*)ctx->ga.p; ib.sx64 = next;
  ib.o32 = d_out; ib.so32 = out_stride;
  prof_mark(ctx, (cudaStream_t)stream, "attack_filtfilt_bwd");
  if (warm <= 0)
    k_iir_seq8<IIR_SRC_REV_F64, IIR_DST_REVTRIM_F32><<<(n_clips + 3) / 4, 32, 0, st>>>(ib);
  else
    k_iir<IIR_SRC_REV_F64, IIR_DST_REVTRIM_F32><<<g, 128, 0, st>>>(ib);
  ctx->launches += 2;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_delete(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                                const int32_t* d_start, int n_delete, float* d_out,
                                int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && d_start && n_delete >= 0 && n_delete < n, "bad argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "attack_delete");
  k_attack_delete<<<ew_grid(n - n_delete, n_clips), 256, 0, (cudaStream_t)stream>>>(
      d_in, in_stride, n - n_delete, d_start, n_delete, d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_suppress(aw_ctx* ctx, const float* d_in, int n_clips, int n,
                                  int64_t in_stride, const int32_t* d_start, int n_zero,
                                  float* d_out, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && d_start, "bad argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "attack_suppress");
  k_attack_suppress<<<ew_grid(n, n_clips), 256, 0, (cudaStream_t)stream>>>(
      d_in, in_stride, n, d_start, n_zero, d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_cropout(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                                 int n_drop, float* d_out, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out && n_drop >= 0 && n_drop < n, "bad argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "attack_affine");
  k_attack_affine<<<ew_grid(n - n_drop, n_clips), 256, 0, (cudaStream_t)stream>>>(
      d_in + n_drop, in_stride, n - n_drop, 1.0f, nullptr, 0, 0.f, d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_affine(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                                float gain, const float* d_noise, int64_t noise_stride, float sigma,
                                float* d_out, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_out, "null argument");
  if (ctx) cudaSetDevice(ctx->device);
  prof_mark(ctx, (cudaStream_t)stream, "attack_affine");
  k_attack_affine<<<ew_grid(n, n_clips), 256, 0, (cudaStream_t)stream>>>(
      d_in, in_stride, n, gain, d_noise, noise_stride, sigma, d_out, out_stride);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

extern "C" int aw_attack_spectral_quantize(aw_ctx* ctx, const float* d_mag, int n_clips, int n_frames, int nbins,
                                           float step_db, float floor_db, float* d_dmag, void* stream) {
  AW_REQUIRE(ctx && d_mag && d_dmag, "null argument");
  AW_REQUIRE(step_db > 0.f && nbins >= 1 && nbins <= AW_MAX_BINS, "bad argument");
  if (ctx) cudaSetDevice(ctx->device);
  // 20 log10(m) / step = log2(m) * k_log ;  10^(step * r / 20) = 2^(r * k_exp)   (float32, as the oracle)
  const float k_log = (float)(20.0 * log10(2.0) / (double)step_db);
  const float k_exp = (float)((double)step_db / (20.0 * log10(2.0)));
  const float ratio = (float)pow(10.0, (double)floor_db / 20.0);
  const long long frames = (long long)n_clips * n_frames;
  prof_mark(ctx, (cudaStream_t)stream, "attack_spec_quant");
  k_spectral_quantize<<<(unsigned)((frames + 3) / 4), 128, 0, (cudaStream_t)stream>>>(d_mag, frames, nbins, k_log,
                                                                                   k_exp, ratio, d_dmag);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}

// reverberation / echo: causal convolution by partitioned overlap-save (conv.cuh)
extern "C" int aw_attack_convolve(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                                  const float* d_spec, int n_filters, int n_parts, const int32_t* filter_of_clip,
                                  float* d_out, int64_t out_stride, void* stream) {
  AW_REQUIRE(ctx && d_in && d_spec && d_out, "null argument");
  AW_REQUIRE(n_clips >= 1 && n_clips <= 65535, "aw_attack_convolve: n_clips must be in [1, 65535] (got %d)", n_clips);
  // sample indices of the last block reach n + 1535 in 32-bit arithmetic
  AW_REQUIRE(n >= 1 && n <= INT_MAX - 2048, "aw_attack_convolve: n must be in [1, %d] (got %d)", INT_MAX - 2048, n);
  AW_REQUIRE(in_stride >= n && out_stride >= n, "aw_attack_convolve: strides must be >= n");
  AW_REQUIRE(n_filters >= 1, "aw_attack_convolve: n_filters must be >= 1 (got %d)", n_filters);
  AW_REQUIRE(n_parts >= 1 && n_parts <= AW_CONV_MAXPARTS, "aw_attack_convolve: n_parts must be in [1, %d] (got %d)",
             AW_CONV_MAXPARTS, n_parts);
  if (filter_of_clip)
    for (int i = 0; i < n_clips; ++i)
      AW_REQUIRE(filter_of_clip[i] >= 0 && filter_of_clip[i] < n_filters,
                 "aw_attack_convolve: filter_of_clip[%d] = %d must be in [0, %d)", i, filter_of_clip[i], n_filters);
  cudaSetDevice(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int nb = (n + AW_CONV_P - 1) / AW_CONV_P;
  if (ensure(ctx->conv_x, (size_t)n_clips * nb * AW_CONV_SLOTS * sizeof(float2))) return 1;
  if (filter_of_clip) {
    if (ensure(ctx->conv_idx, (size_t)n_clips * 4)) return 1;
    AW_CUDA(cudaMemcpyAsync(ctx->conv_idx.p, filter_of_clip, (size_t)n_clips * 4, cudaMemcpyHostToDevice, st));
  }
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.x = d_in; a.x_stride = in_stride; a.n = n; a.nb = nb;
  a.X = (float2*)ctx->conv_x.p;
  a.H = (const float2*)d_spec; a.K = n_parts;
  a.filter = filter_of_clip ? (const int*)ctx->conv_idx.p : nullptr;
  a.twiddle = ctx->d_twiddle;
  a.y = d_out; a.y_stride = out_stride;
  prof_mark(ctx, st, "conv_fwd");
  k_conv_fwd<<<dim3((nb + AW_CONV_FWD_BLOCKS - 1) / AW_CONV_FWD_BLOCKS, n_clips), 128, AW_CONV_FWD_SMEM, st>>>(a);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  if (raise_smem_limit(ctx, (const void*)k_conv_mac_inv, AW_CONV_INV_SMEM)) return 1;
  prof_mark(ctx, st, "conv_mac_inv");
  k_conv_mac_inv<<<dim3((nb + AW_CONV_R - 1) / AW_CONV_R, n_clips), 512, AW_CONV_INV_SMEM, st>>>(a);
  ctx->launches++;
  AW_LAUNCH_CHECK();
  return 0;
}
