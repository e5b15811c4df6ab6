// The backward K = 64 layer (dP3 = dH4 W3, 64 -> 1024 channels; reference detection/modules/conv1d.py:38-42
// through autograd) as a pure streaming problem.
//
// Its GEMM is 30 GFLOP against 470 MB of activations P3 that the epilogue has to read (LeakyReLU', recovery of
// the InstanceNorm output) and, in the apply pass, 470 MB of dH3 it has to write: the tensor pipe idles and the
// time is the epilogue's memory traffic.  In k_gemm_tc that traffic is issued by eight epilogue warps with
// ordinary loads -- at most one 2 KB chunk per warp in flight (the hardware scoreboards are too few to keep
// more outstanding without the consumer of chunk c waiting for chunk c+1, see DESIGN.md), i.e. ~32 KB per SM:
// 2.3 TB/s, a third of HBM.  Here the P3 tile travels like an operand: the TMA producer streams it into a
// three-slot shared-memory ring (96 KB in flight per SM, no registers, no scoreboards), the epilogue warps read
// it in the accumulator's own layout (lane = row; the 128-byte swizzle makes that conflict-free, so there is no
// transpose staging either), and the apply pass hands its output tile back to TMA as a bulk tensor store.
//
//   EPI_BWD_STATS  column sums  sum_r dHhat, sum_r dHhat * Hhat  per 128-row tile (nothing stored)
//   EPI_BWD_APPLY  dH = rstd (dHhat - a1 - Hhat a2), pad rows 0, stored through shared memory + TMA
//
// 128 x 128 tiles, one 64-wide k-block per MMA group, fp32 accumulators double-buffered in TMEM (256 columns),
// 16-bit operands / activations only (the TF32 path keeps k_gemm_tc).  warp 0 TMA, warp 1 MMA, warps 2..9 epilogue.
#pragma once
#include "gemm.cuh"

namespace aw {

#define AW_G64_BN 128
#define AW_G64_NST 2            // operand stages (K = 64: one k-block per tile)
// activation tiles in flight: three for the statistics pass; the apply pass also holds two output tiles
__host__ __device__ constexpr int gemm64_nact(int epi) { return epi == EPI_BWD_APPLY ? 2 : 3; }
#define AW_G64_STAGE (128 * 128 + AW_G64_BN * 128)     // A 16 KB + B 16 KB
#define AW_G64_TILE (128 * AW_G64_BN * 2)              // a 128 x 128 16-bit tile = two 64-column boxes

template <int EPI>
constexpr int gemm64_smem() {
  return 1024 + AW_G64_NST * AW_G64_STAGE + gemm64_nact(EPI) * AW_G64_TILE +
         (EPI == EPI_BWD_APPLY ? 2 * AW_G64_TILE : 0) + 256 /*barriers*/ +
         (EPI == EPI_BWD_APPLY ? 2 * AW_G64_BN * 16 /*stats*/ : 2 * 2 * 4 * AW_G64_BN * 4 /*partials*/);
}

struct Gemm64Args {
  float* part; int ldp;          // STATS: [row_tiles][ldp][2]
  const float* stat;             // APPLY: [clip][ldo][2] (mean, rstd) of the layer's forward InstanceNorm
  const float* bstat;            // APPLY: [clip][ldo][2] (a1, a2)
  int ldo;                       // channels of the layer (row length of act / out)
  int tiles_per_clip, Tp;
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ float2 unpack16(uint32_t w, __half) {
  return __half22float2(*reinterpret_cast<const __half2*>(&w));
}
__device__ __forceinline__ float2 unpack16(uint32_t w, __nv_bfloat16) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t pack16(float a, float b, __half) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack16(float a, float b, __nv_bfloat16) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

template <typename T, int EPI>
__global__ void __launch_bounds__(320, 1)
k_gemm_bwd64(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
             const __grid_constant__ CUtensorMap map_act, const __grid_constant__ CUtensorMap map_out, int K,
             int n_row_tiles, int n_col_tiles, Gemm64Args ep) {
  static_assert(sizeof(T) == 2, "16-bit activations only");
  static_assert(EPI == EPI_BWD_STATS || EPI == EPI_BWD_APPLY, "backward small-K epilogues only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int BN = AW_G64_BN, BK = 64, NST = AW_G64_NST, NACT = gemm64_nact(EPI);
  uint8_t* stages = smem;
  uint8_t* act_ring = stages + NST * AW_G64_STAGE;
  uint8_t* out_buf = act_ring + NACT * AW_G64_TILE;                        // APPLY: 2 tiles
  uint8_t* tail = out_buf + (EPI == EPI_BWD_APPLY ? 2 * AW_G64_TILE : 0);
  uint64_t* full = reinterpret_cast<uint64_t*>(tail);                      // [NST]
  uint64_t* empty = full + NST;                                            // [NST]
  uint64_t* tfull = empty + NST;                                           // [2]
  uint64_t* tempty = tfull + 2;                                            // [2]
  uint64_t* afull = tempty + 2;                                            // [NACT]
  uint64_t* aempty = afull + NACT;                                         // [NACT]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty + NACT);
  float4* s_stat = reinterpret_cast<float4*>(tail + 256);                  // APPLY: [2][BN] (mean, rstd, a1, a2)
  float* s_part = reinterpret_cast<float*>(tail + 256);                    // STATS: [2][2][4][BN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = K / BK;
  const int n_tiles = n_row_tiles * n_col_tiles;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_act) : "memory");
    if (EPI == EPI_BWD_APPLY) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_out) : "memory");
    for (int s = 0; s < NST; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull + b, 1); mbar_init(tempty + b, 8); }
    for (int s = 0; s < NACT; ++s) { mbar_init(afull + s, 1); mbar_init(aempty + s, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(2 * BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------- TMA producer: operands and the activation tile of every tile -------------------
    if (lane == 0) {
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int row0 = (tile / n_col_tiles) * 128, n0 = (tile % n_col_tiles) * BN;
        const int as = it % NACT;
        mbar_wait(aempty + as, ((it / NACT) & 1) ^ 1);
        mbar_expect_tx(afull + as, AW_G64_TILE);
        tma_load_2d(act_ring + as * AW_G64_TILE, &map_act, afull + as, n0, row0);
        tma_load_2d(act_ring + as * AW_G64_TILE + AW_G64_TILE / 2, &map_act, afull + as, n0 + 64, row0);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(empty + s, ph ^ 1);
          mbar_expect_tx(full + s, AW_G64_STAGE);
          tma_load_2d(stages + s * AW_G64_STAGE, &map_a, full + s, kb * BK, row0);
          tma_load_2d(stages + s * AW_G64_STAGE + 128 * 128, &map_b, full + s, kb * BK, n0);
          if (++s == NST) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------ MMA issuer ------------------------------------------
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (GemmElem<T>::FMT << 7) | (GemmElem<T>::FMT << 10) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      int s = 0, it = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int ab = it & 1;
        mbar_wait(tempty + ab, ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(ab * BN);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(full + s, ph);
          tc_fence_after();
          const uint64_t ad = make_sw128_desc(smem_u32(stages + s * AW_G64_STAGE));
          const uint64_t bd = make_sw128_desc(smem_u32(stages + s * AW_G64_STAGE + 128 * 128));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            GemmElem<T>::mma(d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (kb | k) != 0);
          tc_commit(empty + s);
          if (++s == NST) { s = 0; ph ^= 1; }
        }
        tc_commit(tfull + ab);
      }
    }
  } else {
    // -------------------------------------------- epilogue --------------------------------------------
    const int e = warp - 2, q = warp & 3, half = e >> 2;
    const int t = threadIdx.x - 64;                                  // 0..255
    const int row = q * 32 + lane;                                   // row of the tile = TMEM lane
    // swizzled byte offset of 16-byte chunk j (0..7) of this row inside a 64-column box
    const uint32_t row_off = (uint32_t)row * 128u;
    const uint32_t rx = (uint32_t)(row & 7);
    // statistics of a tile: thread t stages column t / 2, (t & 1 ? bstat : stat)
    auto stat_fetch = [&](int tile_) -> float2 {
      const int rt = tile_ / n_col_tiles, n0_ = (tile_ % n_col_tiles) * BN;
      const long long o = ((long long)(rt / ep.tiles_per_clip) * ep.ldo + n0_ + (t >> 1)) * 2;
      return __ldg(reinterpret_cast<const float2*>(((t & 1) ? ep.bstat : ep.stat) + o));
    };
    float2 st_next = make_float2(0.f, 0.f);
    if (EPI == EPI_BWD_APPLY && (int)blockIdx.x < n_tiles) {
      const float2 s0 = stat_fetch(blockIdx.x);
      reinterpret_cast<float2*>(s_stat)[(0 * BN + (t >> 1)) * 2 + (t & 1)] = s0;
    }
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int ab = it & 1, as = it % NACT;
      const int row_tile = tile / n_col_tiles, n0 = (tile % n_col_tiles) * BN;
      const bool has_next = tile + (int)gridDim.x < n_tiles;
      if (EPI == EPI_BWD_APPLY) {
        if (has_next) st_next = stat_fetch(tile + gridDim.x);          // lands while this tile is processed
        // the bulk store that read out_buf[ab] two tiles ago must have finished reading shared memory
        if (t == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");                   // s_stat[ab] complete; out_buf[ab] free
      const int clip = row_tile / ep.tiles_per_clip;
      const bool valid = (row_tile - clip * ep.tiles_per_clip) * 128 + row < ep.Tp;
      const uint8_t* abox = act_ring + as * AW_G64_TILE + half * (AW_G64_TILE / 2) + row_off;
      uint8_t* obox = out_buf + ab * AW_G64_TILE + half * (AW_G64_TILE / 2) + row_off;
      float* sp = s_part + ab * (2 * 4 * BN);
      mbar_wait(afull + as, (it / NACT) & 1);
      mbar_wait(tfull + ab, (it >> 1) & 1);
      tc_fence_after();
      uint32_t vbuf[2][32];
      tc_ld32_async(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * BN + half * 64), vbuf[0]);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t (&v)[32] = vbuf[c];
        tc_wait_ld(v);
        if (c == 0) {
          tc_ld32_async(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * BN + half * 64 + 32), vbuf[1]);
        } else {                                                       // accumulator fully read: hand it back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(tempty + ab)) : "memory");
        }
        // this row's 32 activations of the chunk: four 16-byte pieces of the swizzled box
        uint4 av[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          av[j] = *reinterpret_cast<const uint4*>(abox + ((((uint32_t)(c * 4 + j)) ^ rx) << 4));
        const uint32_t aw[16] = {av[0].x, av[0].y, av[0].z, av[0].w, av[1].x, av[1].y, av[1].z, av[1].w,
                                 av[2].x, av[2].y, av[2].z, av[2].w, av[3].x, av[3].y, av[3].z, av[3].w};
        if (EPI == EPI_BWD_APPLY) {
          const float4* ss = s_stat + ab * BN + half * 64 + c * 32;
          uint32_t ow[16];
#pragma unroll
          for (int k2 = 0; k2 < 16; ++k2) {
            const float2 p = unpack16(aw[k2], T());
            float o[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int k = 2 * k2 + u;
              const float pv = u ? p.y : p.x, w = __uint_as_float(v[k]);
              const bool pos = pv > 0.f;
              const float g = pos ? w : AW_LEAKY * w;                  // d(IN out) = dP * LeakyReLU'(P)
              const float hh = pos ? pv : pv * (1.0f / AW_LEAKY);      // IN out recovered from P
              const float4 s4 = ss[k];                                 // broadcast: (mean, rstd, a1, a2) of the column
              const float ov = s4.y * (g - s4.z - hh * s4.w);          // dH = rstd (dHhat - a1 - Hhat a2)
              o[u] = valid ? ov : 0.f;
            }
            ow[k2] = pack16(o[0], o[1], T());
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<uint4*>(obox + ((((uint32_t)(c * 4 + j)) ^ rx) << 4)) =
                make_uint4(ow[4 * j], ow[4 * j + 1], ow[4 * j + 2], ow[4 * j + 3]);
        } else {
          float g[32], hg[32];                                         // dHhat, Hhat * dHhat
#pragma unroll
          for (int k2 = 0; k2 < 16; ++k2) {
            const float2 p = unpack16(aw[k2], T());
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int k = 2 * k2 + u;
              const float pv = u ? p.y : p.x, w = __uint_as_float(v[k]);
              const bool pos = pv > 0.f;
              g[k] = pos ? w : AW_LEAKY * w;
              hg[k] = (pos ? pv : pv * (1.0f / AW_LEAKY)) * g[k];
            }
          }
          const float s1 = warp_colsum32(g, lane), s2 = warp_colsum32(hg, lane);   // lane l: column l of the chunk
          sp[(0 * 4 + q) * BN + half * 64 + c * 32 + lane] = s1;
          sp[(1 * 4 + q) * BN + half * 64 + c * 32 + lane] = s2;
        }
      }
      // the activation slot is free for the producer
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(aempty + as)) : "memory");
      if (EPI == EPI_BWD_APPLY) {
        if (has_next) reinterpret_cast<float2*>(s_stat)[((ab ^ 1) * BN + (t >> 1)) * 2 + (t & 1)] = st_next;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to the bulk store
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (t == 0) {
          tma_store_2d(&map_out, out_buf + ab * AW_G64_TILE, n0, row_tile * 128);
          tma_store_2d(&map_out, out_buf + ab * AW_G64_TILE + AW_G64_TILE / 2, n0 + 64, row_tile * 128);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      } else {
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (t < BN) {
          float s1 = 0.f, s2 = 0.f;
#pragma unroll
          for (int w4 = 0; w4 < 4; ++w4) {
            s1 += sp[(0 * 4 + w4) * BN + t];
            s2 += sp[(1 * 4 + w4) * BN + t];
          }
          float* p = ep.part + ((long long)row_tile * ep.ldp + n0 + t) * 2;
          p[0] = s1;
          p[1] = s2;
        }
      }
    }
    if (EPI == EPI_BWD_APPLY && t == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * BN) : "memory");
}

}  // namespace aw
