// gemm_tc.cu -- bf16 tcgen05 GEMM with fused epilogues for the BERT encoder (sm_100a).
//
//   C[M, N] = epilogue( A[M, K] * W[N, K]^T + bias[N] )          A, W, C bf16; fp32 accumulate
//
// Replaces the nn.Linear calls inside SentenceTransformer.encode (reference call sites
// services/embedding_service.py:81,97-102,120): QKV projection, attention output projection,
// FFN up (+ erf-GELU) and FFN down (+ residual).  Persistent kernel: one CTA PAIR per TPC (cluster of 2,
// tcgen05 cta_group::2) walks 256 x 256 output tiles -- each CTA loads its own 128 rows of A and half of the W
// tile through TMA (128-byte swizzle) into a 5-stage mbarrier ring, the leader issues tcgen05.mma
// (M=256, N=256, K=16), the accumulators sit in TMEM, double-buffered (2 x 256 columns) so the epilogue of tile i
// overlaps the MMAs of tile i+1.  (NC = 1: single CTAs on 128 x 256 tiles, the A/B reference and the fallback.)
//
// Epilogue: thread == TMEM lane == output row, so a direct global store would scatter 16-byte
// pieces over 32 rows per instruction (ncu r01b: the K=768 GEMMs were bound by exactly that:
// 49 % / 68 % of peak for the O and QKV projections against 89 % for K=3072).  Instead each
// column-half group of 4 warps owns one 128 x 64 staging box in shared memory (128-byte
// swizzle, conflict-free 16-byte accesses), converts its accumulators into it and one thread
// hands the box to TMA (cp.async.bulk.tensor store: full 128-byte lines to L2).  The residual
// of the O / FFN-down projections arrives the same way: a TMA load of the matching box of the
// residual stream into the staging box, prefetched as soon as the previous store has drained.
//
// Warp roles (320 threads): warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer,
// warps 2..9 epilogue (lane quarter = warp % 4, column half = (warp - 2) / 4).
//
// Deferred LayerNorm.  The two LayerNorm launches per layer were 9 % of the encoder (HBM-bound, r01c launch
// list); they are folded into the GEMMs on either side instead.  A GEMM whose output feeds a LayerNorm
// (O projection, FFN down) also emits per-row partial (sum, sum of squares) of its 128 output columns per
// column half -- [N/128][rows] float2, no atomics, deterministic; a consumer adds the SLOTS = H / 128 partials of a row
// (6 at hidden 768, 8 at 1024: a template parameter, so the sum stays straight-line code).  A GEMM that READS a LayerNorm output
// takes the un-normalised stream x as A with W' = W diag(gamma) pre-folded on the host and applies
//   y = rs * (x W'^T) - rs * mu * c + b',   c[n] = sum_k W'[n,k],  b' = b + W beta
// per row in its epilogue (the identity CUTLASS's gemm+layernorm fusion uses); a residual epilogue that needs
// LN(x) itself rebuilds it from the TMA-loaded box: (x - mu) rs gamma[n] (+ beta folded into the bias).
//
// Roofline: bf16 tensor pipe; 2*M*N*K flops per launch.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "encoder_kernels.h"
#include "ptx.cuh"

namespace icd {
namespace {

constexpr int BM = 128;  // output rows per CTA (TMEM lanes)
constexpr int BN = 256;  // output columns per tile (TMEM columns per accumulator buffer)
constexpr int BK = 64;
constexpr int kABytes = BM * BK * 2;  // 16 KiB
constexpr int kMaxStages = 6;
// NC = CTAs per tile: 1 -> 128 x 256 tiles; 2 -> a CTA pair (cluster of 2, cta_group::2) owns a 256 x 256 tile: each
// CTA loads its own 128 rows of A and HALF of the W tile (128 of the 256 N rows), the pair's MMAs read both halves,
// so the L2 -> shared-memory traffic per flop drops by a third (48 -> 32 KiB per CTA per K block)
template <int NC>
struct Cfg {
  static constexpr int kBBytes = (BN / NC) * BK * 2;      // 32 / 16 KiB
  static constexpr int kStageBytes = kABytes + kBBytes;   // 48 / 32 KiB
  static constexpr int kStages = NC == 1 ? 3 : 5;         // 144 / 160 KiB of stages
};
constexpr int kThreads = 320;
constexpr int kEpiWarps = 8;
constexpr int kTmemCols = 512;
constexpr int kBoxCols = 64;                    // staging box: 128 rows x 64 bf16 (128-byte rows)
constexpr int kBoxBytes = BM * kBoxCols * 2;    // 16 KiB
constexpr int kBoxesPerHalf = (BN / 2) / kBoxCols;  // 2
constexpr int kStagingBoxes = 4;                // 2 column halves x 2 (double-buffered: a store drains while the next box fills)
constexpr int kBiasBytes = 2 * 2 * (BN / 2) * 4;  // [half][bias | second column vector][128] fp32
template <int NC>
constexpr int smem_bytes() {
  return Cfg<NC>::kStages * Cfg<NC>::kStageBytes + kStagingBoxes * kBoxBytes + kBiasBytes + 256 /*barriers*/;
}
static_assert(smem_bytes<1>() <= 227 * 1024 && smem_bytes<2>() <= 227 * 1024, "shared memory budget");

struct GemmParams {
  const float* bias;  // [N]
  const float* vec2;  // [N] c (A is a pre-LayerNorm stream) or gamma (residual is one); null otherwise
  const float2* stats_in;  // [slots_in][stats_stride] partial (sum, sum sq) of the rows of A / of the residual, or null
  float2* stats_out;       // [N / 128][stats_stride] partials of this GEMM's output rows, or null
  int stats_stride;
  float inv_h, eps;   // 1 / (row length the statistics cover), LayerNorm eps
  int M, N, K;
  int epi;            // GemmEpilogue
};

// named barrier over the 128 threads of one column-half epilogue group (ids 1 and 2; 0 is __syncthreads)
__device__ __forceinline__ void group_sync(int half) {
  asm volatile("bar.sync %0, 128;" ::"r"(half + 1) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// EPI / LNIN / STATS are compile-time so that the 32 columns of an accumulator chunk form one straight-line block
// (r01d: with run-time epilogue switches every 8-column group was fenced by uniform branches, and the shared-memory
// loads of the column vectors stalled their first use -- 2 epilogue warps per scheduler cannot hide that).
//   LNIN: A is an un-normalised stream, apply its row statistics (QKV / FFN-up in deferred-LayerNorm mode)
//   STATS: emit the row statistics of the output (residual epilogues in deferred-LayerNorm mode)
//   SLOTS: 128-column partials per row of the incoming statistics (hidden size / 128)
template <int NC, int EPI, bool LNIN, bool STATS, int SLOTS>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_res,
               const GemmParams p) {
  // no static shared memory in this kernel: the dynamic window starts 1024-aligned (128-byte swizzle atoms)
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int kStages = Cfg<NC>::kStages, kStageBytes = Cfg<NC>::kStageBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* stage_c = smem + kStages * kStageBytes;  // [2 halves][2 buffers][128 x 64 bf16], 1024-aligned
  float* bias_s = reinterpret_cast<float*>(stage_c + kStagingBoxes * kBoxBytes);  // [2 halves][2][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_c + kStagingBoxes * kBoxBytes + kBiasBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tfull_bar = bars + 2 * kMaxStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* res_bar = tempty_bar + 2;  // [2 halves][2 buffers] residual box landed
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(res_bar + 4);

  // tile walk: a tile is BM * NC rows x BN columns; `unit` = CTA (NC = 1) or CTA pair (NC = 2)
  const uint32_t rank = NC == 2 ? ptx::cluster_ctarank() : 0u;  // 0 = leader of the pair (issues the MMAs)
  const int unit = (int)blockIdx.x / NC, units = (int)gridDim.x / NC;
  const int m_tiles = (p.M + BM * NC - 1) / (BM * NC);
  const int n_tiles = p.N / BN;
  const int tiles = m_tiles * n_tiles;
  const int nkb = p.K / BK;

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
    ptx::prefetch_tmap(&tmap_out);
    if (EPI == EPI_BIAS_RESIDUAL) ptx::prefetch_tmap(&tmap_res);
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(ptx::smem_u32(&full_bar[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(ptx::smem_u32(&tfull_bar[b]), 1);
      ptx::mbar_init(ptx::smem_u32(&tempty_bar[b]), kEpiWarps * NC);  // the epilogue warps of every CTA of the tile
      ptx::mbar_init(ptx::smem_u32(&res_bar[2 * b]), 1);
      ptx::mbar_init(ptx::smem_u32(&res_bar[2 * b + 1]), 1);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    if (NC == 2) {
      ptx::tmem_alloc_pair(ptx::smem_u32(tmem_holder), kTmemCols);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(ptx::smem_u32(tmem_holder), kTmemCols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if (NC == 2) ptx::cluster_sync(); else __syncthreads();  // barriers of BOTH CTAs are initialised from here on
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  // prologue done: the next kernel of the forward may start its own; A, the residual and the LayerNorm statistics are
  // outputs of the previous kernel, so nothing is loaded before it has completed
  ptx::griddep_launch();
  ptx::griddep_wait();

  if (warp == 0) {
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = unit; tile < tiles; tile += units) {
        const int m0 = (tile / n_tiles) * (BM * NC) + (int)rank * BM;          // this CTA's rows of A
        const int nb0 = (tile % n_tiles) * BN + (int)rank * (BN / NC);       // this CTA's share of the W tile
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(ptx::smem_u32(&empty_bar[stage]), phase ^ 1);
          unsigned char* sa = smem + (size_t)stage * kStageBytes;
          if (NC == 1) {
            const uint32_t fb = ptx::smem_u32(&full_bar[stage]);
            ptx::mbar_expect_tx(fb, kStageBytes);
            ptx::tma_load_2d(ptx::smem_u32(sa), &tmap_a, fb, kb * BK, m0);
            ptx::tma_load_2d(ptx::smem_u32(sa + kABytes), &tmap_b, fb, kb * BK, nb0);
          } else {
            // both CTAs' bytes are counted on the LEADER's barrier (only its MMA thread waits for the stage)
            if (rank == 0) ptx::mbar_expect_tx(ptx::smem_u32(&full_bar[stage]), 2 * kStageBytes);
            const uint32_t fb = ptx::mapa(ptx::smem_u32(&full_bar[stage]), 0);
            ptx::tma_load_2d_pair(ptx::smem_u32(sa), &tmap_a, fb, kb * BK, m0);
            ptx::tma_load_2d_pair(ptx::smem_u32(sa + kABytes), &tmap_b, fb, kb * BK, nb0);
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(BM * NC, BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = unit; tile < tiles; tile += units, ++it) {
        const int buf = it & 1;
        ptx::mbar_wait(ptx::smem_u32(&tempty_bar[buf]), ((it >> 1) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(ptx::smem_u32(&full_bar[stage]), phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + (size_t)stage * kStageBytes);
          const uint32_t sb = sa + kABytes;
#pragma unroll
          for (int k4 = 0; k4 < BK / 16; ++k4) {
            if (NC == 1)
              ptx::mma_ss(d_tmem, ptx::make_desc_k128(sa + k4 * 32), ptx::make_desc_k128(sb + k4 * 32), idesc,
                          (kb | k4) ? 1u : 0u);
            else
              ptx::mma_ss_pair(d_tmem, ptx::make_desc_k128(sa + k4 * 32), ptx::make_desc_k128(sb + k4 * 32), idesc,
                               (kb | k4) ? 1u : 0u);
          }
          // frees the stage in both CTAs when the MMAs retire
          if (NC == 1) ptx::tc_commit(ptx::smem_u32(&empty_bar[stage]));
          else ptx::tc_commit_pair(ptx::smem_u32(&empty_bar[stage]), 3);
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (NC == 1) ptx::tc_commit(ptx::smem_u32(&tfull_bar[buf]));
        else ptx::tc_commit_pair(ptx::smem_u32(&tfull_bar[buf]), 3);  // accumulator halves ready in both CTAs
      }
    }
  } else {
    // epilogue: thread = row of the tile (TMEM lane); the 4 warps of a column half share one staging box
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row_in_tile = 32 * quarter + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * quarter) << 16);
    const bool leader = (warp == 2 + 4 * half) && lane == 0;  // issues this group's TMA traffic
    constexpr bool with_res = EPI == EPI_BIAS_RESIDUAL;
    // two staging boxes per column half: while TMA drains box j (its reads queue behind the main loop's loads in
    // the TMA unit -- ncu r01c showed the group waiting ~4 k cycles per box on a single buffer) box j+1 fills
    unsigned char* box0 = stage_c + (size_t)half * 2 * kBoxBytes;
    const uint32_t box0_u32 = ptx::smem_u32(box0);
    // this thread's row inside a box: 128 bytes, 16-byte chunk c lives at chunk (c ^ (row & 7))
    const int row_off = row_in_tile * 128;
    const int sw = row_in_tile & 7;
    const uint32_t rbar0 = ptx::smem_u32(&res_bar[2 * half]);
    uint32_t res_phase = 0;  // bit b = parity of this group's residual barrier b
    float* bias_t = bias_s + half * 2 * (BN / 2);  // this group's [bias | vec2], one tile at a time
    float* vec2_t = bias_t + BN / 2;
    constexpr bool ln_in = LNIN;  // A rows are un-normalised: scale/shift per row here
    constexpr bool want_stats = STATS;
    const bool have_stats = (LNIN || with_res) && p.stats_in != nullptr;  // a plain residual carries none
    if (with_res && leader && unit < tiles) {
      const int m0 = (unit / n_tiles) * (BM * NC) + (int)rank * BM, n0 = (unit % n_tiles) * BN;
      ptx::mbar_expect_tx(rbar0, kBoxBytes);
      ptx::tma_load_2d(box0_u32, &tmap_res, rbar0, n0 + half * (BN / 2), m0);
    }
    int it = 0;
    int jb = 0;  // boxes this group has produced so far; buffer = jb & 1
    // Per-tile operands of this thread, requested one tile ahead so their L2 latency hides behind the previous
    // tile's epilogue (r01d: six dependent statistics loads per tile in front of the accumulator wait were 12 % of
    // the FFN-up GEMM's stall samples): the bias / second-vector element this thread publishes through shared
    // memory and the LayerNorm partials of its row.
    float nx_bias = 0.0f, nx_vec2 = 1.0f;
    float2 nx_stat[SLOTS];
    auto request = [&](int t) {
      const int tm0 = (t / n_tiles) * (BM * NC) + (int)rank * BM, tn0 = (t % n_tiles) * BN;
      nx_bias = p.bias[tn0 + half * (BN / 2) + row_in_tile];
      if ((LNIN || with_res) && p.vec2) nx_vec2 = p.vec2[tn0 + half * (BN / 2) + row_in_tile];
      if (have_stats) {
#pragma unroll
        for (int j = 0; j < SLOTS; ++j) nx_stat[j] = p.stats_in[(size_t)j * p.stats_stride + tm0 + row_in_tile];
      }
    };
    if (unit < tiles) request(unit);
    for (int tile = unit; tile < tiles; tile += units, ++it) {
      const int buf = it & 1;
      const int m0 = (tile / n_tiles) * (BM * NC) + (int)rank * BM, n0 = (tile % n_tiles) * BN;
      const float bv = nx_bias, v2 = nx_vec2;
      // LayerNorm statistics of this thread's row (of A, or of the residual): rs = 1/sigma, nmr = -mu/sigma
      float rs = 1.0f, nmr = 0.0f;
      if (have_stats) {
        float s = 0.0f, ss = 0.0f;
#pragma unroll
        for (int j = 0; j < SLOTS; ++j) {
          s += nx_stat[j].x;
          ss += nx_stat[j].y;
        }
        const float mu = s * p.inv_h;
        rs = rsqrtf(fmaxf(fmaf(-mu, mu, ss * p.inv_h), 0.0f) + p.eps);
        nmr = -mu * rs;
      }
      float row_s = 0.0f, row_ss = 0.0f;  // partial statistics of this row's 128 output columns
      ptx::mbar_wait(ptx::smem_u32(&tfull_bar[buf]), (it >> 1) & 1);
      ptx::tc_fence_after();
      // every thread of the group left the previous tile's last box through a group_sync, so the vectors are free;
      // the group_sync below publishes them
      bias_t[row_in_tile] = bv;
      vec2_t[row_in_tile] = v2;
      if (tile + units < tiles) request(tile + units);
#pragma unroll 1
      for (int bx = 0; bx < kBoxesPerHalf; ++bx, ++jb) {
        const int col0 = half * (BN / 2) + bx * kBoxCols;  // first column of this box within the tile
        const int sb = jb & 1;
        unsigned char* my_row = box0 + sb * kBoxBytes + row_off;
        // buffer sb is free: the leader arrives here only after the store of box jb-2 has been read out
        group_sync(half);
        if (with_res) {
          ptx::mbar_wait(rbar0 + 8 * sb, (res_phase >> sb) & 1);
          res_phase ^= 1u << sb;
        }
#pragma unroll
        for (int c32 = 0; c32 < kBoxCols / 32; ++c32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)(buf * BN + col0 + c32 * 32), r);
          ptx::tmem_ld_wait();
          if (bx == kBoxesPerHalf - 1 && c32 == kBoxCols / 32 - 1) {
            // last read of this accumulator buffer by this warp: hand it back to the MMA warp
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (NC == 1) ptx::mbar_arrive(ptx::smem_u32(&tempty_bar[buf]));
              else ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tempty_bar[buf]), 0));  // the leader's barrier
            }
          }
          const float4* bias4 = reinterpret_cast<const float4*>(bias_t + bx * kBoxCols + c32 * 32);
          const float4* vec4 = reinterpret_cast<const float4*>(vec2_t + bx * kBoxCols + c32 * 32);
#pragma unroll
          for (int v = 0; v < 4; ++v) {  // 8 columns per 16-byte chunk
            float x[8], g[8];
            {
              const float4 b0 = bias4[2 * v], b1 = bias4[2 * v + 1];
              x[0] = b0.x, x[1] = b0.y, x[2] = b0.z, x[3] = b0.w;
              x[4] = b1.x, x[5] = b1.y, x[6] = b1.z, x[7] = b1.w;
            }
            if (ln_in || with_res) {
              const float4 g0 = vec4[2 * v], g1 = vec4[2 * v + 1];
              g[0] = g0.x, g[1] = g0.y, g[2] = g0.z, g[3] = g0.w;
              g[4] = g1.x, g[5] = g1.y, g[6] = g1.z, g[7] = g1.w;
            }
            if (ln_in) {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] = fmaf(__uint_as_float(r[8 * v + e]), rs, fmaf(nmr, g[e], x[e]));
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] += __uint_as_float(r[8 * v + e]);
            }
            uint4* slot = reinterpret_cast<uint4*>(my_row + (((c32 * 4 + v) ^ sw) << 4));
            if (EPI == EPI_BIAS_GELU) {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[e] = gelu_erf(x[e]);
            } else if (with_res) {
              // residual = LayerNorm of the loaded stream when statistics came along (rs, nmr, gamma; beta sits in the
              // bias), the stream itself otherwise (rs = 1, nmr = 0, gamma = 1)
              const uint4 rr = *slot;
              x[0] = fmaf(fmaf(bf16lo_to_f32(rr.x), rs, nmr), g[0], x[0]);
              x[1] = fmaf(fmaf(bf16hi_to_f32(rr.x), rs, nmr), g[1], x[1]);
              x[2] = fmaf(fmaf(bf16lo_to_f32(rr.y), rs, nmr), g[2], x[2]);
              x[3] = fmaf(fmaf(bf16hi_to_f32(rr.y), rs, nmr), g[3], x[3]);
              x[4] = fmaf(fmaf(bf16lo_to_f32(rr.z), rs, nmr), g[4], x[4]);
              x[5] = fmaf(fmaf(bf16hi_to_f32(rr.z), rs, nmr), g[5], x[5]);
              x[6] = fmaf(fmaf(bf16lo_to_f32(rr.w), rs, nmr), g[6], x[6]);
              x[7] = fmaf(fmaf(bf16hi_to_f32(rr.w), rs, nmr), g[7], x[7]);
            }
            if (want_stats) {
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                row_s += x[e];
                row_ss = fmaf(x[e], x[e], row_ss);
              }
            }
            uint4 o;
            o.x = pack_bf16(x[0], x[1]);
            o.y = pack_bf16(x[2], x[3]);
            o.z = pack_bf16(x[4], x[5]);
            o.w = pack_bf16(x[6], x[7]);
            *slot = o;
          }
        }
        // generic-proxy writes -> visible to the async proxy, then one thread hands the box to TMA
        ptx::fence_proxy_async_smem();
        group_sync(half);
        if (leader) {
          ptx::tma_store_2d(&tmap_out, box0_u32 + sb * kBoxBytes, n0 + col0, m0);
          ptx::tma_store_commit();
          ptx::tma_store_wait_read<1>();  // the store of box jb-1 has drained: the other buffer is free
          if (with_res) {
            // prefetch the residual of the next box (same tile, or the first box of this CTA's next tile)
            int nm0 = m0, nc = n0 + col0 + kBoxCols;
            bool more = true;
            if (bx == kBoxesPerHalf - 1) {
              const int nt = tile + units;
              more = nt < tiles;
              nm0 = (nt / n_tiles) * (BM * NC) + (int)rank * BM;
              nc = (nt % n_tiles) * BN + half * (BN / 2);
            }
            if (more) {
              const uint32_t nb = (uint32_t)(sb ^ 1);
              ptx::mbar_expect_tx(rbar0 + 8 * nb, kBoxBytes);
              ptx::tma_load_2d(box0_u32 + nb * kBoxBytes, &tmap_res, rbar0 + 8 * nb, nc, nm0);
            }
          }
        }
      }
      if (want_stats && p.stats_out)
        p.stats_out[(size_t)((n0 >> 7) + half) * p.stats_stride + m0 + row_in_tile] = make_float2(row_s, row_ss);
    }
    if (leader) ptx::tma_store_wait_all();  // global writes complete before the kernel ends
  }

  ptx::tc_fence_before();
  // pair: neither CTA may leave (or free its TMEM) while the other can still signal its barriers
  if (NC == 2) ptx::cluster_sync(); else __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if (NC == 2) ptx::tmem_dealloc_pair(tmem_base, kTmemCols);
    else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

int gemm_tile_n() { return BN; }

// CTA pairs; profiling builds can select the single-CTA kernel with ICD_GEMM_PAIR=0 (A/B timing)
static int pair_mode() {
#ifdef ICD_PROFILING
  static const int mode = [] {
    const char* v = getenv("ICD_GEMM_PAIR");
    return (v && *v) ? (atoi(v) != 0 ? 2 : 1) : 2;
  }();
  return mode;
#else
  return 2;
#endif
}

template <int NC, int EPI, bool LNIN, bool STATS, int SLOTS>
static int launch_variant(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout, const CUtensorMap& tres,
                          const GemmParams& p, cudaStream_t st) {
  constexpr int kSmemBytes = smem_bytes<NC>();
  auto kernel = gemm_tc_kernel<NC, EPI, LNIN, STATS, SLOTS>;
  ICD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int tiles = ((p.M + BM * NC - 1) / (BM * NC)) * (p.N / BN);
  int units = kSMs / NC;
  if (NC == 2) {
    // persistent kernel: as many pairs as the device can keep resident at once (a TPC with one SM fused off
    // cannot host a pair)
    static int resident = 0;
    if (resident == 0) {
      cudaLaunchConfig_t cfg{};
      cfg.blockDim = dim3(kThreads);
      cfg.dynamicSmemBytes = kSmemBytes;
      cfg.gridDim = dim3(kSMs);
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      int n = 0;
      ICD_CUDA(cudaOccupancyMaxActiveClusters(&n, kernel, &cfg));
      resident = std::max(1, n);
    }
    units = std::min(units, resident);
  }
  ICD_CUDA(launch_chained(kernel, dim3(std::min(tiles, units) * NC), dim3(kThreads), (size_t)kSmemBytes, st, NC, ta, tb, tout, tres, p));
  count_launch();
  return ICD_OK;
}

// SLOTS only matters where statistics come in (LNIN, or a residual carrying them): the plain-A variants are built once
template <int NC, int SLOTS>
static int launch_nc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout, const CUtensorMap& tres,
                     const GemmParams& p, cudaStream_t st) {
  const bool lnin = p.stats_in != nullptr && p.epi != EPI_BIAS_RESIDUAL;
  const bool stats = p.stats_out != nullptr;
  switch (p.epi) {
    case EPI_BIAS:
      return lnin ? launch_variant<NC, EPI_BIAS, true, false, SLOTS>(ta, tb, tout, tres, p, st)
                  : launch_variant<NC, EPI_BIAS, false, false, 6>(ta, tb, tout, tres, p, st);
    case EPI_BIAS_GELU:
      return lnin ? launch_variant<NC, EPI_BIAS_GELU, true, false, SLOTS>(ta, tb, tout, tres, p, st)
                  : launch_variant<NC, EPI_BIAS_GELU, false, false, 6>(ta, tb, tout, tres, p, st);
    case EPI_BIAS_RESIDUAL:
      if (!p.stats_in)  // a plain residual: no statistics to add up
        return stats ? launch_variant<NC, EPI_BIAS_RESIDUAL, false, true, 6>(ta, tb, tout, tres, p, st)
                     : launch_variant<NC, EPI_BIAS_RESIDUAL, false, false, 6>(ta, tb, tout, tres, p, st);
      return stats ? launch_variant<NC, EPI_BIAS_RESIDUAL, false, true, SLOTS>(ta, tb, tout, tres, p, st)
                   : launch_variant<NC, EPI_BIAS_RESIDUAL, false, false, SLOTS>(ta, tb, tout, tres, p, st);
  }
  set_error("gemm_tc: unknown epilogue %d", p.epi);
  return ICD_E_ARG;
}

int launch_gemm_tc(const GemmArgs& a, cudaStream_t st) {
  if (a.N % BN != 0 || a.K % BK != 0 || a.M <= 0) {
    set_error("gemm_tc: needs N %% %d == 0 and K %% %d == 0 (M=%d N=%d K=%d)", BN, BK, a.M, a.N, a.K);
    return ICD_E_ARG;
  }
  if ((a.stats_in || a.stats_out) &&
      (a.stats_stride < ((a.M + 2 * BM - 1) / (2 * BM)) * 2 * BM ||
       (a.stats_in && ((a.stats_cols != 768 && a.stats_cols != 1024) || !a.vec2)))) {
    set_error("gemm_tc: LayerNorm statistics need a row stride covering whole tiles, the column vector, and a row length of "
              "768 or 1024");
    return ICD_E_ARG;
  }
  if (!a.tmap_out || (a.epi == EPI_BIAS_RESIDUAL && !a.tmap_res)) {
    set_error("gemm_tc: missing output / residual tensor map");
    return ICD_E_ARG;
  }
  CUtensorMap ta, tb, tout, tres;
  memcpy(&ta, a.tmap_a, sizeof(ta));
  memcpy(&tb, a.tmap_b, sizeof(tb));
  memcpy(&tout, a.tmap_out, sizeof(tout));
  memcpy(&tres, a.tmap_res ? a.tmap_res : a.tmap_out, sizeof(tres));
  GemmParams p{};
  p.bias = a.bias;
  p.vec2 = a.vec2;
  p.stats_in = reinterpret_cast<const float2*>(a.stats_in);
  p.stats_out = reinterpret_cast<float2*>(a.stats_out);
  p.stats_stride = a.stats_stride;
  p.inv_h = a.stats_cols > 0 ? 1.0f / (float)a.stats_cols : 0.0f;
  p.eps = a.eps;
  p.M = a.M;
  p.N = a.N;
  p.K = a.K;
  p.epi = a.epi;
#ifdef ICD_PROFILING
  if (pair_mode() != 2)  // single-CTA tiles: A/B timing only
    return a.stats_cols == 1024 ? launch_nc<1, 8>(ta, tb, tout, tres, p, st) : launch_nc<1, 6>(ta, tb, tout, tres, p, st);
#endif
  return a.stats_cols == 1024 ? launch_nc<2, 8>(ta, tb, tout, tres, p, st) : launch_nc<2, 6>(ta, tb, tout, tres, p, st);
}

int gemm_make_map_a(void* map128, const void* base, int64_t rows, int K) {
  return make_tmap_bf16_2d(map128, base, (uint64_t)rows, (uint64_t)K, BM, BK, true);
}
// output / residual boxes have the shape of an A box (128 rows x 64 columns, SWIZZLE_128B), so a buffer that is
// also read as the next GEMM's A operand needs only one map
int gemm_make_map_out(void* map128, const void* base, int64_t rows, int N) {
  return make_tmap_bf16_2d(map128, base, (uint64_t)rows, (uint64_t)N, BM, kBoxCols, true);
}
// W box: the rows of the tile one CTA loads (all 256, or its half of the pair's tile)
int gemm_make_map_b(void* map128, const void* base, int64_t rows, int K) {
  return make_tmap_bf16_2d(map128, base, (uint64_t)rows, (uint64_t)K, BN / pair_mode(), BK, true);
}

}  // namespace icd
