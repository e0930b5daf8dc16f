// scan_tc.cu -- tensor-core exact inner-product scan with fused per-query top-k (sm_100a).
//
// Replaces the brute-force FLAT/IP search inside MilvusClient.search (reference call site
// services/milvus_service.py:280-285) for batched queries.  scores = Q[B,dim] * C[N,dim]^T is
// never materialised:
//
//   * a CTA owns one tile of 128 queries for its whole life.  The tile lives in TENSOR MEMORY
//     as the MMA A operand (128 lanes x dim/2 columns of packed bf16, <= 384 columns), so
//     shared memory is free for streaming the table.
//   * table rows stream HBM -> shared memory through TMA in a ring of mbarrier-tracked stages
//     and are the MMA B operand (K-major).  The table is described to TMA as a 3-D tensor
//     {64 elements, rows, K blocks} so ONE bulk copy brings a whole stage -- 128 (pairs: 64) rows x (kbs x 64)
//     bf16, laid out as kbs consecutive row-tile x 64 tiles in the 128-byte-swizzle canonical layout.  kbs is
//     chosen per launch (up to 6 = 768-byte bursts per row for pairs, 3 for single CTAs: launch_tensor_scan_bn).
//   * tcgen05.mma (M=128 queries, N=128 rows, K=16) accumulates a 128x128 fp32 tile in TMEM.
//     N must be >= 128: with A in TMEM every MMA re-reads the 128x16 A slice (4 KiB) at the
//     TMEM read rate, ~64 cycles, so N=64 (32 cycles of math) runs the pipe at half rate
//     (measured: 38 % tensor-active with N=64).  The accumulators take the columns Q leaves
//     free.  For dim = 768 the tile fills 384 columns and leaves room for ONE 128-column buffer: the MMAs
//     of tile i+1 wait until the epilogue has drained tile i (64 KiB through the same 64 B/clk TMEM read
//     path the A operand uses, ~1 k cycles per 3 k-cycle tile: r01b measured 70 % tensor-active at
//     B = 1024).  In the tensor-bound regime (>= 2 query tiles per row stream) the last third of K
//     therefore lives in SHARED memory instead (64 KiB, canonical K-major 128-byte-swizzle tiles, SS
//     MMAs for those K blocks): Q then takes 256 TMEM columns, two accumulator buffers fit, and the
//     drain of tile i overlaps the MMAs of tile i+1.  The HBM-bound regime keeps the whole tile in
//     TMEM and all of shared memory for the row stream.
//   * epilogue: thread == TMEM lane == query.  It reads its 64 scores with tcgen05.ld,
//     compares against its private k-th best (a register) and only on the rare hit inserts
//     into its private sorted list in shared memory.  Level weights (ICD_WEIGHT_PRE) are
//     applied here.
//   * cross-CTA pruning: every CTA publishes its k-th best score per query to a global bound
//     (atomicMax on an order-preserving integer key) and admits a row only if it also reaches
//     the bound the other row groups have proven; without it each of the 148 row groups warms
//     its own lists and the insert path, not HBM, bounds the kernel (ncu, B=128: 42 % of
//     epilogue samples in the insert loop, 57 % DRAM utilisation).
//   * CTA pairs (NC = 2, launches with an even number of query tiles): two CTAs of one TPC hold
//     neighbouring query tiles and run ONE tcgen05.mma.cta_group::2 (M = 256 queries, N = 128 rows) per K
//     step, issued by the pair's leader.  Each CTA loads only HALF of every row tile (64 rows) and the tensor
//     cores read both halves, so the shared-memory port carries half the fill and half the B reads per SM
//     (with TMA fill 64 B/clk + B reads 64 B/clk + the shared-memory third of Q the single-CTA form asks
//     117 % of the 128 B/clk port) and the L2 -> SM traffic of the row stream halves as well.  Measured
//     (r01d, 10 M rows): B = 256 0.707 -> 0.750 of sustained bf16 peak, B = 1024 and 4096 unchanged within
//     noise (0.83 / 0.79: those run into the 1 kW power cap at ~1.66 GHz, not into a port).
//     ICD_SCAN_QTMEM=6 keeps half of K in shared memory instead of a third: no better.
//   * grid = G row groups x T query tiles; each CTA writes one sorted list per query to the
//     partial buffer [B, G, k] that topk_merge.cu reduces.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM lane quarter = warp % 4).
//
// Roofline: HBM for B <~ 200 (one pass over the table per launch), bf16 tensor pipe above.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace icd {
namespace {

constexpr int BM = 128;  // queries per CTA
constexpr int BK = 64;   // bf16 per TMA box row (128 bytes)
constexpr int kMaxStages = 12;
constexpr int kThreads = 192;
constexpr int kTmemCols = 512;
constexpr int kSmemLimit = 227 * 1024;
constexpr int kPreSlots = 32;  // running maxima per (query, row group) in the pre-pass
constexpr int kPreFolds = 4;   // row groups fold into this many classes (g mod 4): 128 disjoint row sets per query, so the
                               // slot-maxima bound serves every kc <= 128 (topk_merge.cu, bound_from_slots_kernel)

struct ScanParams {
  const uint8_t* levels;
  const __nv_bfloat16* q;  // [B, dim]
  float* part_score;       // [B, G, kc]
  int* part_id;
  int* gbound;             // [B] order-preserving keys of the proven per-query k-th-best bound, or null
  int64_t n_rows;
  int dim, nkb;  // nkb = dim / 64
  int B, kc, weight_pre;
  int G, T;      // row groups, query tiles in this launch
  int qt0;       // first query tile of this launch
  int nst;       // pipeline stages
  int kbs;       // K blocks (128 x 64 tiles) per stage; divides nkb
  int nacc;      // accumulator buffers (1 or 2) in the TMEM columns behind the query tile
  int acc_col0;  // first accumulator column (== dim / 2 rounded up to 128)
  int nkb_tmem;  // K blocks of the query tile held in TMEM; the remaining nkb - nkb_tmem live in shared memory
  int tstride;   // scan every tstride-th row tile only (1 = all rows; > 1 = the sampling pre-pass)
  int* progress; // [G * T] tiles issued by each CTA's producer (drift limiter), or null
  int drift;     // a producer may run at most this many tiles ahead of the slowest CTA of its row group
  const uint32_t* mask;  // row bitmap (bit i & 31 of word i >> 5 = row i may be returned), or null = every row
#ifdef ICD_PROFILING
  int tiled;     // timing experiment: read the table AS IF it were stored tile-major [tile][K block][128 rows][64]
                 // (8 KiB contiguous runs per K block instead of 768-byte row segments); results are meaningless
#endif
};

// Private candidate list of one query (thread): kc entries sorted by (score desc, id asc) in
// shared memory, entry j of this thread at [j * BM].  Rows arrive in ascending id order, so a
// strict '>' admission test plus "insert after equal scores" keeps the id tie-break exact.
// (An unsorted list with worst-slot tracking was measured slower: 60 % vs 71 % of HBM at B=128.)
// Admitted scores wait in a small per-thread FIFO (local memory: dynamically indexed, L1-resident) and reach the sorted
// list here, all lanes of the warp together.  Every queued score is tested again against the list's current k-th best.
// `cnt` = entries filled so far: the walk starts at the first free entry instead of at the end of the list, so a list that
// a tight pre-pass bound keeps nearly empty pays a handful of steps per insert, not kc.
// Returns (k-th best, filled entries).  One call site per accumulator tile plus the rare "queue nearly full" sites, so
// the unrolled 128-column epilogue stays small (inlined per column, the insert path made the kernel 12.8 k instructions
// and twice as slow as the instruction cache missed: r02u).
constexpr int kQueue = 8;
__device__ __noinline__ uint2 drain_queue(float* ls, int* li, int kc, int cnt, float thr, const float* qs, const int* qi, int qn) {
  for (int e = 0; e < qn; ++e) {
    const float s = qs[e];
    if (s > thr) {
      const int id = qi[e];
      int j = cnt < kc ? cnt : kc - 1;  // first free entry, or the last one of a full list (s > ls[(kc-1)*BM] then)
      cnt = cnt < kc ? cnt + 1 : kc;
      while (j > 0 && ls[(j - 1) * BM] < s) {
        ls[j * BM] = ls[(j - 1) * BM];
        li[j * BM] = li[(j - 1) * BM];
        --j;
      }
      ls[j * BM] = s;
      li[j * BM] = id;
      thr = ls[(kc - 1) * BM];
    }
  }
  return make_uint2(__float_as_uint(thr), (uint32_t)cnt);
}

// The four mask words of the 128-row tile starting at row0 (a multiple of 128); words past the end of the mask
// (ceil(n_rows / 32) words) read as 0.  Unmasked instantiations see compile-time all-ones words, so every mask test
// folds away and they are the unfiltered kernel.
template <bool MASKED>
__device__ __forceinline__ uint4 tile_mask(const uint32_t* mask, int64_t row0, int64_t n_rows) {
  if constexpr (!MASKED) return make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
  const uint32_t* w = mask + (row0 >> 5);
  return make_uint4(row0 < n_rows ? __ldg(w) : 0u, row0 + 32 < n_rows ? __ldg(w + 1) : 0u,
                    row0 + 64 < n_rows ? __ldg(w + 2) : 0u, row0 + 96 < n_rows ? __ldg(w + 3) : 0u);
}
__device__ __forceinline__ uint32_t mask_word(const uint4& m, int i) { return i == 0 ? m.x : i == 1 ? m.y : i == 2 ? m.z : m.w; }

// BN = table rows per accumulator tile (MMA N); NC = CTAs per MMA (2 = CTA pair, cta_group::2).
// KBS / NKBT > 0: the stage shape (K blocks per stage) and the TMEM / shared-memory split of the query tile are
// compile-time constants for dim = 768, so the MMA issue loop unrolls into ~4 instructions per tcgen05.mma.  The generic
// loop (KBS = 0: run-time kbs / nkb_tmem, 64-bit descriptor arithmetic, TS-or-SS branch per MMA) costs 16.6 instructions
// = ~73 issue cycles per 64-cycle MMA (ncu r02a, B = 256: the elected thread was busy issuing 73 % of the time, waiting
// for data 3 % and for the epilogue 14 %): the tensor pipe was bounded by instruction issue, not by operands.
//
// MASKED = a row mask (p.mask) restricts the rows that may be returned (filtered search).  A template parameter: as a
// run-time branch it cost the epilogue-bound small table (40 474 rows, B = 1024) 9 % with no mask (r03, filter_ab.py).
// PRE = the sampling pre-pass.  Its only product is a per-query lower bound of the kc-th best score, so it keeps no
// candidate lists: the epilogue folds every sampled score into kPreSlots running maxima (slot = accumulator column mod 32;
// slots partition the sampled rows, so the kc-th largest slot maximum is reached by at least kc distinct rows) with
// straight-line FMNMX code.  r02h (ncu, 12.5 M rows): the list-based pre-pass spent 0.72 / 0.40 / 0.28 ms at B = 1024 / 256 /
// 128 -- 5-9 % of the scan it precedes -- almost entirely in the divergent sorted-list inserts of its warm-up (each insert
// call ~450 cycles for the whole warp, ~2 700 calls per warp); the sampled rows themselves stream in ~0.03 ms.
template <int BN, int NC, int KBS, int NKBT, bool PRE, bool MASKED>
__global__ void __launch_bounds__(kThreads, 1)
scan_tc_kernel(const __grid_constant__ CUtensorMap tmap, const ScanParams p) {
  constexpr int kBoxBytes = (BN / NC) * BK * 2;  // this CTA's share of one BN x 64 bf16 tile
  const uint32_t rank = NC == 2 ? ptx::cluster_ctarank() : 0u;  // 0 = the pair's leader (issues the MMAs)
  extern __shared__ __align__(1024) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x / p.T;
  const int qt = p.qt0 + blockIdx.x % p.T;

  // shared memory carve-up
  const int stage_bytes = p.kbs * kBoxBytes;
  unsigned char* stage_base = smem;                                           // nst stages, 1024-aligned
  unsigned char* q_tail = smem + (size_t)p.nst * stage_bytes;  // (nkb - nkb_tmem) tiles of 128 queries x 64 bf16, 1024-aligned
  constexpr int kQTileBytes = BM * BK * 2;                      // 16 KiB
  float* list_s = reinterpret_cast<float*>(q_tail + (size_t)(p.nkb - p.nkb_tmem) * kQTileBytes);  // [kc][BM]
  int* list_i = reinterpret_cast<int*>(list_s + (size_t)p.kc * BM);           // [kc][BM]
  uint64_t* bars = reinterpret_cast<uint64_t*>(list_i + (size_t)p.kc * BM);
  uint64_t* full_bar = bars;                    // [nst]
  uint64_t* empty_bar = bars + kMaxStages;      // [nst]
  uint64_t* tfull_bar = bars + 2 * kMaxStages;  // [2]
  uint64_t* tempty_bar = tfull_bar + 2;         // [2]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  // row tiles of this group
  const int64_t total_tiles = ((p.n_rows + BN - 1) / BN + p.tstride - 1) / p.tstride;
  const int64_t t0 = total_tiles * g / p.G;
  const int64_t t1 = total_tiles * (g + 1) / p.G;

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tmap(&tmap);
    for (int s = 0; s < p.nst; ++s) {
      ptx::mbar_init(ptx::smem_u32(&full_bar[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(ptx::smem_u32(&tfull_bar[b]), 1);
      ptx::mbar_init(ptx::smem_u32(&tempty_bar[b]), 4 * NC);  // one arrival per epilogue warp of every CTA of the MMA
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
  if (NC == 2) ptx::cluster_sync(); else __syncthreads();  // barriers of both CTAs are initialised from here on
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // epilogue threads: lane quarter and query of this thread
  const int ep_lane = 32 * (warp & 3) + lane;  // TMEM lane == query within the tile
  const int query = qt * BM + ep_lane;
  float* my_s = list_s + ep_lane;
  int* my_i = list_i + ep_lane;

  if (warp >= 2) {
    // private list init
    if (!PRE) {
      for (int j = 0; j < p.kc; ++j) {
        my_s[j * BM] = -INFINITY;
        my_i[j * BM] = -1;
      }
    }
    // query tile -> TMEM: lane = query, 32-bit column c holds elements (2c, 2c+1); K blocks >= nkb_tmem go to
    // shared memory as K-major tiles in the 128-byte-swizzle canonical layout (row = query, 16-byte chunk c of the
    // row at chunk c ^ (row & 7)), the layout the SS MMA descriptor expects
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * (warp & 3)) << 16);
    const uint4* qrow = reinterpret_cast<const uint4*>(p.q + (size_t)query * p.dim);
    // two K blocks (2 x 64 bf16 = 16 x uint4 of this query's row) per step, the loads of a step issued before its
    // stores: a step's L2 / HBM latency is paid once, not per 16 columns (r02t: ~10 us of every launch went here)
    auto put = [&](int kb, const uint32_t* r) {
      if (kb < p.nkb_tmem) {
        ptx::tmem_st_32x32b_x16(lane_addr + (uint32_t)(kb * 32), r);
        ptx::tmem_st_32x32b_x16(lane_addr + (uint32_t)(kb * 32 + 16), r + 16);
      } else {
        unsigned char* row = q_tail + (size_t)(kb - p.nkb_tmem) * kQTileBytes + ep_lane * 128;
#pragma unroll
        for (int chunk = 0; chunk < 8; ++chunk)
          *reinterpret_cast<uint4*>(row + ((chunk ^ (ep_lane & 7)) << 4)) =
              make_uint4(r[4 * chunk], r[4 * chunk + 1], r[4 * chunk + 2], r[4 * chunk + 3]);
      }
    };
    for (int kb = 0; kb < p.nkb; kb += 2) {
      uint32_t r[64];
      const bool two = kb + 1 < p.nkb;
#pragma unroll
      for (int v = 0; v < 16; ++v) {
        uint4 t = make_uint4(0u, 0u, 0u, 0u);
        if (query < p.B && (v < 8 || two)) t = qrow[kb * 8 + v];
        r[4 * v + 0] = t.x;
        r[4 * v + 1] = t.y;
        r[4 * v + 2] = t.z;
        r[4 * v + 3] = t.w;
      }
      put(kb, r);
      if (two) put(kb + 1, r + 32);
    }
    ptx::tmem_st_wait();
    ptx::fence_proxy_async_smem();  // the tail tiles are read by the tensor core (async proxy)
  }
  ptx::tc_fence_before();
  if (NC == 2) ptx::cluster_sync(); else __syncthreads();  // the leader's MMAs read BOTH CTAs' query tiles
  ptx::tc_fence_after();

  if (warp == 0) {
    // ===================== TMA producer =====================
    // Drift limiter: the T CTAs of a row group stream the same rows; left alone they drift apart
    // by more than the L2 holds and every one of them re-reads the rows from HBM (ncu, B=1024:
    // 3.0x the algorithmic DRAM bytes).  Each producer publishes the tile it is about to issue
    // and does not run more than `drift` tiles ahead of the slowest CTA of its group, so one
    // HBM read serves the whole group out of L2.  (All CTAs are co-resident: grid <= 148, 1/SM.)
    int* prog = p.progress ? p.progress + (size_t)g * p.T : nullptr;
    const int me = blockIdx.x % p.T;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int64_t t = t0; t < t1; ++t, ++it) {
      if (prog && (it & 1) == 0) {
        if (lane == 0) asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(prog + me), "r"(it) : "memory");
        for (uint32_t spins = 0; spins < (1u << 16); ++spins) {
          int v = 0x7fffffff;
          for (int l = lane; l < p.T; l += 32) {
            int w;
            asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(w) : "l"(prog + l) : "memory");
            v = min(v, w);
          }
          v = __reduce_min_sync(0xffffffffu, v);
          if (v + p.drift >= it) break;
          __nanosleep(256);
        }
      }
      if (lane == 0) {
        const int row = (int)(t * p.tstride * BN) + (int)rank * (BN / NC);  // this CTA's rows of the tile
        for (int kb = 0; kb < p.nkb; kb += p.kbs) {
          ptx::mbar_wait(ptx::smem_u32(&empty_bar[stage]), phase ^ 1);
          if (NC == 1) {
            const uint32_t fb = ptx::smem_u32(&full_bar[stage]);
            ptx::mbar_expect_tx(fb, (uint32_t)stage_bytes);
#ifdef ICD_PROFILING
            if (p.tiled) ptx::tma_load_4d(ptx::smem_u32(stage_base + (size_t)stage * stage_bytes), &tmap, fb, 0, row % BN, kb, row / BN);
            else
#endif
            ptx::tma_load_3d(ptx::smem_u32(stage_base + (size_t)stage * stage_bytes), &tmap, fb, 0, row, kb);
          } else {
            // both CTAs' bytes are counted on the LEADER's barrier (only its MMA thread waits for the stage)
            if (rank == 0) ptx::mbar_expect_tx(ptx::smem_u32(&full_bar[stage]), 2u * (uint32_t)stage_bytes);
            const uint32_t fb = ptx::mapa(ptx::smem_u32(&full_bar[stage]), 0);
#ifdef ICD_PROFILING
            if (p.tiled) ptx::tma_load_4d_pair(ptx::smem_u32(stage_base + (size_t)stage * stage_bytes), &tmap, fb, 0, row % BN, kb, row / BN);
            else
#endif
            ptx::tma_load_3d_pair(ptx::smem_u32(stage_base + (size_t)stage * stage_bytes), &tmap, fb, 0, row, kb);
          }

          if (++stage == p.nst) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      __syncwarp();
    }
    if (prog && lane == 0) asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(prog + me), "r"(0x7fffffff) : "memory");
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (KBS > 0 && rank == 0 && ptx::elect_one()) {
      // ---- specialised issue loop (dim = 768: 12 K blocks, KBS per stage, the first NKBT of the query tile in TMEM)
      constexpr uint32_t idesc = ptx::make_idesc_bf16(BM * NC, BN);
      constexpr int kNKB = 12;
      constexpr int kKBS = KBS > 0 ? KBS : 1;
      constexpr uint32_t kStageStep = (uint32_t)(kKBS * kBoxBytes) >> 4;  // descriptor units (16 bytes) per stage
      const uint32_t stage_lo0 = ptx::desc_lo_k128(ptx::smem_u32(stage_base));
      const uint32_t qtail_lo = ptx::desc_lo_k128(ptx::smem_u32(q_tail));
      const uint32_t full0 = ptx::smem_u32(&full_bar[0]), empty0 = ptx::smem_u32(&empty_bar[0]);
      const uint32_t nst = (uint32_t)p.nst;
      const bool two_acc = p.nacc == 2;
      uint32_t stage = 0, phase = 0;
      int it = 0;
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const int buf = two_acc ? (it & 1) : 0;
        const uint32_t use = two_acc ? (uint32_t)(it >> 1) : (uint32_t)it;
        ptx::mbar_wait(ptx::smem_u32(&tempty_bar[buf]), (use & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(p.acc_col0 + buf * BN);
#pragma unroll
        for (int s = 0; s < kNKB / kKBS; ++s) {
          ptx::mbar_wait(full0 + stage * 8, phase);
          ptx::tc_fence_after();
          const uint32_t b_lo = stage_lo0 + stage * kStageStep;
#pragma unroll
          for (int j = 0; j < kKBS; ++j) {
#pragma unroll
            for (int k4 = 0; k4 < BK / 16; ++k4) {
              const int kb = s * kKBS + j;                                     // compile-time after unrolling
              const uint32_t boff = (uint32_t)(j * (kBoxBytes >> 4) + k4 * 2);  // +2 per 32 bytes of K, +tile per K block
              if (kb < NKBT) {
                const uint32_t a_tmem = tmem_base + (uint32_t)((kb * (BK / 16) + k4) * 8);
                if (s == 0 && j == 0 && k4 == 0) ptx::mma_ts_lo<NC, 0>(d_tmem, a_tmem, b_lo + boff, idesc);
                else ptx::mma_ts_lo<NC, 1>(d_tmem, a_tmem, b_lo + boff, idesc);
              } else {
                const uint32_t a_lo = qtail_lo + (uint32_t)((kb - NKBT) * (kQTileBytes >> 4) + k4 * 2);
                if (s == 0 && j == 0 && k4 == 0) ptx::mma_ss_lo<NC, 0>(d_tmem, a_lo, b_lo + boff, idesc);
                else ptx::mma_ss_lo<NC, 1>(d_tmem, a_lo, b_lo + boff, idesc);
              }
            }
          }
          if (NC == 1) ptx::tc_commit(empty0 + stage * 8);
          else ptx::tc_commit_pair(empty0 + stage * 8, 3);
          if (++stage == nst) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (NC == 1) ptx::tc_commit(ptx::smem_u32(&tfull_bar[buf]));
        else ptx::tc_commit_pair(ptx::smem_u32(&tfull_bar[buf]), 3);
      }
    } else if (KBS == 0 && rank == 0 && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(BM * NC, BN);
      const uint64_t qtail_desc0 = ptx::make_desc_k128(ptx::smem_u32(q_tail));
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const int buf = (p.nacc == 2) ? (it & 1) : 0;
        const uint32_t use = (p.nacc == 2) ? (uint32_t)(it >> 1) : (uint32_t)it;  // n-th use of this buffer
        ptx::mbar_wait(ptx::smem_u32(&tempty_bar[buf]), (use & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(p.acc_col0 + buf * BN);
        for (int kb = 0; kb < p.nkb; kb += p.kbs) {
          ptx::mbar_wait(ptx::smem_u32(&full_bar[stage]), phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(stage_base + (size_t)stage * stage_bytes);
          const uint64_t desc0 = ptx::make_desc_k128(sa);
          for (int j = 0; j < p.kbs; ++j) {
#pragma unroll
            for (int k4 = 0; k4 < BK / 16; ++k4) {
              // +2 per 32 bytes of K inside the 128-byte swizzle row, +512 per 8 KiB tile (16-byte units)
              const uint64_t bdesc = desc0 + (uint64_t)(j * (kBoxBytes >> 4) + k4 * 2);
              const uint32_t acc_flag = (kb | j | k4) ? 1u : 0u;
              if (kb + j < p.nkb_tmem) {
                const uint32_t a_tmem = tmem_base + (uint32_t)(((kb + j) * (BK / 16) + k4) * 8);
                if (NC == 1) ptx::mma_ts(d_tmem, a_tmem, bdesc, idesc, acc_flag);
                else ptx::mma_ts_pair(d_tmem, a_tmem, bdesc, idesc, acc_flag);
              } else {
                const uint64_t adesc = qtail_desc0 + (uint64_t)((kb + j - p.nkb_tmem) * (kQTileBytes >> 4) + k4 * 2);
                if (NC == 1) ptx::mma_ss(d_tmem, adesc, bdesc, idesc, acc_flag);
                else ptx::mma_ss_pair(d_tmem, adesc, bdesc, idesc, acc_flag);
              }
            }
          }
          // frees the stage (in both CTAs) when the MMAs retire
          if (NC == 1) ptx::tc_commit(ptx::smem_u32(&empty_bar[stage]));
          else ptx::tc_commit_pair(ptx::smem_u32(&empty_bar[stage]), 3);
          if (++stage == p.nst) {
            stage = 0;
            phase ^= 1;
          }
        }
        // accumulator tile complete (each CTA's epilogue drains its own 128 queries)
        if (NC == 1) ptx::tc_commit(ptx::smem_u32(&tfull_bar[buf]));
        else ptx::tc_commit_pair(ptx::smem_u32(&tfull_bar[buf]), 3);
      }
    }
  } else if (PRE) {
    // ===================== epilogue of the pre-pass: slot maxima =====================
    const bool live = query < p.B;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * (warp & 3)) << 16);
    float smax[kPreSlots];
#pragma unroll
    for (int j = 0; j < kPreSlots; ++j) smax[j] = -INFINITY;
    // masked-out rows contribute -inf: the slots then partition the ALLOWED sampled rows, so the kc-th largest slot
    // maximum is still reached by >= kc rows that may be returned (the bound stays a lower bound of the filtered
    // kc-th best); mask words are read one tile ahead like the pruning bound of the main epilogue
    uint4 next_mw = t0 < t1 ? tile_mask<MASKED>(p.mask, t0 * p.tstride * BN, p.n_rows) : make_uint4(0u, 0u, 0u, 0u);
    int it = 0;
    for (int64_t t = t0; t < t1; ++t, ++it) {
      const uint4 mw = next_mw;
      if (t + 1 < t1) next_mw = tile_mask<MASKED>(p.mask, (t + 1) * p.tstride * BN, p.n_rows);
      const int buf = (p.nacc == 2) ? (it & 1) : 0;
      const uint32_t use = (p.nacc == 2) ? (uint32_t)(it >> 1) : (uint32_t)it;
      ptx::mbar_wait(ptx::smem_u32(&tfull_bar[buf]), use & 1);
      ptx::tc_fence_after();
      const uint32_t acc = lane_addr + (uint32_t)(p.acc_col0 + buf * BN);
      const int64_t row0 = t * p.tstride * BN;
      const int valid = (int)min((int64_t)BN, p.n_rows - row0);
      // 32 columns at a time: 32 + 32 live registers instead of BN + 32 (the pre-pass has TMEM bandwidth to spare)
#pragma unroll
      for (int c32 = 0; c32 < BN / 32; ++c32) {
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(acc + c32 * 32, r);
        ptx::tmem_ld_wait();
        if (c32 == BN / 32 - 1) {  // last read of this accumulator buffer: hand it back
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (NC == 1) ptx::mbar_arrive(ptx::smem_u32(&tempty_bar[buf]));
            else ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tempty_bar[buf]), 0));
          }
        }
        const uint32_t bits = mask_word(mw, c32);
        if (valid == BN && !p.weight_pre && (!MASKED || bits == 0xffffffffu)) {
#pragma unroll
          for (int c = 0; c < 32; ++c) smax[c] = fmaxf(smax[c], __uint_as_float(r[c]));
        } else {
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            const int cc = c32 * 32 + c;
            float sv = __uint_as_float(r[c]);
            if (p.weight_pre) sv *= level_weight_f((cc < valid) ? p.levels[row0 + cc] : (uint8_t)2);
            // rows past the end (TMA zero fill) and masked-out rows
            const bool keep = MASKED ? (cc < valid && ((bits >> c) & 1u)) : cc < valid;
            smax[c] = fmaxf(smax[c], keep ? sv : -INFINITY);
          }
        }
      }
    }
    if (live) {
      float* out_s = p.part_score + ((size_t)query * p.G + g) * kPreSlots;
#pragma unroll
      for (int j = 0; j < kPreSlots; ++j) out_s[j] = smax[j];
    }
  } else {
    // ===================== epilogue: fused top-k =====================
    // Admitted scores do not go into the sorted list one by one: a lane parks them in its FIFO and the warp empties all
    // queues together once per tile (drain_queue).  On large tables admissions are rare either way; on small ones
    // (40 474 rows: ~80 admitted rows per query over 317 tiles, i.e. ~8 per warp and tile, each in a different lane and
    // column) every admission used to cost the whole warp one divergent insert call -- r02t (ncu, B = 8192): 1 360
    // instructions per warp and tile, 480 of them inside list_insert, the MMA thread waiting on the accumulator
    // barrier 106 polls per tile.  Queued, the same admissions cost one convergent drain per tile.
    // Rows still reach a lane's list in ascending id order (columns are tested in ascending order, the queue is
    // FIFO), which the strict '>' admission relies on for the id tie-break.
    const bool live = query < p.B;
    float thr = live ? -INFINITY : INFINITY;  // k-th best of this CTA's list (strict admission)
    float adm = thr;                          // admission threshold: max(thr, just below the global bound)
    float published = -INFINITY;
    int cnt = 0;                              // filled entries of this thread's list
    float qs[kQueue];                         // parked candidates
    int qi[kQueue];
    int qn = 0;
    const int kc = p.kc;
    auto drain = [&]() {
      const uint2 tc = drain_queue(my_s, my_i, kc, cnt, thr, qs, qi, qn);
      thr = __uint_as_float(tc.x);
      cnt = (int)tc.y;
      qn = 0;
      adm = fmaxf(adm, thr);
    };
    int* gb = (p.gbound && live) ? p.gbound + query : nullptr;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * (warp & 3)) << 16);
    int it = 0;
    // the bound is read one tile ahead: its L2 round trip (~700 cycles) overlaps the previous tile's epilogue instead of
    // standing in front of this one's (a bound that is one tile old is still a bound)
    int key = (int)0x80808080;
    if (gb) asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(key) : "l"(gb));
    // the row mask likewise: the four words of a tile are loaded while the previous tile is processed.  A masked-out
    // column fails the admission test below, so it never enters a list and never raises the published bound.
    uint4 next_mw = t0 < t1 ? tile_mask<MASKED>(p.mask, t0 * p.tstride * BN, p.n_rows) : make_uint4(0u, 0u, 0u, 0u);
    for (int64_t t = t0; t < t1; ++t, ++it) {
      const uint4 mw = next_mw;
      if (t + 1 < t1) next_mw = tile_mask<MASKED>(p.mask, (t + 1) * p.tstride * BN, p.n_rows);
      if (gb) {
        // bound proven by any row group: rows strictly below it cannot reach the global top-k
        // (equal scores are still admitted: the id tie-break is decided at the merge)
        const float bound = key_float(key);
        adm = fmaxf(thr, nextafterf(bound, -INFINITY));
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(key) : "l"(gb));
      }
      const int buf = (p.nacc == 2) ? (it & 1) : 0;
      const uint32_t use = (p.nacc == 2) ? (uint32_t)(it >> 1) : (uint32_t)it;
      ptx::mbar_wait(ptx::smem_u32(&tfull_bar[buf]), use & 1);
      ptx::tc_fence_after();
      // drain the whole 128-column accumulator row to registers, then hand the buffer back
      uint32_t r[BN];
      const uint32_t acc = lane_addr + (uint32_t)(p.acc_col0 + buf * BN);
#pragma unroll
      for (int c32 = 0; c32 < BN / 32; ++c32) ptx::tmem_ld_32x32b_x32(acc + c32 * 32, r + c32 * 32);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (NC == 1) ptx::mbar_arrive(ptx::smem_u32(&tempty_bar[buf]));
        else ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tempty_bar[buf]), 0));  // the leader's barrier
      }

      const int64_t row0 = t * p.tstride * BN;
      const int valid = (int)min((int64_t)BN, p.n_rows - row0);
#pragma unroll
      for (int c32 = 0; c32 < BN / 32; ++c32) {
        if (p.weight_pre) {
          // level bytes of these 32 rows (same for every thread: broadcast loads)
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            const int cc = c32 * 32 + c;
            const uint8_t lv = (cc < valid) ? p.levels[row0 + cc] : (uint8_t)2;
            r[cc] = __float_as_uint(__uint_as_float(r[cc]) * level_weight_f(lv));
          }
        }
        // maxima of the eight groups of four CONSECUTIVE columns: a group is looked into only if its maximum passes
        float m8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c0 = c32 * 32 + 4 * j;
          m8[j] = fmaxf(fmaxf(__uint_as_float(r[c0]), __uint_as_float(r[c0 + 1])),
                        fmaxf(__uint_as_float(r[c0 + 2]), __uint_as_float(r[c0 + 3])));
        }
        const float m = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
        const uint32_t bits = mask_word(mw, c32);
        if (m > adm) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (m8[j] > adm) {
              if (qn > kQueue - 4) drain();  // room for the four columns of this group
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int cc = c32 * 32 + 4 * j + e;
                const float sv = __uint_as_float(r[cc]);
                if (sv > adm && cc < valid && ((bits >> (4 * j + e)) & 1u)) {
                  qs[qn] = sv;
                  qi[qn] = (int)(row0 + cc);
                  ++qn;
                }
              }
            }
          }
        }
      }
      if (__any_sync(0xffffffffu, qn > 0)) drain();
      if (gb && thr > published) {
        atomicMax(gb, float_key(thr));
        published = thr;
      }
    }
    // one sorted list per (query, group)
    if (live) {
      float* out_s = p.part_score + ((size_t)query * p.G + g) * p.kc;
      int* out_i = p.part_id + ((size_t)query * p.G + g) * p.kc;
      for (int j = 0; j < p.kc; ++j) {
        out_s[j] = my_s[j * BM];
        out_i[j] = my_i[j * BM];
      }
    }
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

size_t smem_bytes(int bn, int nst, int kbs, int kc, int q_tail_tiles) {
  return (size_t)nst * kbs * (bn * BK * 2) + (size_t)q_tail_tiles * (BM * BK * 2) + (size_t)kc * BM * 8 +
         (2 * kMaxStages + 4) * 8 + 16;
}

}  // namespace

int make_tmap_bf16_2d(void* map128, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                      uint32_t box_cols, bool swizzle128) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    ICD_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres));
    if (!sym || qres != cudaDriverEntryPointSuccess) {
      set_error("cuTensorMapEncodeTiled is not available from this driver");
      return ICD_E_CUDA;
    }
    fn = reinterpret_cast<EncodeFn>(sym);
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = fn(reinterpret_cast<CUtensorMap*>(map128), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(base), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu box=%ux%u)", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, box_rows, box_cols);
    return ICD_E_CUDA;
  }
  return ICD_OK;
}

int make_tmap_bf16_3d(void* map128, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                      uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  ICD_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres));
  if (!sym || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return ICD_E_CUDA;
  }
  cuuint64_t gdim[3] = {d0, d1, d2};
  cuuint64_t gstride[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estride[3] = {1, 1, 1};
  CUresult r = reinterpret_cast<EncodeFn>(sym)(reinterpret_cast<CUtensorMap*>(map128), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                                               3, const_cast<void*>(base), gdim, gstride, box, estride,
                                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)r);
    return ICD_E_CUDA;
  }
  return ICD_OK;
}

#ifdef ICD_PROFILING
// timing experiment only: the same bytes viewed as [tiles][K blocks][128 rows][64 elements] (tile-major)
static int make_tmap_bf16_4d_tiled(void* map128, const void* base, uint64_t tiles, uint32_t nkb, uint32_t box_rows, uint32_t box_kb) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  ICD_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres));
  cuuint64_t gdim[4] = {64, 128, nkb, tiles};
  cuuint64_t gstride[3] = {128, 128 * 128, (cuuint64_t)128 * 128 * nkb};
  cuuint32_t box[4] = {64, box_rows, box_kb, 1};
  cuuint32_t estride[4] = {1, 1, 1, 1};
  CUresult r = reinterpret_cast<EncodeFn>(sym)(reinterpret_cast<CUtensorMap*>(map128), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                                               const_cast<void*>(base), gdim, gstride, box, estride,
                                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(4d) failed with CUresult %d", (int)r);
    return ICD_E_CUDA;
  }
  return ICD_OK;
}
#endif

// tuning knobs: defaults (profiling builds, -DICD_PROFILING: from the environment -- ICD_SCAN_BN = 64 | 128, ICD_SCAN_DRIFT = tiles, 0 = limiter
// off, ICD_SCAN_TMAX = query tiles sharing one row stream per launch, ICD_SCAN_KBS = K blocks per stage,
// ICD_SCAN_SAMPLE = pre-pass stride, 0 = off, -1 = by table size); icd_tune() overrides them at run time.
static int env_int(const char* name, int dflt) {
#ifdef ICD_PROFILING
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
#else
  (void)name;   // production builds ignore the environment: knobs move only through icd_tune()
  return dflt;
#endif
}
struct Tunables {
  int bn, drift, tmax, kbs, kbs_pair, sample, qsplit, pair, qtmem, generic, tiled, pre_slots, small_pre, gen;
  Tunables() {
    bn = 128;
    drift = std::max(0, env_int("ICD_SCAN_DRIFT", 4));
    tmax = std::min(32, std::max(1, env_int("ICD_SCAN_TMAX", 16)));
    kbs = std::min(6, std::max(1, env_int("ICD_SCAN_KBS", 3)));            // K blocks per stage, single CTAs
    kbs_pair = std::min(6, std::max(1, env_int("ICD_SCAN_KBS_PAIR", 6)));  // ... CTA pairs (half-height boxes)
    sample = env_int("ICD_SCAN_SAMPLE", -1);
    qsplit = env_int("ICD_SCAN_QSPLIT", -1);  // -1 auto (tensor-bound launches), 0 off, 1 always
    pair = env_int("ICD_SCAN_PAIR", -1);      // CTA pairs: -1 auto (even number of query tiles >= 2), 0 off
    qtmem = env_int("ICD_SCAN_QTMEM", 0);      // K blocks of the query tile kept in TMEM when split (0 = all that fit: 8)
    tiled = 0;
    pre_slots = 1;
    small_pre = 1;   // pre-pass on tables below 512 k rows (icd_tune "scan_small_pre", 0 = round-2 behaviour: none)
    generic = env_int("ICD_SCAN_GENERIC", 0);   // 1 = always the generic (run-time shape) issue loop: A/B only
    gen = 0;
  }
};
static Tunables& tun() {
  static Tunables t;
  return t;
}
static int scan_bn() { return tun().bn; }
static int scan_drift() { return tun().drift; }
static int scan_tmax() { return tun().tmax; }

int tensor_scan_tune(const char* key, int value) {
  Tunables& t = tun();
  if (!strcmp(key, "scan_drift")) t.drift = std::max(0, value);
  else if (!strcmp(key, "scan_tmax")) t.tmax = std::min(32, std::max(1, value));
  else if (!strcmp(key, "scan_kbs")) t.kbs = std::min(6, std::max(1, value));
  else if (!strcmp(key, "scan_kbs_pair")) t.kbs_pair = std::min(6, std::max(1, value));
  else if (!strcmp(key, "scan_sample")) t.sample = value;
  else if (!strcmp(key, "scan_qsplit")) t.qsplit = value;
  else if (!strcmp(key, "scan_pair")) t.pair = value;
  else if (!strcmp(key, "scan_qtmem")) t.qtmem = std::max(0, value);
  else if (!strcmp(key, "scan_generic")) t.generic = value != 0;
  else if (!strcmp(key, "scan_pre_slots")) t.pre_slots = value != 0;
  else if (!strcmp(key, "scan_small_pre")) t.small_pre = value != 0;
#ifdef ICD_PROFILING
  else if (!strcmp(key, "scan_tiled")) t.tiled = value != 0;
#endif
  else return ICD_E_ARG;
  ++t.gen;  // tensor maps depend on bn / kbs: indexes rebuild theirs when the generation moves
  return ICD_OK;
}
int tensor_scan_generation() { return tun().gen; }

int tensor_scan_max_partials() { return kSMs; }
int tensor_scan_pre_slots() { return kPreSlots; }
int tensor_scan_pre_capacity() { return kPreSlots * kPreFolds; }
int tensor_scan_pre_mode() { return tun().pre_slots; }
int tensor_scan_sample_stride(int64_t n_rows, int kc) {
  const int forced = tun().sample;
  if (forced >= 0) return forced <= 1 ? 0 : forced;
  if (kc > kPreSlots * kPreFolds || tun().pre_slots == 0) {
    // list-based pre-pass (its warm-up inserts cost as much as they save on small tables): calibrated in round 1
    return n_rows >= (2 << 20) ? 256 : (n_rows >= (1 << 19) ? 64 : 0);
  }
  // slot-maxima pre-pass: its cost is the sampled rows' share of the stream (rows / stride), its gain the main scan's
  // warm-up inserts (~ log of the stride), so the optimum keeps the SAMPLE at about 200 k rows whatever the table size:
  // stride 8 at 1 M rows (0.48 vs 1.02 ms with 256), 64 at 12.5 M, 256 at 100 M (profiles/r02k_prepass_stride_ab.jsonl)
  // Small tables (the reference's own 40 474 rows, BASELINE configs[1]): WITHOUT a bound every (query, row group) list
  // warms up on its own -- kc (1 + ln(rows per group / kc)) divergent inserts per thread, ~2 ms at B = 1024 against
  // ~0.05 ms of MMA work (r02m) -- so here the pre-pass is worth even half of the table: every second row tile.
  if (n_rows < (1 << 17)) return tun().small_pre ? 2 : 0;
  if (n_rows < (1 << 19)) return tun().small_pre ? 4 : 0;
  int stride = 4;
  while (stride < 256 && (double)n_rows / (2.0 * stride) > 141000.0) stride *= 2;  // nearest power of two to rows / 200 k
  return stride;
}
int tensor_scan_progress_ints() { return 64 * kSMs; }

bool tensor_scan_supported(int dim, int k) {
  return dim % BK == 0 && dim >= BK && dim <= 768 && k >= 1 && k <= ICD_MAX_K;
}

static int stage_kblocks(int dim) {
  const int nkb = dim / BK;
  const int want = tun().kbs;
  for (int kbs = std::min(want, nkb); kbs > 1; --kbs)
    if (nkb % kbs == 0) return kbs;
  return 1;
}

int tensor_scan_make_map(void* map128, const void* table, int64_t n_rows, int dim) {
  // 3-D view {64 elements, rows, K blocks}: strides {dim*2 bytes, 128 bytes}
  return make_tmap_bf16_3d(map128, table, BK, (uint64_t)n_rows, (uint64_t)(dim / BK), (uint64_t)dim * 2, BK * 2, BK,
                           (uint32_t)scan_bn(), (uint32_t)stage_kblocks(dim));
}

// co-resident CTA pairs the device can hold for this kernel (every CTA of a launch must be resident: the drift
// limiter and the pruning bound make them wait on each other)
template <int BN>
static int resident_pairs(size_t smem) {
  static int cached = 0;
  if (cached) return cached;
  cudaFuncSetAttribute(scan_tc_kernel<BN, 2, 0, 0, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(kSMs);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, scan_tc_kernel<BN, 2, 0, 0, false, false>, &cfg) != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  cached = std::max(0, n);
  return cached;
}

template <int BN, int NC, int KBS, int NKBT, bool PRE, bool MASKED>
static int launch_one_pre(const CUtensorMap& tmap, const ScanParams& p, int grid, size_t smem, cudaStream_t st) {
  auto kernel = scan_tc_kernel<BN, NC, KBS, NKBT, PRE, MASKED>;
  static bool attr_set = false;
  if (!attr_set) {
    ICD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  if (NC == 2) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  ICD_CUDA(cudaLaunchKernelEx(&cfg, kernel, tmap, p));
  count_launch();
  return ICD_OK;
}

template <int BN, int NC, int KBS, int NKBT>
static int launch_one(const CUtensorMap& tmap, const ScanParams& p, int grid, size_t smem, cudaStream_t st, bool pre) {
  if (p.mask)
    return pre ? launch_one_pre<BN, NC, KBS, NKBT, true, true>(tmap, p, grid, smem, st)
               : launch_one_pre<BN, NC, KBS, NKBT, false, true>(tmap, p, grid, smem, st);
  return pre ? launch_one_pre<BN, NC, KBS, NKBT, true, false>(tmap, p, grid, smem, st)
             : launch_one_pre<BN, NC, KBS, NKBT, false, false>(tmap, p, grid, smem, st);
}

template <int BN>
static int launch_tensor_scan_bn(const TensorScanArgs& a, const void* map128, cudaStream_t st) {
  const int T_total = (a.B + BM - 1) / BM;
  const int tstride = std::max(1, a.tile_stride);
  const int64_t total_tiles = ((a.n_rows + BN - 1) / BN + tstride - 1) / tstride;
  // query tiles per launch: as equal as possible over ceil(T_total / tmax) launches, so that every
  // launch fills the SMs (G * T_launch <= 148) and at most tmax CTAs share one row stream
  const int n_launch = (T_total + scan_tmax() - 1) / scan_tmax();
  const int T_launch = (T_total + n_launch - 1) / n_launch;
  // CTA pairs: every launch must hold an even number of query tiles (the pair = two neighbouring tiles)
  bool pair = BN == 128 && tun().pair != 0 && T_launch >= 2 && T_launch % 2 == 0 && T_total % T_launch == 0;
  int sms = kSMs;
  if (pair) {
    const int rp = resident_pairs<BN>((size_t)kSmemLimit);
    if (rp * 2 < T_launch) pair = false;
    else sms = std::min(kSMs, rp * 2);
  }
  const int NC = pair ? 2 : 1;
  int G = std::max(1, sms / T_launch);
  G = (int)std::min<int64_t>(G, total_tiles);
  G = std::min(G, a.P);
  *a.groups_used = G;

  // Query tile placement: all of K in TMEM, or (tensor-bound launches, dim wider than 512) the K blocks that do not
  // leave room for a second accumulator buffer in shared memory (a third of K at dim = 768; the knob scan_qtmem moves
  // more of it: measured no better, r01d pair sweep).
  const int nkb = a.dim / BK;
  const int nkb_fit2 = (kTmemCols - 2 * BN) / (BK / 2);  // K blocks that fit beside two BN-column accumulators
  // the split pays at every batch size (r01e: B = 8 0.94 -> 1.02, B = 32 0.93 -> 0.97, B = 128 0.885 -> 0.92 of the
  // HBM peak: the drain no longer holds up the next tile's MMAs); it is dropped when the candidate lists (large k)
  // leave fewer than three pipeline stages beside the 64 KiB tail
  const bool want_split = tun().qsplit != 0 && nkb > nkb_fit2 && BN == 128;
  // K blocks per stage: longer K slices per bulk copy are longer DRAM bursts and fewer barrier round trips per
  // tile (r01e, 10 M rows, pairs, B = 1024: 2 -> 0.82, 3 -> 0.88, 4 -> 0.91, 6 -> 0.94 of sustained bf16 peak; single
  // CTAs at B = 128 peak at 3).  Largest divisor of nkb <= the knob that still leaves >= 3 stages beside the Q tail;
  // if none does, the split goes first, then the stage shrinks.
  const int kbs_want = std::min(pair ? tun().kbs_pair : tun().kbs, nkb);
  const int kc_smem = a.pre_slots ? 0 : a.k;  // the slot-maxima pre-pass keeps no lists: its stages get that room
  int kbs = 0, nkb_tmem = nkb, q_tail_tiles = 0, nst = 0;
  for (int pass = 0; pass < 2 && kbs == 0; ++pass) {
    const bool split = pass == 0 && want_split;
    if (pass == 0 && !want_split) continue;
    int tmem_kb = nkb;
    if (split) {
      tmem_kb = tun().qtmem > 0 ? std::min(tun().qtmem, nkb_fit2) : nkb_fit2;
      tmem_kb = std::max(tmem_kb, nkb - 8);  // at most 8 tail tiles (128 KiB) in shared memory
    }
    for (int c = kbs_want; c >= 1 && kbs == 0; --c) {
      if (nkb % c) continue;
      int n = kMaxStages;
      while (n > 2 && smem_bytes(BN / NC, n, c, kc_smem, nkb - tmem_kb) > (size_t)kSmemLimit) --n;
      if (smem_bytes(BN / NC, n, c, kc_smem, nkb - tmem_kb) > (size_t)kSmemLimit) continue;
      if (split && n < 3) continue;
      kbs = c, nst = n, nkb_tmem = tmem_kb, q_tail_tiles = nkb - tmem_kb;
    }
  }
  if (kbs == 0) {
    set_error("tensor scan: k=%d does not fit shared memory", a.k);
    return ICD_E_UNSUPPORTED;
  }
  const size_t smem = smem_bytes(BN / NC, nst, kbs, kc_smem, q_tail_tiles);
  // a table that stays in L2 needs no drift limiter (its polls only cost latency there)
  const bool l2_table = (size_t)a.n_rows * a.dim * 2 <= ((size_t)64 << 20);
  // the stage shape is chosen per launch, so the 3-D view {64 elements, rows, K blocks} of the table is encoded here
  // (a host-side call of a few microseconds); each CTA of a pair loads half of a row tile
  (void)map128;
  CUtensorMap tmap;
  {
    alignas(128) unsigned char pm[128];
#ifdef ICD_PROFILING
    if (tun().tiled && BN == 128) {
      ICD_TRY(make_tmap_bf16_4d_tiled(pm, a.table, (uint64_t)(a.n_rows / BN), (uint32_t)(a.dim / BK), (uint32_t)(BN / NC), (uint32_t)kbs));
    } else
#endif
    ICD_TRY(make_tmap_bf16_3d(pm, a.table, BK, (uint64_t)a.n_rows, (uint64_t)(a.dim / BK), (uint64_t)a.dim * 2, BK * 2, BK,
                              (uint32_t)(BN / NC), (uint32_t)kbs));
    memcpy(&tmap, pm, sizeof(CUtensorMap));
  }
  int launch = 0;
  for (int qt0 = 0; qt0 < T_total; qt0 += T_launch, ++launch) {
    ScanParams p{};
    p.levels = a.levels;
    p.q = reinterpret_cast<const __nv_bfloat16*>(a.q_bf16);
    p.part_score = a.part_score;
    p.part_id = a.part_id;
    p.gbound = a.gbound;
    p.n_rows = a.n_rows;
    p.dim = a.dim;
    p.nkb = a.dim / BK;
    p.B = a.B;
    p.kc = kc_smem;
    p.weight_pre = a.weight_pre;
    p.G = G;
    p.T = std::min(T_launch, T_total - qt0);
    p.qt0 = qt0;
    p.nst = nst;
    p.kbs = kbs;
    p.nkb_tmem = nkb_tmem;
    p.acc_col0 = ((nkb_tmem * (BK / 2) + 127) / 128) * 128;
    p.nacc = (kTmemCols - p.acc_col0) / BN >= 2 ? 2 : 1;
    p.tstride = tstride;
    p.drift = scan_drift();
    p.mask = a.mask;
    p.progress = (a.progress && p.drift > 0 && p.T > 1 && launch < 64 && !l2_table) ? a.progress + (size_t)launch * kSMs : nullptr;
#ifdef ICD_PROFILING
    p.tiled = (tun().tiled && BN == 128) ? 1 : 0;
#endif
    // specialised issue loops for the shapes the launcher actually picks at dim = 768 (everything else: generic)
    const bool pre = a.pre_slots != 0;
    const bool spec = BN == 128 && a.dim == 768 && nkb_tmem == 8 && tun().generic == 0;
    if (pair && spec && kbs == 6) ICD_TRY((launch_one<BN, 2, 6, 8>(tmap, p, G * p.T, smem, st, pre)));
    else if (pair && spec && kbs == 4) ICD_TRY((launch_one<BN, 2, 4, 8>(tmap, p, G * p.T, smem, st, pre)));  // kc = 36 lists
    else if (pair && spec && kbs == 3) ICD_TRY((launch_one<BN, 2, 3, 8>(tmap, p, G * p.T, smem, st, pre)));
    else if (pair) ICD_TRY((launch_one<BN, 2, 0, 0>(tmap, p, G * p.T, smem, st, pre)));
    else if (spec && kbs == 3) ICD_TRY((launch_one<BN, 1, 3, 8>(tmap, p, G * p.T, smem, st, pre)));
    else if (spec && kbs == 2) ICD_TRY((launch_one<BN, 1, 2, 8>(tmap, p, G * p.T, smem, st, pre)));
    else ICD_TRY((launch_one<BN, 1, 0, 0>(tmap, p, G * p.T, smem, st, pre)));
  }
  return ICD_OK;
}

int launch_tensor_scan(const TensorScanArgs& a, const void* map128, cudaStream_t st) {
  if (!tensor_scan_supported(a.dim, a.k)) {
    set_error("tensor scan: unsupported dim=%d k=%d", a.dim, a.k);
    return ICD_E_UNSUPPORTED;
  }
  // BN = 128 only: with the query tile in tensor memory an N = 64 MMA runs the pipe at half rate (r01: 38 % tensor-active)
  return launch_tensor_scan_bn<128>(a, map128, st);
}

}  // namespace icd
